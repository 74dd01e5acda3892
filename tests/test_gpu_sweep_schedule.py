"""The persistent schedule of the pipelined sweep (csrc/sweep_kernel.cuh, PipeSched): where the (32-chain group, block) units allow
an even spread over the device's S = 4 x SMs schedulers, warps take the units' intervals by ticket and hand each chain's state on
at interval boundaries.  The schedule is chosen from U = units: 2S warps when U >= 2S, S warps when S <= U < 1.23 S, one unit per
warp otherwise.  Each band is run against the register-tile kernel (set_sweep_mode(1)): decisions equal, ll and X° to FP64 rounding.
Which warp runs which task changes from run to run; the results must not."""
import math

import numpy as np
import pytest
import torch

from dmt_b200 import _lib, configs
from harness import make_ctx, rel_err

pytestmark = [pytest.mark.gpu, pytest.mark.own_lanes]

K = 40  # intervals of 8 steps


def schedulers():
    return 4 * torch.cuda.get_device_properties(0).multi_processor_count


def blocks(lengths):
    out, k = [], 0
    for n in lengths:
        out.append((k, k + n - 1))
        k += n
    assert k == K
    return out


def case(band):
    """chains and the two layouts: a regular one and a staggered one whose end blocks are half as long"""
    S = schedulers()
    if band == "two_warps":      # U >= 2S on both layouts
        lay = [[4] * 10, [2] + [4] * 9 + [2]]
        M = 32 * math.ceil(2 * S / 10) - 3                 # (a partial last chain group)
    elif band == "two_warps_min":  # U = 2S + 1 on the first layout: one ticket of slack between a unit's intervals
        nb = max([n for n in range(2, 21) if (2 * S + 1) % n == 0], default=None)
        if nb is None:
            pytest.skip("2S + 1 has no divisor in 2..20")
        q, r = divmod(K, nb)
        lay = [[q + 1] * r + [q] * (nb - r), [2] + [4] * 9 + [2]]
        M = 32 * ((2 * S + 1) // nb)
    else:                        # S <= U < 1.23 S on both layouts
        lay = [[4] * 10, [2] + [4] * 9 + [2]]
        M = 32 * (S // 10 + 1)
        assert S <= (M // 32) * 10 and (M // 32) * 11 < 1.23 * S
    return M, [(blocks(lay[0]), 0.7), (blocks(lay[1]), 0.8)]


def start(M, layouts, cached, seed=31):
    prob = configs.make_problem("lorenz", M, K=K, obs_dt=0.1, dt=0.1 / 8, seed=12, layouts=layouts + [([(0, K - 1)], 0.0)], rho=0.7)
    ctx = make_ctx(prob, seed=seed)
    ctx.recompute_guiding_term(2, _lib.P_ONLY)
    assert ctx.init_paths(2, iter0=500, max_tries=50) == 0
    ctx.set_lazy_noise(True)
    if cached:
        ctx.enable_guiding_cache(0); ctx.enable_guiding_cache(1)
    return ctx


@pytest.mark.parametrize("cached", [False, True], ids=["uncached", "cached"])
@pytest.mark.parametrize("band", ["two_warps", "two_warps_min", "one_warp"])
def test_scheduled_sweep_equals_register_tile_sweep(band, cached):
    M, layouts = case(band)
    a, b = start(M, layouts, cached), start(M, layouts, cached)
    a.set_sweep_mode(1)
    b.set_sweep_mode(2)
    n_acc = 0
    for it in range(6):
        l = it % 2
        a.blocking_sweep(l, it // 2); b.blocking_sweep(l, it // 2)
        assert b.last_forward_kernel() == "sweep_pipe_kernel<lanes=1, lazy>"
        assert np.array_equal(a.get_success(l), b.get_success(l))
        good = a.get_success(l).all(axis=0)
        assert np.isfinite(a.get_ll(l, 0)).all()
        assert rel_err(b.get_ll(l, 0), a.get_ll(l, 0)) < 1e-10 and rel_err(b.get_ll(l, 1), a.get_ll(l, 1)) < 1e-10
        assert rel_err(b.get_X(1)[:, :, good], a.get_X(1)[:, :, good]) < 1e-10
        a.accept_reject_path(l, it // 2); b.accept_reject_path(l, it // 2)
        assert np.array_equal(a.get_last_accept(l), b.get_last_accept(l))
        n_acc += a.get_last_accept(l).sum()
        assert rel_err(b.get_X(0), a.get_X(0)) < 1e-10
    assert n_acc > 0
    a.close(); b.close()


@pytest.mark.parametrize("band", ["two_warps", "one_warp"])
def test_scheduled_sweep_is_deterministic(band):
    M, layouts = case(band)
    a, b = start(M, layouts, True), start(M, layouts, True)
    a.set_sweep_mode(2); b.set_sweep_mode(2)
    for it in range(4):
        l = it % 2
        for c in (a, b):
            c.blocking_sweep(l, it)
            c.accept_reject_path(l, it)
        assert a.last_forward_kernel() == "sweep_pipe_kernel<lanes=1, lazy>"
        for side in (0, 1):
            assert np.array_equal(a.get_ll(l, side), b.get_ll(l, side))
            assert np.array_equal(a.get_X(side), b.get_X(side))
        assert np.array_equal(a.get_last_accept(l), b.get_last_accept(l))
    a.close(); b.close()
