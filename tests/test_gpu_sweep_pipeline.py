"""The software-pipelined blocking-sweep kernel (csrc/sweep_kernel.cuh: guiding term through a TMA shared-memory ring, X
double-buffered in registers) and the lazy-noise mode, against the register-tile kernel it replaces.  (Against the ORACLE the
pipelined kernel is covered by every blocking test of test_gpu_parity.py / test_gpu_full_size.py in their `lanes_auto` runs.)"""
import numpy as np
import pytest

import dmt_b200
from dmt_b200 import _lib, configs
from harness import make_ctx, rel_err

pytestmark = [pytest.mark.gpu, pytest.mark.own_lanes]

NAMES = ["fhn", "lv", "lorenz", "prok", "jr", "ou2"]


def problem(name, M, K=8, nsteps=11, seed=12):
    layouts = [([(0, 2), (3, 5), (6, 7)], [0.6, 0.7, 0.8]), ([(0, 3), (4, 7)], 0.5), ([(0, K - 1)], 0.0)]
    if name == "jr":   # (the tame Jansen-Rit instance of test_gpu_parity.blocking_problem: the BASELINE constants are singular under blocking)
        from test_gpu_parity import JR_TAME
        prob = configs.make_problem("jr", M, K=K, obs_dt=0.1, dt=0.1 / nsteps, seed=seed, layouts=layouts, rho=0.7, theta=JR_TAME)
        prob.eps = 1e-4
        return prob
    return configs.make_problem(name, M, K=K, obs_dt=0.1, dt=0.1 / nsteps, seed=seed, layouts=layouts, rho=0.7)


def start(prob, seed=31, **kw):
    ctx = make_ctx(prob, seed=seed, ll_hist_len=8, **kw)
    ctx.recompute_guiding_term(2, _lib.P_ONLY)
    assert ctx.init_paths(2, iter0=500, max_tries=50) == 0
    return ctx


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("M", [41, 64, 7])
@pytest.mark.parametrize("lanes", [1, "ws", "sp"])
def test_pipelined_sweep_equals_register_tile_sweep(name, M, lanes):
    """same inputs, same random stream, same arithmetic: equal up to FP64 rounding (different FMA contraction), decisions equal;
    with one lane per (chain, block), with the warp-specialised kernel (csrc/sweep_ws_kernel.cuh: generator, inverse solve, proposal
    recursion and proposal likelihood on different warps, coupled by shared-memory rings), and with the step-parallel kernel
    (csrc/sweep_sp_kernel.cuh: four lanes per (chain, block), lane = step of the tile; ll and ll° summed in a different order)"""
    prob = problem(name, M)
    a, b = start(prob), start(prob)
    a.set_sweep_mode(1)
    if isinstance(lanes, str):
        b.set_sweep_mode({"ws": 3, "sp": 5}[lanes])
    else:
        b.set_sweep_mode(2); b.set_fwd_lanes(lanes)
    n_acc = 0
    for it in range(6):
        l = it % 2
        a.blocking_sweep(l, it // 2); b.blocking_sweep(l, it // 2)
        assert np.array_equal(a.get_success(l), b.get_success(l))
        good = a.get_success(l).all(axis=0)
        assert rel_err(b.get_W(0), a.get_W(0)) < 1e-10
        assert np.isfinite(a.get_ll(l, 0)).all()
        assert rel_err(b.get_ll(l, 0), a.get_ll(l, 0)) < 1e-10 and rel_err(b.get_ll(l, 1), a.get_ll(l, 1)) < 1e-10
        assert rel_err(b.get_X(1)[:, :, good], a.get_X(1)[:, :, good]) < 1e-10 and rel_err(b.get_W(1)[:, :, good], a.get_W(1)[:, :, good]) < 1e-10
        a.accept_reject_path(l, it // 2); b.accept_reject_path(l, it // 2)
        assert np.array_equal(a.get_last_accept(l), b.get_last_accept(l))
        n_acc += a.get_last_accept(l).sum()
        assert rel_err(b.get_X(0), a.get_X(0)) < 1e-10
    assert n_acc > 0
    a.close(); b.close()


def test_pipelined_sweep_refuses_what_it_cannot_do():
    prob = problem("lorenz", 16)
    prob.P = 1; prob.v = prob.v[:, :, :1].copy(); prob.xbar = prob.xbar[:, :, :1].copy()
    prob.x0 = np.repeat(prob.x0[:, :1], 16, axis=1); prob.layouts = [([(0, 7)], 0.5)]
    ctx = make_ctx(prob, seed=1)
    ctx.recompute_guiding_term(0, _lib.P_ONLY)
    assert ctx.init_paths(0, 0, 20) == 0
    ctx.set_sweep_mode(2)
    with pytest.raises(dmt_b200.DmtError):          # one shared parameter set: a warp's sectors are not contiguous per chain
        ctx.find_W_loglikhd_draw(0, 1)
    ctx.set_sweep_mode(0)
    ctx.find_W_loglikhd_draw(0, 1)                  # automatic: falls back to the register-tile kernel (another CUDA kernel, not a CPU path)
    with pytest.raises(dmt_b200.DmtError):
        ctx.set_sweep_mode(6)
    with pytest.raises(dmt_b200.DmtError):
        ctx.set_sweep_mode(4)
    with pytest.raises(dmt_b200.DmtError):
        ctx.set_sweep_mode(3); ctx.find_W_loglikhd_draw(0, 1)
    with pytest.raises(dmt_b200.DmtError):
        ctx.set_sweep_mode(5); ctx.find_W_loglikhd_draw(0, 1)
    ctx.close()


@pytest.mark.parametrize("name", ["lorenz", "fhn", "prok"])
@pytest.mark.parametrize("mode", [1, 2, 3, 5])
def test_lazy_noise_changes_nothing_but_the_moment_W_is_computed(name, mode):
    """dmt_set_lazy_noise: the sweep stops storing W_acc / W°; paths, log-likelihoods and decisions are unchanged, and the accepted
    noise read back later is K5 of the accepted path under the law swept last — what find_W_for_X! returns."""
    prob = problem(name, 45)
    a, b = start(prob), start(prob)
    a.set_sweep_mode(2); b.set_sweep_mode(mode)
    b.set_lazy_noise(True)
    for it in range(6):
        l = it % 2
        a.blocking_sweep(l, it // 2); b.blocking_sweep(l, it // 2)
        assert np.array_equal(a.get_success(l), b.get_success(l))
        good = a.get_success(l).all(axis=0)
        assert rel_err(b.get_ll(l, 0), a.get_ll(l, 0)) < 1e-12 and rel_err(b.get_ll(l, 1), a.get_ll(l, 1)) < 1e-12
        assert rel_err(b.get_X(1)[:, :, good], a.get_X(1)[:, :, good]) < 1e-12
        a.accept_reject_path(l, it // 2); b.accept_reject_path(l, it // 2)
        assert np.array_equal(a.get_last_accept(l), b.get_last_accept(l))
        assert rel_err(b.get_X(0), a.get_X(0)) < 1e-12
    # the noise on demand: after the accept step W_acc is the proposal's noise where accepted, the recovered noise elsewhere
    Wa = a.get_W(0)
    Wb = b.get_W(0)                                  # K5 over layout 1 (swept last), launched by the read itself
    assert rel_err(Wb, Wa) < 1e-7                    # K5 o K2 round trip (the proposal path was MADE from Wa's entries)
    assert np.array_equal(b.get_W(0), Wb)            # materialised once, then just read
    # a plain (non-blocking) pCN draw reads W: both contexts continue identically
    for c in (a, b):
        c.recompute_guiding_term(2, _lib.P_ONLY); c.loglikhd(2, 0, 0); c.set_rho(2, [0.8])
    b.blocking_sweep(0, 7); a.blocking_sweep(0, 7)   # one more lazy sweep, then a draw WITHOUT find_W_for_X!: W must be rebuilt first
    for c in (a, b):
        c.accept_reject_path(0, 7)
        c.recompute_guiding_term(2, _lib.P_ONLY); c.loglikhd(2, 0, 0)
        c.draw_proposal_path(2, 9)
    assert np.array_equal(a.get_success(2), b.get_success(2))
    assert rel_err(b.get_ll(2, 1), a.get_ll(2, 1)) < 1e-6 and rel_err(b.get_X(1), a.get_X(1)) < 1e-6
    # switching the mode off materialises W and goes back to eager stores
    b.set_lazy_noise(False)
    a.blocking_sweep(1, 11); b.blocking_sweep(1, 11)
    assert rel_err(b.get_W(0), a.get_W(0)) < 1e-6 and rel_err(b.get_W(1), a.get_W(1)) < 1e-6
    a.close(); b.close()


def test_lazy_noise_with_guiding_cache_and_law_change():
    """lazy W together with the guiding cache (private per-layout store) and a parameter change in between: the law change
    materialises W first (the noise belongs to the OLD law), then invalidates the cache"""
    prob = problem("lorenz", 40)
    a, b = start(prob), start(prob)
    for c in (a, b):
        c.enable_guiding_cache(0); c.enable_guiding_cache(1)
    b.set_lazy_noise(True)
    for it in range(4):
        l = it % 2
        for c in (a, b):
            c.blocking_sweep(l, it); c.accept_reject_path(l, it)
    th = prob.theta * (1 + 1e-3)
    for c in (a, b):
        c.set_params(th, side=0, stores=3)           # b: ensure_W runs here, before the laws move
        c.set_aux_linearised(prob.xbar, side=0, store=0); c.set_aux_linearised(prob.xbar, side=0, store=1)
    assert rel_err(b.get_W(0), a.get_W(0)) < 1e-7
    for it in range(4, 6):
        l = it % 2
        for c in (a, b):
            c.blocking_sweep(l, it); c.accept_reject_path(l, it)
        assert np.array_equal(a.get_last_accept(l), b.get_last_accept(l))
        assert rel_err(b.get_X(0), a.get_X(0)) < 1e-12 and rel_err(b.get_ll(l, 0), a.get_ll(l, 0)) < 1e-12
    a.close(); b.close()
