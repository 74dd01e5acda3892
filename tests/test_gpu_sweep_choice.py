"""Which kernel the fused blocking-sweep pass runs under the automatic choice (dmt_set_sweep_mode(0), include/dmt.h): one blocking
sweep, then dmt_get_last_forward_kernel.  The band edges follow the device's resident-wave sizes, so the expected names are the ones
a B200 takes; the sizes sit inside the bands of a 10-block layout (warp-specialised, step-parallel, two register-tile lanes,
pipelined)."""
import pytest

from dmt_b200 import _lib, configs
from harness import make_ctx

pytestmark = [pytest.mark.gpu, pytest.mark.own_lanes]

K = 20  # intervals of 8 steps; layout 0: 10 blocks of 2 intervals, layout 1: one block (init)


def sweep_kernel(name, M, lazy=True, fwd_lanes=0):
    layouts = [([(2 * b, 2 * b + 1) for b in range(10)], 0.9), ([(0, K - 1)], 0.0)]
    prob = configs.make_problem(name, M, K=K, obs_dt=0.1, dt=0.1 / 8, seed=5, layouts=layouts)
    ctx = make_ctx(prob, seed=7)
    ctx.recompute_guiding_term(1, _lib.P_ONLY)
    ctx.init_paths(1, iter0=100, max_tries=5)       # (the choice does not depend on the paths)
    ctx.set_lazy_noise(lazy)
    if fwd_lanes:
        ctx.set_fwd_lanes(fwd_lanes)
    ctx.blocking_sweep(0, 1)
    kernel = ctx.last_forward_kernel()
    ctx.close()
    return kernel


LORENZ = [  # chains, lazy noise, kernel
    (256, True, "sweep_ws_kernel<wide, lazy>"),           # (32-chain, block) units fit one round of CTAs
    (512, True, "sweep_sp_kernel<step lanes=4, lazy>"),   # then step-parallel up to 14,080 (chain, block) units
    (1024, True, "sweep_sp_kernel<step lanes=4, lazy>"),
    (1536, True, "fwd_kernel<op=6, lanes=2, lazy>"),      # then two register-tile lanes while the doubled grid fits one wave
    (4096, True, "sweep_pipe_kernel<lanes=1, lazy>"),     # then the pipelined kernel
    (256, False, "sweep_ws_kernel<wide, eager>"),
    (512, False, "sweep_sp_kernel<step lanes=4>"),
    (1024, False, "sweep_sp_kernel<step lanes=4>"),
    (1536, False, "fwd_kernel<op=6, lanes=2>"),
    (4096, False, "fwd_kernel<op=6, lanes=1>"),           # eager noise: the register-tile kernel
]
FHN = [
    (256, True, "sweep_ws_kernel<wide, lazy>"),
    (1024, True, "sweep_pipe_kernel<lanes=1, lazy>"),     # one Wiener coordinate: no step-parallel and no two-lane band
    (1024, False, "fwd_kernel<op=6, lanes=1>"),
]


def ids(cases):
    return ["%d-%s" % (M, "lazy" if lazy else "eager") for M, lazy, _ in cases]


@pytest.mark.parametrize("M,lazy,kernel", LORENZ, ids=ids(LORENZ))
def test_lorenz_ten_blocks(M, lazy, kernel):
    assert sweep_kernel("lorenz", M, lazy=lazy) == kernel


def test_one_shared_parameter_set_takes_the_register_tile_kernel():
    # (blocking needs one parameter set per chain: the same fused pass on one terminal block, find_W_for_X!; loglikhd!; draw_proposal_path!)
    prob = configs.make_problem("lorenz", 256, 1, K=K, obs_dt=0.1, dt=0.1 / 8, seed=5, layouts=[([(0, K - 1)], 0.9)])
    ctx = make_ctx(prob, seed=7)
    ctx.recompute_guiding_term(0, _lib.P_ONLY)
    ctx.init_paths(0, iter0=100, max_tries=5)
    ctx.set_lazy_noise(True)
    ctx.find_W_loglikhd_draw(0, 1)
    assert ctx.last_forward_kernel() == "fwd_kernel<op=6, lanes=2, lazy>"
    ctx.close()


@pytest.mark.parametrize("M,lazy,kernel", FHN, ids=ids(FHN))
def test_one_wiener_coordinate(M, lazy, kernel):
    assert sweep_kernel("fhn", M, lazy=lazy) == kernel


@pytest.mark.parametrize("M,lanes", [(256, 1), (4096, 4)])
def test_forced_lanes_take_the_register_tile_kernel(M, lanes):
    assert sweep_kernel("lorenz", M, fwd_lanes=lanes) == "fwd_kernel<op=6, lanes=%d, lazy>" % lanes
