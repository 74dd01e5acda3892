"""The C ABI orders every copy and fill on a stream it owns: the context's compute stream, or the copy stream of the
asynchronous read-backs.  Nothing goes on the legacy default stream, which a context's non-blocking stream does not
order against, and nothing waits for the whole device, which would also wait for other contexts on the same GPU."""
import os
import re

import numpy as np
import pytest

from dmt_b200 import _lib, configs
from harness import make_ctx

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "diffusionmcmctools.jl_b200", "csrc", "dmt_api.cu")


def source():
    return open(SRC).read()


def call_args(src, name):
    """The top-level arguments of every call of `name` in the code (comments stripped)."""
    code = re.sub(r"//[^\n]*", "", src)
    calls = []
    for m in re.finditer(r"\b%s\s*\(" % name, code):
        depth, i, args, start = 1, m.end(), [], m.end()
        while depth:
            ch = code[i]
            if ch in "([{":
                depth += 1
            elif ch in ")]}":
                depth -= 1
            elif ch == "," and depth == 1:
                args.append(code[start:i].strip())
                start = i + 1
            i += 1
        args.append(code[start:i - 1].strip())
        calls.append(args)
    return calls


def test_no_legacy_stream_and_no_device_wide_sync():
    src = source()
    for banned in ("cudaMemcpy(", "cudaMemset(", "cudaStreamLegacy", "cudaDeviceSynchronize"):
        assert banned not in src, banned


def test_every_async_copy_and_fill_names_its_stream():
    src = source()
    n = 0
    for name, nargs in (("cudaMemcpyAsync", 5), ("cudaMemsetAsync", 4)):
        for args in call_args(src, name):
            assert len(args) == nargs, (name, args)
            assert re.fullmatch(r"(\w+(->|\.))*(stream|copy_stream)", args[-1]), (name, args)
            n += 1
    assert n >= 50


def init_problem(K=6):
    return configs.make_problem("lorenz", 64, K=K, dt=0.01, seed=1, layouts=[([(0, 2), (3, 5)], 0.8), ([(0, K - 1)], 0.0)])


@pytest.mark.gpu
def test_a_registered_layout_is_ready_for_the_next_call():
    """The next call after dmt_set_blocks sees everything it uploaded: ll = -Inf (the Block constructor, src/block.jl:74),
    the broadcast ρ, and the block ranges that the guiding term and init_paths read.  make_ctx registers the init layout
    [(0, K-1)] last; it leaves the PPb tile map as it was."""
    prob = init_problem()
    ctx = make_ctx(prob, seed=42)
    for side in (0, 1):
        assert np.isneginf(ctx.get_ll(1, side)).all()
    assert np.array_equal(ctx.get_rho_chains(1), np.zeros((1, prob.M)))
    ctx.set_blocks(0, [(0, 2), (3, 5)], [0.3, 0.7])          # re-registered, same shape
    assert np.isneginf(ctx.get_ll(0, 1)).all()
    assert np.array_equal(ctx.get_rho_chains(0), np.repeat([[0.3], [0.7]], prob.M, axis=1))
    ctx.close()

    paths = []
    for sync in (False, True):
        ctx = make_ctx(prob, seed=42)
        if sync:
            ctx.sync()
        ctx.recompute_guiding_term(1, _lib.P_ONLY)
        n_failed = ctx.init_paths(1, 0, 20)
        paths.append((n_failed, ctx.get_X(0), ctx.get_W(0)))
        ctx.close()
    (f0, X0, W0), (f1, X1, W1) = paths
    assert f0 == f1 and np.array_equal(X0, X1) and np.array_equal(W0, W1)
