"""Posterior summaries of the accepted paths on the device (dmt_path_moments_add / dmt_get_path_moments / dmt_get_pset_path_moments,
host.PathMoments): the Welford update restated in NumPy bit for bit through blocking sweeps whose accepted buffers differ per chain
and interval, the pooled per-data-set moments and R-hat against the formulas of include/dmt.h, a known answer, the exact smoothing
distribution of a linear target, checkpoints, errors and heterogeneous ensembles."""
import numpy as np
import pytest

import dmt_b200
from dmt_b200 import _lib, configs, hetero
from dmt_b200 import host as H
from harness import make_ctx, rel_err
from test_gpu_statistics import rts_smoother

pytestmark = [pytest.mark.gpu, pytest.mark.own_lanes]   # the moments kernel does not depend on the forward kernel's lanes


def recordings_of(prob):
    return dict(theta=prob.theta, L=prob.L, Sigma=prob.Sigma, v=prob.v, x0=prob.x0, xbar=prob.xbar)


def blocking_ctx(M=64, seed=7):
    """Lorenz, K = 40 intervals of 50 steps (not a multiple of 4: padded tiles), two staggered layouts + a whole-path layout for
    init_paths!, lazy noise"""
    K = 40
    layouts = configs.blocking_layouts(K, 20, 0.9) + [([(0, K - 1)], 0.0)]
    prob = configs.make_problem("lorenz", M, K=K, obs_dt=0.1, dt=0.1 / 50, seed=3, layouts=layouts)
    ctx = make_ctx(prob, seed=seed)
    ctx.recompute_guiding_term(2, _lib.P_ONLY)
    assert ctx.init_paths(2, iter0=900, max_tries=50) == 0
    ctx.set_lazy_noise(True)
    return prob, ctx


def welford_np(xs):
    """include/dmt.h's update in float64 NumPy, one rounding per operation (NumPy does not contract to FMA)"""
    mean, m2 = xs[0].copy(), np.zeros_like(xs[0])
    for n, x in enumerate(xs[1:], start=2):
        w = 1.0 / n
        delta = x - mean
        mean = mean + delta * w
        m2 = m2 + delta * (x - mean)
    return mean, m2


def test_welford_bitwise_through_blocking_sweeps_and_nothing_else_changes():
    """(1) bitwise against the NumPy restatement, per chain and point, also through a repeating, reordered chain selection;
    (2) the same run without accumulation gives bit-identical X, ll, ll° and decisions, and each update is exactly one launch
    (under lazy noise: no W rebuild)"""
    _, a = blocking_ctx()
    _, b = blocking_ctx()
    xs, mixed = [], False
    for it in range(12):
        l = it % 2
        for c in (a, b):
            c.blocking_sweep(l, it); c.accept_reject_path(l, it)
        acc = b.get_last_accept(l)
        assert np.array_equal(a.get_last_accept(l), acc)
        mixed |= bool(acc.any() and not acc.all())
        if it >= 2:
            n0 = _lib.launch_count()
            b.path_moments_add()
            assert _lib.launch_count() - n0 == 1
            xs.append(b.get_X(0))
        for s in (0, 1):
            assert np.array_equal(a.get_ll(l, s), b.get_ll(l, s))
    assert mixed, "no iteration mixed accepted and rejected blocks: the buffer parity was not exercised"
    for s in (0, 1):
        assert np.array_equal(a.get_X(s), b.get_X(s))
    mean, m2, n = b.get_path_moments()
    assert n == len(xs) == 10 == b.moments_count
    want_mean, want_m2 = welford_np(xs)
    assert np.array_equal(mean, want_mean) and np.array_equal(m2, want_m2)
    assert (m2 > 0).mean() > 0.9                                          # the paths really moved
    sel = [5, 0, 63, 5]
    ms, m2s, ns = b.get_path_moments(sel)
    assert ns == n and np.array_equal(ms, want_mean[:, :, sel]) and np.array_equal(m2s, want_m2[:, :, sel])
    a.close(); b.close()


def test_known_answer_rho_one():
    """rho = 1: the proposal is driven by the accepted noise itself, so after one accept every further accepted path is the same
    path: m2 == 0 exactly, mean == the path bit for bit, pooled R-hat NaN (W == 0)"""
    prob = configs.make_problem("lorenz", 64, P=4, K=4, obs_dt=0.1, dt=0.1 / 22, seed=5, rho=1.0)
    ctx = make_ctx(prob, seed=3)
    ctx.recompute_guiding_term(0, _lib.P_ONLY)
    assert ctx.init_paths(0, 0, 20) == 0
    ctx.loglikhd(0, 0, 0)
    ctx.draw_proposal_path(0, 0); ctx.accept_reject_path(0, 0)
    for it in range(1, 6):
        ctx.draw_proposal_path(0, it); ctx.accept_reject_path(0, it)
        ctx.path_moments_add()
    X = ctx.get_X(0)
    mean, m2, n = ctx.get_path_moments()
    assert n == 5 and np.array_equal(mean, X) and np.all(m2 == 0.0)
    pm, pv, rh = ctx.get_pset_path_moments()
    assert np.all(np.isnan(rh))
    ctx.close()


def pooled_np(mean, m2, n, pset, P):
    out = [np.empty(mean.shape[:2] + (P,)) for _ in range(3)]
    for q in range(P):
        ch = np.flatnonzero(pset == q)
        m = ch.size
        mu = mean[:, :, ch]
        mbar = mu.sum(-1) / m
        sdev = ((mu - mbar[..., None]) ** 2).sum(-1)
        sm2 = m2[:, :, ch].sum(-1)
        W = sm2 / (m * (n - 1.0)) if n > 1 else np.full_like(sm2, np.nan)
        B = n * sdev / (m - 1)
        with np.errstate(invalid="ignore", divide="ignore"):
            rh = np.sqrt((((n - 1.0) / n) * W + B / n) / W)
        rh[W == 0] = np.nan
        out[0][..., q], out[1][..., q], out[2][..., q] = mbar, (sm2 / n + sdev) / m, rh
    return out


@pytest.mark.parametrize("P", [4, 1])
def test_pooled_moments_match_the_formulas(P):
    M = 64
    prob = configs.make_problem("lorenz", M, P=P, K=6, obs_dt=0.1, dt=0.1 / 30, seed=8, rho=0.9)
    ctx = make_ctx(prob, seed=4)
    ctx.recompute_guiding_term(0, _lib.P_ONLY)
    assert ctx.init_paths(0, 0, 20) == 0
    ctx.loglikhd(0, 0, 0)
    ctx.draw_proposal_path(0, 0); ctx.accept_reject_path(0, 0)
    ctx.path_moments_add()
    r1 = ctx.get_pset_path_moments()
    assert np.all(np.isnan(r1[2]))                                        # count < 2: R-hat undefined
    for it in range(1, 8):
        ctx.draw_proposal_path(0, it); ctx.accept_reject_path(0, it)
        ctx.path_moments_add()
    mean, m2, n = ctx.get_path_moments()
    pset = prob.pset_of_chain if prob.pset_of_chain is not None else np.zeros(M, int)
    if P == 4:
        assert np.array_equal(pset[:8], [0, 1, 2, 3, 0, 1, 2, 3])      # interleaved map
    want = pooled_np(mean, m2, n, pset, P)
    got = ctx.get_pset_path_moments()
    assert rel_err(got[0], want[0]) < 1e-12
    assert rel_err(got[1], want[1]) < 1e-10
    assert rel_err(got[2], want[2]) < 1e-10
    assert np.all(np.isnan(got[2][0])) and np.all(np.isfinite(got[2][1:]))   # NaN exactly at the known start point
    again = ctx.get_pset_path_moments()
    assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(got, again))
    ctx.close()


def test_linear_target_pooled_moments_are_the_smoothing_distribution():
    """OU target equal to its auxiliary law (test_gpu_statistics): the guided proposal is exact, every pCN move is accepted and
    init_paths! already draws from the smoothing distribution, so all chains are stationary from the first iteration.  The pooled
    mean / variance must then match the Kalman / RTS smoother up to the O(dt) Euler bias plus Monte Carlo error (tolerances of
    test_gpu_statistics, which uses one draw per chain; here there are n per chain).  R-hat: for a path affine in the noise, pCN
    with rho makes every coordinate an AR(1) with coefficient rho, integrated autocorrelation time tau = (1 + rho) / (1 - rho) = 3;
    with stationary starts R-hat^2 = (n-1)/n + B/(n W) ~ 1 + (tau - 1)/n = 1.007 at n = 300, i.e. R-hat ~ 1.003 (the Monte Carlo
    error of B over 4096 chains is ~2 % of the B/(nW) term), well below 1.01."""
    M, K, n_it = 4096, 4, 300
    prob = configs.make_problem("ou2", M, P=1, K=K, dt=0.002, seed=4, rho=0.5)
    th = prob.theta
    Bm = th[:4].reshape(2, 2); beta = th[4:6]; a = np.diag(th[6:8] ** 2)
    ctx = make_ctx(prob, seed=12, ll_hist_len=8)
    ctx.recompute_guiding_term(0, _lib.P_ONLY)
    assert ctx.init_paths(0, 0, 5) == 0
    ctx.loglikhd(0, 0, 0)
    for it in range(n_it):
        ctx.draw_proposal_path(0, it); ctx.accept_reject_path(0, it)
        ctx.path_moments_add()
    assert ctx.get_accept_history(0, 0, 7).all()                          # exact proposals are always accepted
    mean, var, rhat = ctx.get_pset_path_moments()
    pt0 = np.concatenate([[0], np.cumsum(prob.n_pts)])
    times, idx_of, obs_idx = [0.0], {}, []
    for k in range(K):
        tk = prob.tt[pt0[k]:pt0[k + 1]]
        for j in range(1, len(tk)):
            times.append(tk[j]); idx_of[(k, j)] = len(times) - 1
        obs_idx.append(len(times) - 1)
    ms, Ps = rts_smoother(Bm, beta, a, prob.x0[:, 0], np.array(times), obs_idx, prob.L, prob.Sigma, [prob.v[k, :, 0] for k in range(K)])
    for (k, j) in [(0, 20), (1, 25), (2, 10), (3, 40), (3, 50)]:
        g, p = idx_of[(k, j)], pt0[k] + j
        sd = np.sqrt(np.diag(Ps[g]))
        assert np.all(np.abs(mean[p, :, 0] - ms[g]) < 5 * sd / np.sqrt(M) + 0.02 * sd), (k, j, mean[p, :, 0], ms[g])
        assert np.all(np.abs(np.sqrt(var[p, :, 0]) - sd) < 0.06 * sd), (k, j, np.sqrt(var[p, :, 0]), sd)
    assert np.all(np.isnan(rhat[0]))                                      # the known start point
    interior = rhat[1:]
    assert np.all(np.isfinite(interior)) and interior.max() < 1.01 and interior.min() > 0.99, (interior.min(), interior.max())
    ctx.close()


def test_checkpoint_resume_carries_the_moments(tmp_path):
    """N updates, save_state, a fresh ensemble, load_state, N more updates == 2N uninterrupted updates, bit for bit"""
    K, N = 8, 4
    layouts = [([(0, 2), (3, 5), (6, 7)], 0.8), ([(0, 3), (4, 7)], 0.7)]
    prob = configs.make_problem("lorenz", 40, K=K, dt=0.01, seed=9, layouts=layouts)

    def fresh():
        se = H.SamplingEnsemble(prob.model, recordings_of(prob), (prob.n_pts, prob.tt), seed=5, two_sided_laws=False)
        se.init_paths()
        return se, [H.BlockEnsemble(se, r, rho, 0) for r, rho in layouts], H.PathMoments(se, every=2, start=1)

    def sweeps(bes, pm, its):
        for i in its:
            for be in bes:
                H.blocking_sweep(be, i)
                H.accept_reject_proposal_path(be, i)
            pm(i)

    se, bes, pm = fresh()
    sweeps(bes, pm, range(2 * N))
    assert pm.count == N
    ck = str(tmp_path / "state.npz")
    H.save_state(se, ck, bes)
    sweeps(bes, pm, range(2 * N, 4 * N))
    assert pm.count == 2 * N
    want = se.ctx.get_path_moments() + (se.ctx.get_X(0),)
    mean_c, var_c = pm.chain_moments([3, 1])                              # var = m2 / count
    assert np.array_equal(mean_c, want[0][:, :, [3, 1]]) and np.array_equal(var_c, want[1][:, :, [3, 1]] / (2 * N))
    se.ctx.close()
    se2, bes2, pm2 = fresh()
    H.load_state(se2, ck, bes2)
    assert pm2.count == N
    sweeps(bes2, pm2, range(2 * N, 4 * N))
    got = se2.ctx.get_path_moments() + (se2.ctx.get_X(0),)
    assert got[2] == want[2] == 2 * N
    for x, y in zip((got[0], got[1], got[3]), (want[0], want[1], want[3])):
        assert np.array_equal(x, y)
    # a checkpoint without moments resets them
    se2.ctx.close()
    se3, bes3, pm3 = fresh()
    sweeps(bes3, pm3, range(2))
    assert pm3.count == 1
    ck0 = str(tmp_path / "plain.npz")
    se3.ctx.path_moments_reset(); H.save_state(se3, ck0, bes3)
    se3.ctx.path_moments_add()
    H.load_state(se3, ck0, bes3)
    assert pm3.count == 0 and "moments_count" not in np.load(ck0)
    pm3(3)
    assert pm3.count == 1
    pm3.reset()
    assert pm3.count == 0
    with pytest.raises(dmt_b200.DmtError) as e:
        se3.ctx.get_path_moments()
    assert e.value.code == 3
    se3.ctx.close()


def test_errors():
    prob = configs.make_problem("fhn", 8, K=3, dt=0.01, seed=1)
    ctx = make_ctx(prob)
    ctx.recompute_guiding_term(0, _lib.P_ONLY)
    assert ctx.init_paths(0, 0, 20) == 0
    for f in (ctx.get_path_moments, ctx.get_pset_path_moments):
        with pytest.raises(dmt_b200.DmtError) as e:
            f()
        assert e.value.code == 3                                          # DMT_ERR_STATE: nothing accumulated
    ctx.path_moments_add()
    for bad in ([8], [0, -1]):
        with pytest.raises(dmt_b200.DmtError) as e:
            ctx.get_path_moments(bad)
        assert e.value.code == 1                                          # DMT_ERR_ARG
    mean, m2, n = ctx.get_path_moments()
    with pytest.raises(dmt_b200.DmtError) as e:
        ctx.set_path_moments(mean, m2, 0)
    assert e.value.code == 1
    ctx.set_path_moments(mean + 1.0, m2, 3)                               # set -> get round-trips exactly
    m_b, m2_b, n_b = ctx.get_path_moments()
    assert n_b == 3 and np.array_equal(m_b, mean + 1.0) and np.array_equal(m2_b, m2)
    ctx.close()


def _rec_list(prob, model):
    return [dict(model=model, theta=prob.theta, L=prob.L, Sigma=prob.Sigma, v=prob.v[:, :, c], x0=prob.x0[:, c],
                 xbar=prob.xbar[:, :, c], tts=(prob.n_pts, prob.tt)) for c in range(prob.M)]


def test_heterogeneous_chain_moments_follow_the_buckets():
    pa = configs.make_problem("fhn", 3, K=6, dt=0.005, seed=1, rho=0.8)
    pc = configs.make_problem("lorenz", 2, K=5, dt=0.01, seed=3, rho=0.8)
    ra, rc = _rec_list(pa, _lib.FHN), _rec_list(pc, _lib.LORENZ)
    recs = [ra[0], rc[0], ra[1], rc[1], ra[2]]
    he = hetero.HeterogeneousEnsemble(recs, seed=17, two_sided_laws=False)
    he.init_paths()
    hbe = hetero.HeterogeneousBlockEnsemble(he, lambda K: [(0, K // 2 - 1), (K // 2, K - 1)], 0.8, 0)
    for i in range(4):
        hetero.blocking_sweep(hbe, i)
        hetero.accept_reject_proposal_path(hbe, i)
        hetero.path_moments_add(he)
    per_rec = hetero.chain_moments(he)
    assert len(per_rec) == 5 and per_rec[1][0].shape[1] == 3 and per_rec[0][0].shape[1] == 2
    for r in range(5):
        b, i = he.where[r]
        mean, var = H.PathMoments(he.buckets[b]).chain_moments([i])
        assert np.array_equal(per_rec[r][0], mean[:, :, 0]) and np.array_equal(per_rec[r][1], var[:, :, 0])
    assert all(np.all(v >= 0) for _, v in per_rec) and np.any(per_rec[1][1] > 0)
    he.close()
