"""Heterogeneous ensembles (SURVEY §8f item 4).

The reference's SamplingEnsemble takes one auxiliary-law vector, one recording and one time grid PER RECORDING
(/root/reference/src/sampling_ensemble.jl:26-38), so recordings of one ensemble may differ in the number of observations, in the
time grids and even in the diffusion model.  A device context holds recordings that share all three (one kernel launch covers them
with uniform control flow), so a heterogeneous ensemble is bucketed here, on the host, into homogeneous SamplingEnsembles — one
context and one CUDA stream each, all on the same GPU — and every BlockEnsemble call fans out over the buckets.  Launches are
asynchronous, so small buckets overlap on the device; scalars (fetch_ll) are summed over buckets.
"""
import numpy as np

from . import _lib
from . import host as H
from .param_names import ParamNamesAllObs


def _bucket_key(rec):
    n_pts, tt = rec["tts"]
    return (int(rec["model"]), tuple(int(n) for n in n_pts), np.asarray(tt, dtype=np.float64).tobytes(),
            np.asarray(rec["L"], dtype=np.float64).tobytes(), np.asarray(rec["Sigma"], dtype=np.float64).tobytes())


def bucket_recordings(recordings):
    """recording ids grouped by (model, time grid, observation operator), buckets in order of first appearance"""
    keys, members = {}, []
    for r, rec in enumerate(recordings):
        k = _bucket_key(rec)
        if k not in keys:
            keys[k] = len(members)
            members.append([])
        members[keys[k]].append(r)
    return members


class HeterogeneousEnsemble:
    """recordings: list of dicts, one per recording, with
         model (id), theta [npar], L [m, d], Sigma [m, m], v [K, m], x0 [d], xbar [K, d], tts = (n_pts [K], tt [sum n_pts]).
    Recordings with equal (model, time grid, observation operator) share a bucket; `members[b]` lists the recording ids of
    bucket b in ascending order and `where[r] = (bucket, index inside it)`."""

    def __init__(self, recordings, *, seed=0, device=0, two_sided_laws=True, max_layouts=8, artificial_noise=1e-11):
        self.members = bucket_recordings(recordings)
        self.where = {r: (b, i) for b, m in enumerate(self.members) for i, r in enumerate(m)}
        self.buckets = []
        off = 0
        for m in self.members:
            r0 = recordings[m[0]]
            st = lambda name: np.stack([np.asarray(recordings[r][name], dtype=np.float64) for r in m], axis=-1)
            data = dict(theta=st("theta"), L=r0["L"], Sigma=r0["Sigma"], v=st("v"), x0=st("x0"), xbar=st("xbar"))
            se = H.SamplingEnsemble(r0["model"], data, r0["tts"], seed=seed, device=device, two_sided_laws=two_sided_laws,
                                    max_layouts=max_layouts, artificial_noise=artificial_noise, chain_offset_base=off)
            off += len(m)      # every recording keeps its own random stream whatever the bucketing
            self.buckets.append(se)
        self.M_total = len(recordings)

    def init_paths(self, **kw):
        for se in self.buckets:
            se.init_paths(**kw)

    def num_recordings(self):
        return self.M_total

    def close(self):
        for se in self.buckets:
            se.ctx.close()


class HeterogeneousBlockEnsemble:
    """BlockEnsemble over a HeterogeneousEnsemble.  `block_ranges` is either one list of ranges per bucket or a callable
    K -> ranges (the number of observations differs between buckets); rho as for BlockEnsemble."""

    def __init__(self, he, block_ranges, rho=0.0, ll_hist_len=0):
        self.he = he
        self.parts = []
        for b, se in enumerate(he.buckets):
            rr = block_ranges(se.ctx.K) if callable(block_ranges) else block_ranges[b]
            self.parts.append(H.BlockEnsemble(se, rr, rho, ll_hist_len))

    def num_recordings(self):
        return self.he.M_total


def _fan(fn):
    def f(hbe, *a, **kw):
        return [fn(be, *a, **kw) for be in hbe.parts]
    f.__name__ = fn.__name__
    f.__doc__ = "%s over every bucket of a HeterogeneousBlockEnsemble (host.%s)" % (fn.__name__, fn.__name__)
    return f


draw_proposal_path = _fan(H.draw_proposal_path)
accept_reject_proposal_path = _fan(H.accept_reject_proposal_path)
swap_paths, swap_XX, swap_WW, swap_PP, swap_ll = (_fan(f) for f in (H.swap_paths, H.swap_XX, H.swap_WW, H.swap_PP, H.swap_ll))
loglikhd, loglikhd_o = _fan(H.loglikhd), _fan(H.loglikhd_o)
save_ll = _fan(H.save_ll)
set_obs = _fan(H.set_obs)
recompute_guiding_term = _fan(H.recompute_guiding_term)
find_W_for_X = _fan(H.find_W_for_X)
blocking_sweep = _fan(H.blocking_sweep)
enable_guiding_cache = _fan(H.enable_guiding_cache)
accpt_rate = _fan(H.accpt_rate)             # one vector (per block) per bucket: layouts differ between buckets
enable_rho_adaptation, adapt_rho, disable_rho_adaptation = (_fan(f) for f in (H.enable_rho_adaptation, H.adapt_rho, H.disable_rho_adaptation))


def rho_chains(hbe):
    """per recording (global order): ρ [n_blocks] of each of its blocks (bb.ρ, src/biblock.jl:46; block counts differ between buckets)"""
    per_bucket = [be.rho_chains for be in hbe.parts]
    return [per_bucket[b][:, i].copy() for b, i in (hbe.he.where[r] for r in range(hbe.he.M_total))]


def set_rho_chains(hbe, rho):
    """rho: one value for every block of every recording, or one entry per recording in global order, each a value or [n_blocks]"""
    if np.ndim(rho) == 0:
        for be in hbe.parts:
            H.set_rho_chains(be, rho)
        return
    if len(rho) != hbe.he.M_total:
        raise ValueError("need one ρ entry per recording (%d), got %d" % (hbe.he.M_total, len(rho)))
    for be, m in zip(hbe.parts, hbe.he.members):
        H.set_rho_chains(be, np.stack([np.broadcast_to(np.asarray(rho[r], dtype=np.float64), (be.n_blocks,)) for r in m], axis=1))


def fetch_ll(hbe):
    """Σ over buckets of fetch_ll (src/block_ensemble.jl:140): bucket order is fixed, so the sum is reproducible"""
    return float(sum(H.fetch_ll(be) for be in hbe.parts))


def fetch_ll_o(hbe):
    return float(sum(H.fetch_ll_o(be) for be in hbe.parts))


def set_proposal_law(hbe, theta_o, pnames, critical_change=None, skip=0):
    """set_proposal_law!(be, θ°, pnames, crit) with ONE θ° for the whole ensemble and one ParamNamesAllObs (or pair list) per
    bucket — recordings of different models map the shared θ° onto different parameter vectors."""
    for be, pn in zip(hbe.parts, pnames):
        H.set_proposal_law(be, theta_o, pn, critical_change, skip)


def param_names(hbe, theta_names, param_depend_rev, obs_depend_rev=None):
    """ParamNamesAllObs(be, θnames, all_obs) per bucket from per-RECORDING dependency lists in global recording order"""
    out = []
    for be, m in zip(hbe.parts, hbe.he.members):
        out.append(ParamNamesAllObs.build(be, theta_names, [param_depend_rev[r] for r in m],
                                          None if obs_depend_rev is None else [obs_depend_rev[r] for r in m]))
    return out


def paths(he, side=0):
    """per recording (global order): X [n_points, d] of the accepted (0) or proposal (1) side"""
    per_bucket = [se.ctx.get_X(side) for se in he.buckets]
    return [per_bucket[b][:, :, i] for b, i in (he.where[r] for r in range(he.M_total))]


def path_moments_add(he):
    """add the current accepted paths of every recording to its path moments (host.PathMoments), one launch per bucket"""
    for se in he.buckets:
        se.ctx.path_moments_add()


def chain_moments(he):
    """per recording (global order): (mean [n_points, d], var [n_points, d]) of its accepted path, var = m2 / count"""
    per_bucket = []
    for se in he.buckets:
        mean, m2, n = se.ctx.get_path_moments()
        per_bucket.append((mean, m2 / n))
    return [(per_bucket[b][0][:, :, i], per_bucket[b][1][:, :, i]) for b, i in (he.where[r] for r in range(he.M_total))]
