"""Host-side mirror of the DiffusionMCMCTools.jl API over the device library (libdmt.so).

Same names, argument meaning and call order as the reference (file:line into /root/reference/), with Julia's `f!` written
`f` and `°` written `_o`.  Containers live on the GPU as structure-of-arrays; `Block`/`BiBlock` are index ranges; every
method below is ONE batched kernel launch over all recordings x blocks instead of the reference's serial broadcasts
(src/block_ensemble.jl:50 -> src/block_collection.jl:46 -> src/biblock.jl:80-99).

Julia has no toolchain in this image, so this Python layer plays the role of the Julia glue in tests; the actual glue
(julia/DiffusionMCMCToolsB200.jl) makes the same ccalls.

Parameter-name translation (src/param_names_collections.jl) and the parameter proposal / prior / accept logic stay on the
host (BASELINE.json north_star): `set_proposal_law` takes the already-translated pairs `pnames = [(i_theta°, j_model), ...]`.
"""
import numpy as np

from . import _lib
from .param_names import ParamNamesAllObs

P_only, Po_only = "P_only", "P°_only"  # Val(:P_only), Val(:P°_only)  (src/DiffusionMCMCTools.jl:9-10)


def shard_slice(n_total, rank, world):
    """one contiguous slice of chains per GPU (SURVEY §8e)"""
    base, rem = divmod(n_total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class SamplingEnsemble:
    """SamplingEnsemble(aux_laws, recordings, tts, ...)  (src/sampling_ensemble.jl:17-41) — all recordings of one model on one
    GPU.  `recordings` carries what ObservationSchemes' recordings + GuidedProposals' aux laws carry:
        theta [npar] or [npar, P]; L [m, d]; Sigma [m, m]; v [K, m, P]; x0 [d, M];
        xbar [K, d, P] (Jacobian-linearised auxiliary laws, evaluated on the device)  or  aux = (B [K,d,d,P], beta [K,d,P], atil [K,d,d,P]).
    tts = (n_pts [K], tt [sum n_pts]) is OBS.setup_time_grids' output.  With (rank, world) given, this process keeps the
    contiguous chain slice of `rank` (chains are independent: src/block_ensemble.jl:63-67)."""

    def __init__(self, model, recordings, tts, *, aux_laws_blocking=None, artificial_noise=1e-11, device=0, seed=0, two_sided_laws=True,
                 max_layouts=8, rank=0, world=1, pset_of_chain=None, chain_offset_base=0):
        n_pts, tt = tts
        x0 = np.asarray(recordings["x0"], dtype=np.float64)
        M_tot = x0.shape[1]
        v = np.asarray(recordings["v"], dtype=np.float64)
        P_tot = v.shape[2]
        self.rank, self.world = rank, world
        lo, hi = shard_slice(M_tot, rank, world)
        if P_tot == M_tot:
            plo, phi = lo, hi
        else:
            if world > 1:
                raise ValueError("sharding needs one parameter/data set per recording (P == M)")
            plo, phi = 0, P_tot
        self.chain_lo, self.chain_hi, self.M_total = lo, hi, M_tot
        self.model = model
        self.theta = np.asarray(recordings["theta"], dtype=np.float64)
        if self.theta.ndim == 1:
            self.theta = np.repeat(self.theta[:, None], phi - plo, axis=1)
        else:
            self.theta = self.theta[:, plo:phi].copy()
        self.theta_o = self.theta.copy()
        self.xbar = None
        self.obs_param_hook = None            # (per-recording {interval: ((i_theta, i_obs), ...)}, θ°) -> (L, Sigma, v) of the proposal side
        L, Sigma = recordings["L"], recordings["Sigma"]
        self.ctx = _lib.Ctx(model, n_pts, tt, hi - lo, phi - plo, obs_dim=np.asarray(L).shape[-2] if np.asarray(L).ndim == 2 else np.asarray(L).shape[1],
                            device=device, two_sided_laws=two_sided_laws, n_layouts=max_layouts, chain_offset=chain_offset_base + lo, seed=seed,
                            artificial_noise=artificial_noise, pset_of_chain=pset_of_chain)
        self.two_sided = two_sided_laws
        self._next_layout = 0
        self._init_layout = None
        sides = (0, 1) if two_sided_laws else (0,)
        for s in sides:
            self.ctx.set_params(self.theta, side=s, stores=3)
            self.ctx.set_obs(L, Sigma, v[:, :, plo:phi], side=s)
        if "xbar" in recordings:
            self.xbar = np.asarray(recordings["xbar"], dtype=np.float64)[:, :, plo:phi].copy()
            self.xbar_blocking = self.xbar if aux_laws_blocking is None else np.asarray(aux_laws_blocking)[:, :, plo:phi].copy()
            for s in sides:
                self.ctx.set_aux_linearised(self.xbar, side=s, store=_lib.STORE_PP)
                self.ctx.set_aux_linearised(self.xbar_blocking, side=s, store=_lib.STORE_PPB)
        else:
            B, beta, atil = recordings["aux"]
            Bb, betab, atilb = aux_laws_blocking if aux_laws_blocking is not None else recordings["aux"]
            for s in sides:
                self.ctx.set_aux(B, beta, atil, side=s, store=_lib.STORE_PP)
                self.ctx.set_aux(Bb, betab, atilb, side=s, store=_lib.STORE_PPB)
        self.ctx.set_start(x0[:, lo:hi])

    def init_paths(self, iter0=2 ** 24, max_tries=100):
        """SamplingUnit ctor's init_paths! + u° = deepcopy(u)  (src/sampling_unit.jl:70,83-87; src/sampling_pair.jl:51)"""
        if self._init_layout is None:
            self._init_layout = self._alloc_layout()
            self.ctx.set_blocks(self._init_layout, [(0, self.ctx.K - 1)], 0.0, ll_hist_len=0)
        self.ctx.recompute_guiding_term(self._init_layout, _lib.P_ONLY)
        nf = self.ctx.init_paths(self._init_layout, iter0, max_tries)
        if nf:
            raise RuntimeError("init_paths!: %d recordings still fail after %d tries" % (nf, max_tries))

    def _alloc_layout(self):
        if self._next_layout >= self.ctx.n_layouts:
            raise RuntimeError("more block layouts than max_layouts=%d" % self.ctx.n_layouts)
        self._next_layout += 1
        return self._next_layout - 1

    def comm_init(self, uid):
        """join the NCCL communicator used for the small ll / accept-count allreduce"""
        self.ctx.comm_init(self.world, self.rank, uid)
        self._has_comm = True

    def p2p_init(self):
        """map every rank's exchange buffer (CUDA IPC) so that the stats all-reduce is the library's own one-shot kernel over
        NVLink peer memory instead of a NCCL call; the 64-byte handles travel through the default torch.distributed group"""
        import torch
        import torch.distributed as dist
        mine = torch.from_numpy(self.ctx.p2p_export().copy())
        if dist.get_backend() == "nccl":
            mine = mine.cuda()
        allh = [torch.empty_like(mine) for _ in range(self.world)]
        dist.all_gather(allh, mine)
        self.ctx.p2p_init(self.world, self.rank, np.stack([h.cpu().numpy() for h in allh]))
        self._has_comm = True

    def num_recordings(self):  # OBS.num_recordings(se)  src/sampling_ensemble.jl:46
        return self.M_total


class _BlockSide:
    """bb.b / bb.b° of one (recording, block) — a `Block` (src/block.jl:17-71) as a view into the device ensemble: XX, WW, ll,
    ll_history are read on demand (a few KB through dmt_get_X_chains / dmt_get_W_chains), nothing is cached on the host."""

    def __init__(self, be, rec, blk, side):
        self._be, self._rec, self._blk, self._side = be, rec, blk, side

    @property
    def ll(self):
        return float(self._be.ctx.get_ll(self._be.layout, self._side)[self._blk, self._rec])

    @property
    def ll_history(self):
        return self._be.ctx.get_ll_history(self._be.layout, self._side, 0, self._be.ll_hist_len - 1)[:, self._blk, self._rec]

    @property
    def XX(self):
        """the block's paths, one (t [n_k], x [n_k, d]) pair per observation interval — b.XX (src/block.jl:65)"""
        ctx, (i0, i1) = self._be.ctx, self._be.ranges[self._blk]
        X = ctx.get_X_chains([self._rec], self._side)[:, :, 0]
        return [(ctx.tt[ctx.pt0[k]:ctx.pt0[k + 1]].copy(), X[ctx.pt0[k]:ctx.pt0[k + 1]].copy()) for k in range(i0, i1 + 1)]

    @property
    def WW(self):
        """the block's driving noise as the reference stores it: per interval a Wiener PATH starting at 0 (cumulative sum of the
        library's increments) on the interval's time grid — b.WW (src/block.jl:64)"""
        ctx, (i0, i1) = self._be.ctx, self._be.ranges[self._blk]
        dW = ctx.get_W_chains([self._rec], self._side)[:, :, 0]
        out = []
        for k in range(i0, i1 + 1):
            inc = dW[ctx.step0[k]:ctx.step0[k + 1]]
            out.append((ctx.tt[ctx.pt0[k]:ctx.pt0[k + 1]].copy(), np.concatenate([np.zeros((1, ctx.dw)), np.cumsum(inc, axis=0)])))
        return out


class BiBlockView:
    """`BiBlock` (src/biblock.jl:17-62) of one recording: bb.b, bb.b°, bb.ρ, bb.accpt_history and the BiBlock-level methods that act on
    ONE block of ONE recording.  The numerical calls (draw_proposal_path!, accept_reject_proposal_path!, loglikhd!, ...) are batched
    over all recordings and blocks on the device — call them on the BlockEnsemble; here are the ones that make sense per block."""

    def __init__(self, be, rec, blk):
        self.b, self.b_o = _BlockSide(be, rec, blk, 0), _BlockSide(be, rec, blk, 1)
        self._be, self._rec, self._blk = be, rec, blk

    @property
    def rho(self):
        """bb.ρ (src/biblock.jl:46): the pCN memory of this block of this recording, read from the device"""
        return float(self._be.ctx.get_rho_chains(self._be.layout)[self._blk, self._rec])

    @rho.setter
    def rho(self, value):
        """sets this (recording, block) entry only; on a layout that adapts ρ the adaptation restarts from the new values"""
        ctx, lay = self._be.ctx, self._be.layout
        r = ctx.get_rho_chains(lay)
        r[self._blk, self._rec] = float(value)
        ctx.set_rho_chains(lay, r)

    @property
    def accpt_history(self):
        return self._be.ctx.get_accept_history(self._be.layout, 0, self._be.ll_hist_len - 1)[:, self._blk, self._rec]

    def _mask(self):
        m = np.zeros((self._be.n_blocks, self._be.ctx.M), dtype=np.uint8)
        m[self._blk, self._rec] = 1
        return m

    # swap_XX!(bb) ... swap_paths!(bb)  src/biblock.jl:148-209
    def swap_XX(self):
        self._be.ctx.swap_blocks(self._be.layout, _lib.SWAP_XX, self._mask())

    def swap_WW(self):
        self._be.ctx.swap_blocks(self._be.layout, _lib.SWAP_WW, self._mask())

    def swap_paths(self):
        self._be.ctx.swap_blocks(self._be.layout, _lib.SWAP_XX | _lib.SWAP_WW, self._mask())

    def swap_ll(self):
        self._be.ctx.swap_blocks(self._be.layout, _lib.SWAP_LL, self._mask())

    def swap_PP(self):
        """(needs one parameter set per recording; the host copy of θ stays with the ensemble — see swap_PP(be, mask))"""
        self._be.ctx.swap_blocks(self._be.layout, _lib.SWAP_PP, self._mask())

    def set_accepted(self, i, v):
        """set_accepted!(bb, i, v)  src/biblock.jl:130-135"""
        ctx, lay = self._be.ctx, self._be.layout
        a = ctx.get_accept_history(lay, i, i)[0]
        a[self._blk, self._rec] = bool(v)
        ctx.set_accepted(lay, i, a)

    def set_ll(self, i, v, side=0):
        """set_ll!(bb.b, i, v)  src/block.jl:82-86"""
        ctx, lay = self._be.ctx, self._be.layout
        h = ctx.get_ll_history(lay, side, i, i)[0]
        h[self._blk, self._rec] = float(v)
        ctx.set_ll_history(lay, side, i, h)

    def ll_of_accepted(self, i):
        """ll_of_accepted(bb, i)  src/biblock.jl:218-225"""
        return float((self.b_o if self.accpt_history[i] else self.b).ll_history[i])

    def accpt_rate(self, rng):
        """accpt_rate(bb, range)  src/biblock.jl:228-232"""
        return float(np.mean(self.accpt_history[rng[0]:rng[-1] + 1]))


class BlockCollectionView:
    """`BlockCollection` (src/block_collection.jl:17-36): all blocks of ONE recording."""

    def __init__(self, be, rec):
        self.blocks = [BiBlockView(be, rec, b) for b in range(be.n_blocks)]
        self._be, self._rec = be, rec

    def _mask(self):
        m = np.zeros(self._be.ctx.M, dtype=np.uint8)
        m[self._rec] = 1
        return m

    # src/block_collection.jl:84-118
    def swap_XX(self):
        self._be.ctx.swap(self._be.layout, _lib.SWAP_XX, self._mask())

    def swap_WW(self):
        self._be.ctx.swap(self._be.layout, _lib.SWAP_WW, self._mask())

    def swap_paths(self):
        self._be.ctx.swap(self._be.layout, _lib.SWAP_XX | _lib.SWAP_WW, self._mask())

    def swap_ll(self):
        self._be.ctx.swap(self._be.layout, _lib.SWAP_LL, self._mask())

    def fetch_ll(self):
        """fetch_ll(bc)  src/block_collection.jl:143: the sum over the recording's blocks"""
        return float(self._be.ctx.get_ll(self._be.layout, 0)[:, self._rec].sum())

    def fetch_ll_o(self):
        return float(self._be.ctx.get_ll(self._be.layout, 1)[:, self._rec].sum())

    def accpt_rate(self, rng):
        """accpt_rate(bc, range)  src/block_collection.jl:175-184: one rate per block"""
        return [bb.accpt_rate(rng) for bb in self.blocks]

    def ll_of_accepted(self, i):
        return [bb.ll_of_accepted(i) for bb in self.blocks]


class BlockEnsemble:
    """BlockEnsemble(se, block_ranges, ρρ, ll_hist_len)  (src/block_ensemble.jl:17-34): the same block ranges for every
    recording; the last range is the terminal block (src/block_collection.jl:29).  Ranges are 0-based inclusive pairs."""

    def __init__(self, se, block_ranges, rho=0.0, ll_hist_len=0):
        self.se, self.ctx = se, se.ctx
        self.ranges = [tuple(r) for r in block_ranges]
        self.n_blocks = len(self.ranges)
        self.rho = np.broadcast_to(np.asarray(rho, dtype=np.float64), (self.n_blocks,)).copy()
        self.ll_hist_len = ll_hist_len
        self.layout = se._alloc_layout()
        self.ctx.set_blocks(self.layout, self.ranges, self.rho, ll_hist_len=ll_hist_len)
        self.rho_adaptation = None    # the settings of enable_rho_adaptation while ρ adapts

    @property
    def rho_chains(self):
        """ρ of every block of every local recording, [n_blocks, M] (bb.ρ of each BiBlock, src/biblock.jl:46)"""
        return self.ctx.get_rho_chains(self.layout)

    @property
    def recordings(self):
        return [BlockCollectionView(self, c) for c in range(self.ctx.M)]

    def num_recordings(self):  # src/block_ensemble.jl:36
        return self.se.M_total


# ---- imputation --------------------------------------------------------------------------------------------------------
def draw_proposal_path(be, mcmciter, Z=None):
    """draw_proposal_path!(be)  src/block_ensemble.jl:50.  `mcmciter` is REQUIRED: with (seed, recording, layout, time tile) it
    is the counter of the generator, so calling twice with the same value reproduces the same innovations.  Layouts may share
    one iteration index (the reference loop does): the layout id is part of the counter."""
    be.ctx.draw_proposal_path(be.layout, mcmciter, Z)


def accept_reject_proposal_path(be, mcmciter, E=None):
    """accept_reject_proposal_path!(be, mcmciter)  src/block_ensemble.jl:63-67 (0-based iteration index)"""
    be.ctx.accept_reject_path(be.layout, mcmciter, E)


# ---- swaps (src/block_ensemble.jl:79-112 -> src/biblock.jl:148-209) -------------------------------------------------
def swap_paths(be, mask=None):
    be.ctx.swap(be.layout, _lib.SWAP_XX | _lib.SWAP_WW, mask)


def swap_XX(be, mask=None):
    be.ctx.swap(be.layout, _lib.SWAP_XX, mask)


def swap_WW(be, mask=None):
    be.ctx.swap(be.layout, _lib.SWAP_WW, mask)


def swap_PP(be, mask=None):
    be.ctx.swap(be.layout, _lib.SWAP_PP, mask)
    if mask is None:
        be.se.theta, be.se.theta_o = be.se.theta_o, be.se.theta
    else:
        m = np.asarray(mask, bool)
        t = be.se.theta[:, m].copy(); be.se.theta[:, m] = be.se.theta_o[:, m]; be.se.theta_o[:, m] = t


def swap_ll(be, mask=None):
    be.ctx.swap(be.layout, _lib.SWAP_LL, mask)


# ---- utility (src/block_ensemble.jl:121-179) ---------------------------------------------------------------------------
def loglikhd(be, skip=0):
    be.ctx.loglikhd(be.layout, _lib.ACCEPTED, skip)


def loglikhd_o(be, skip=0):
    be.ctx.loglikhd(be.layout, _lib.PROPOSAL, skip)


def dist_sum(arr):
    """sum a small float64 vector over all ranks of the default torch.distributed group (gloo: CPU tensor, nccl: GPU tensor)"""
    import torch
    import torch.distributed as dist
    t = torch.from_numpy(np.ascontiguousarray(arr, dtype=np.float64).copy())
    if dist.get_backend() == "nccl":
        t = t.cuda()
    dist.all_reduce(t)
    return t.cpu().numpy()


def _global_stats(be):
    """[sum ll, sum ll°, accept counts...] over ALL recordings: the one small allreduce of the path (SURVEY §8e, C1)"""
    st = be.ctx.allreduce_stats(be.layout)  # NCCL inside libdmt when a communicator was initialised, local sums otherwise
    if be.se.world > 1 and not getattr(be.se, "_has_comm", False):
        st = dist_sum(st)
    return st


def fetch_ll(be):
    """fetch_ll(be) = sum over recordings and blocks of b.ll  (src/block_ensemble.jl:140, src/block_collection.jl:144)"""
    return float(_global_stats(be)[0])


def fetch_ll_o(be):
    return float(_global_stats(be)[1])


def save_ll(be, mcmciter):
    be.ctx.save_ll(be.layout, mcmciter)


def set_ll(be, i, v, side=0):
    """set_ll!(b, i, v): ll_history[i] = v  (src/block.jl:82-86); v broadcasts over [n_blocks, M]"""
    be.ctx.set_ll_history(be.layout, side, i, v)


def set_accepted(be, i, v):
    """set_accepted!(bb, i, v): accpt_history[i] = v  (src/biblock.jl:130-135); v broadcasts over [n_blocks, M]"""
    be.ctx.set_accepted(be.layout, i, v)


def recompute_path(be, skip=0, law_side=_lib.PROPOSAL, noise_side=_lib.ACCEPTED):
    """recompute_path!(b°, b.WW; skip) for every block of every recording (src/block.jl:161-187): the path under the proposal
    law driven by the accepted noise, with its log-likelihood"""
    be.ctx.recompute_path(be.layout, law_side, noise_side, skip)


def ll_of_accepted(be, i):
    """[recording][block] log-likelihood of the path accepted at iteration i  (src/biblock.jl:222-224)"""
    acc = be.ctx.get_accept_history(be.layout, i, i)[0]
    ll = be.ctx.get_ll_history(be.layout, 0, i, i)[0]
    llo = be.ctx.get_ll_history(be.layout, 1, i, i)[0]
    return np.where(acc, llo, ll).T


def accpt_rate(be, rng):
    """acceptance rate per block over the inclusive iteration range, LOCAL recordings  (src/biblock.jl:232)"""
    i0, i1 = rng
    return be.ctx.accept_counts(be.layout, i0, i1) / float((i1 - i0 + 1) * be.ctx.M)


# ---- blocking (src/block_ensemble.jl:192-221) --------------------------------------------------------------------------
def set_obs(be):
    be.ctx.set_artificial_obs(be.layout)


def recompute_guiding_term(be, which=None):
    w = {None: _lib.P_BOTH if be.se.two_sided else _lib.P_ONLY, P_only: _lib.P_ONLY, Po_only: _lib.PO_ONLY}[which]
    be.ctx.recompute_guiding_term(be.layout, w)


def find_W_for_X(be):
    be.ctx.find_W_for_X(be.layout)


def enable_guiding_cache(be, enable=True):
    """Not in the reference: keep the v-independent part of the guiding term between sweeps (include/dmt.h, DESIGN.md §4).
    Use it for smoothing with blocking, where only the blocks' frozen end points change between recompute_guiding_term! calls."""
    be.ctx.enable_guiding_cache(be.layout, enable)


def set_rho_chains(be, rho):
    """bb.ρ of every BiBlock at once (src/biblock.jl:46): `rho` broadcasts to [n_blocks, M_total] over ALL recordings; each rank keeps
    its own slice.  On a layout that adapts ρ the adaptation restarts from the new values."""
    full = np.broadcast_to(np.asarray(rho, dtype=np.float64), (be.n_blocks, be.se.M_total))
    be.ctx.set_rho_chains(be.layout, full[:, be.se.chain_lo:be.se.chain_hi])


def enable_rho_adaptation(be, target=0.234, gamma0=1.0, decay=0.66, window=10, rho_min=0.0, rho_max=0.999):
    """Not in the reference (the tutorials set ρ by hand and watch accpt_rate): adapt every (recording, block)'s ρ toward `target`
    acceptance from its own decisions, on the device.  Call adapt_rho(be) after each accept_reject_proposal_path! during burn-in, then
    disable_rho_adaptation(be): draws taken while ρ adapts are not from a fixed Markov kernel.  The rule is in include/dmt.h."""
    be.ctx.set_rho_adaptation(be.layout, target, gamma0, decay, window, rho_min, rho_max)
    be.rho_adaptation = dict(target=float(target), gamma0=float(gamma0), decay=float(decay), window=int(window),
                             rho_min=float(rho_min), rho_max=float(rho_max))


def adapt_rho(be):
    """one adaptation step from the layout's last accept decisions (one kernel launch, no copy)"""
    be.ctx.adapt_rho(be.layout)


def disable_rho_adaptation(be):
    """freeze ρ at its current values"""
    be.ctx.set_rho_adaptation(be.layout, 0.0)
    be.rho_adaptation = None


def blocking_sweep(be, mcmciter):
    """GP.set_obs!(be); recompute_guiding_term!(be, Val(:P_only)); find_W_for_X!(be); loglikhd!(be); draw_proposal_path!(be)
    (docs/src/tutorials/block_collection/inference_with_blocking.md:52-57) as one library call / three kernel launches."""
    be.ctx.blocking_sweep(be.layout, mcmciter)


# ---- parameters (src/block_ensemble.jl:226-255 -> src/biblock.jl:334-371) -------------------------------------------
def is_critical_update(be, pnames):
    """GP.is_critical_update(be, pnames).  The reference's version reads fields no ParamNames struct has
    (src/biblock.jl:315-317, SURVEY Appendix C.2), so for the bare pair list there is nothing to ask; a ParamNamesAllObs tree
    answers what the docstring there describes (param_names.ParamNamesAllObs.is_critical)."""
    if isinstance(pnames, ParamNamesAllObs):
        return pnames.is_critical()
    raise NotImplementedError("pass critical_change explicitly (as every tutorial does) or a ParamNamesAllObs")


def set_proposal_law(be, theta_o, pnames, critical_change=None, skip=0):
    """set_proposal_law!(be, θ°, pnames, critical_change; skip)  src/block_ensemble.jl:242-255.
    pnames: a ParamNamesAllObs (src/param_names_collections.jl:268-288; each recording may map different entries of θ° to its
    law — mixed effects), or already-translated pairs (index into θ°, index into the model's parameter vector) applied to
    every recording.  theta_o: [len] or [len, P]."""
    se = be.se
    th = se.theta.copy()                      # equalize_law_params!: everything not updated is shared with the accepted law
    theta_o = np.asarray(theta_o, dtype=np.float64)
    # GP.equalize_obs_params! / equalize_law_params! FIRST (src/biblock.jl:362-363): b° := b for every record; if b° had to be
    # changed, its guiding term belongs to other parameters and the update becomes critical
    changed = be.ctx.equalize_laws(3)
    obs_update = None
    if isinstance(pnames, ParamNamesAllObs):
        if critical_change is None:
            critical_change = pnames.is_critical()
        if th.shape[1] != se.chain_hi - se.chain_lo:
            raise ValueError("per-recording parameter names need one parameter set per recording (P == M)")
        for r, m in enumerate(pnames.flat_updates(se.model)[se.chain_lo:se.chain_hi]):
            for j_dst, i_src in m.items():
                th[j_dst, r] = theta_o[i_src]
        ou = pnames.obs_updates()[se.chain_lo:se.chain_hi]
        if any(ou):
            if se.obs_param_hook is None:
                raise NotImplementedError("θ° updates observation parameters: set se.obs_param_hook(updates, theta_o) -> (L, Sigma, v)")
            obs_update = se.obs_param_hook(ou, theta_o)
    else:
        if critical_change is None:
            raise ValueError("critical_change must be given with a bare pair list")
        for i_src, j_dst in pnames:
            th[j_dst, :] = theta_o[i_src]
    critical_change = bool(critical_change) or changed
    se.theta_o = th
    be.ctx.set_params(th, side=_lib.PROPOSAL, stores=3)     # DD.set_parameters!(bb.b°.PP / P_last / P_excl / Pb_excl, θ°, ...)  :364-367
    if obs_update is not None:
        Lm, Sg, vv = obs_update
        be.ctx.set_obs(Lm, Sg, vv, side=_lib.PROPOSAL)
    if critical_change and se.xbar is not None:
        # the linearisation points did not move, only theta did: they are already on the device (uploaded by the constructor)
        be.ctx.set_aux_linearised(None, side=_lib.PROPOSAL, store=_lib.STORE_PP)
        be.ctx.set_aux_linearised(None, side=_lib.PROPOSAL, store=_lib.STORE_PPB)
    be.ctx.set_proposal_law(be.layout, critical_change, skip)


# ---- thinned path saving (docs/src/tutorials/biblock/smoothing.md:55: `paths[i ÷ 400] = deepcopy(bb.b.XX)`) ------------------------
class PathSaver:
    """Keeps the accepted paths of a few recordings every `every` iterations without stalling the sampler: each save is an
    asynchronous device-side gather + device-to-host copy on a second stream into page-locked memory.
        saver = PathSaver(se, chains=[0, 5], every=400);  in the loop: saver(i);  at the end: saver.paths() -> [(i, X[NP, d, n]), ...]"""

    def __init__(self, se, chains, every=1, side=0):
        self.se, self.chains, self.every, self.side = se, np.asarray(chains, dtype=np.int32), int(every), side
        self._saved = []

    def _buffer(self):
        shape = (self.se.ctx.NP, self.se.ctx.d, self.chains.size)
        try:
            import torch
            t = torch.empty(shape, dtype=torch.float64, pin_memory=True)
            return t, t.numpy()
        except Exception:
            a = np.empty(shape)
            return a, a

    def __call__(self, mcmciter):
        if mcmciter % self.every:
            return False
        keep, arr = self._buffer()
        self.se.ctx.snapshot_paths_async(self.chains, arr, self.side)
        self._saved.append((mcmciter, keep, arr))
        return True

    def paths(self):
        self.se.ctx.snapshot_wait()
        return [(i, arr) for i, _, arr in self._saved]


class PathMoments:
    """Posterior summary of the accepted paths of EVERY recording, computed where the paths live: the counterpart of PathSaver for
    the whole ensemble.  Each call at iterations start, start + every, ... adds the current accepted paths to per-recording running
    moments on the device (one kernel launch, no copy).
        pm = PathMoments(se, every=10, start=1000);  in the loop: pm(i);  at the end:
        mean, var = pm.chain_moments()          # [NP, d, M] each: the posterior mean and variance of every recording's path
        mean, var, rhat = pm.pset_moments()     # [NP, d, P]: pooled over the chains of each data set, with Gelman-Rubin R-hat
    Point axis as in get_X (concatenated interval grids).  The summaries cover the chains this process holds."""

    def __init__(self, se, every=1, start=0):
        self.se, self.every, self.start = se, int(every), int(start)

    def __call__(self, mcmciter):
        if mcmciter < self.start or (mcmciter - self.start) % self.every:
            return False
        self.se.ctx.path_moments_add()
        return True

    @property
    def count(self):
        return self.se.ctx.moments_count

    def reset(self):
        self.se.ctx.path_moments_reset()

    def chain_moments(self, chains=None):
        """-> (mean, var) [NP, d, n] of the listed recordings (None: all), var = m2 / count (divisor count)"""
        mean, m2, n = self.se.ctx.get_path_moments(chains)
        return mean, m2 / n

    def pset_moments(self):
        """-> (mean, var, rhat) [NP, d, P]; var is the variance of all pooled draws, rhat is NaN where it is undefined"""
        return self.se.ctx.get_pset_path_moments()


class HistoryStreamer:
    """Streams ll_history / accpt_history of a BlockEnsemble to the host in chunks of `every` iterations while the sampler runs
    (b.ll_history, b°.ll_history src/block.jl:57-58; bb.accpt_history src/biblock.jl:47): call it once per iteration AFTER the
    iteration's save_ll! / accept step; `collect()` waits and returns (ll [n, 2, nb, M], acc [n, nb, M]) of everything streamed."""

    def __init__(self, be, every=64):
        self.be, self.every, self._next, self._chunks = be, int(every), 0, []

    def _buffers(self, n):
        nb, M = self.be.n_blocks, self.be.ctx.M
        try:
            import torch
            a, b = torch.empty((n, 2, nb, M), dtype=torch.float64, pin_memory=True), torch.empty((n, nb, M), dtype=torch.uint8, pin_memory=True)
            return (a, b), a.numpy(), b.numpy()
        except Exception:
            a, b = np.empty((n, 2, nb, M)), np.empty((n, nb, M), dtype=np.uint8)
            return (a, b), a, b

    def __call__(self, mcmciter, flush=False):
        """rows self._next .. mcmciter are final; ship them when a chunk is full (or on flush)"""
        n = mcmciter - self._next + 1
        if n <= 0 or (n < self.every and not flush):
            return False
        keep, ll, acc = self._buffers(n)
        self.be.ctx.histories_async(self.be.layout, self._next, mcmciter, ll, acc)
        self._chunks.append((self._next, keep, ll, acc))
        self._next = mcmciter + 1
        return True

    def collect(self):
        self.be.ctx.snapshot_wait()
        if not self._chunks:
            nb, M = self.be.n_blocks, self.be.ctx.M
            return np.empty((0, 2, nb, M)), np.empty((0, nb, M), dtype=bool)
        return np.concatenate([c[2] for c in self._chunks]), np.concatenate([c[3] for c in self._chunks]).astype(bool)


# ---- checkpoint / resume (not in the reference, which keeps its state in Julia objects; SURVEY §5 / §8f item 3) -------------
_ADAPT_KEYS = ("target", "gamma0", "decay", "window", "rho_min", "rho_max")


def save_state(se, path, layouts=()):
    """Everything needed to continue a run bit-exactly: accepted and proposal X and W (resolved through the parity bits), the
    accepted and proposal parameters θ / θ°, per layout the ll fields, the ll / accept histories, ρ of every (block, recording) and,
    while ρ adapts, the adaptation's settings and state, and the path moments (PathMoments) when any were accumulated.  The
    counter-based generator needs no state beyond (seed, layout, iteration)."""
    ctx = se.ctx
    d = dict(X0=ctx.get_X(0), X1=ctx.get_X(1), W0=ctx.get_W(0), W1=ctx.get_W(1), theta=se.theta, theta_o=se.theta_o,
             n_pts=ctx.n_pts, tt=ctx.tt, chain_lo=se.chain_lo, chain_hi=se.chain_hi)
    for be in layouts:
        d["ll0_%d" % be.layout] = ctx.get_ll(be.layout, 0)
        d["ll1_%d" % be.layout] = ctx.get_ll(be.layout, 1)
        d["rho_%d" % be.layout] = ctx.get_rho_chains(be.layout)
        if be.rho_adaptation is not None:
            a = be.rho_adaptation
            d["rho_adapt_%d" % be.layout] = np.array([a[k] for k in _ADAPT_KEYS], dtype=np.float64)
            d["rho_s_%d" % be.layout], d["rho_nacc_%d" % be.layout], d["rho_calls_%d" % be.layout] = ctx.get_rho_adaptation_state(be.layout)
        if be.ll_hist_len > 0:
            d["acc_hist_%d" % be.layout] = ctx.get_accept_history(be.layout, 0, be.ll_hist_len - 1)
            for s in (0, 1):
                d["ll_hist%d_%d" % (s, be.layout)] = ctx.get_ll_history(be.layout, s, 0, be.ll_hist_len - 1)
    if ctx.moments_count > 0:
        d["moments_mean"], d["moments_m2"], d["moments_count"] = ctx.get_path_moments()
    np.savez_compressed(path, **d)


def load_state(se, path, layouts=()):
    """Restore a state written by save_state into an ensemble built with the same recordings, grids, seed and layouts.
    The laws are restored too: θ / θ° go back to the device (through the law parity, so it does not matter how many
    swap_PP! the saved run had made), the Jacobian-linearised auxiliary laws are re-evaluated at the stored points, and the guiding
    term of every layout in `layouts` is recomputed (in order; layouts sharing the store are recomputed by the sweep loop anyway).
    Path moments are restored when the checkpoint has them and reset when it has none."""
    z = np.load(path)
    ctx = se.ctx
    if not (np.array_equal(z["n_pts"], ctx.n_pts) and np.array_equal(z["tt"], ctx.tt) and int(z["chain_lo"]) == se.chain_lo and int(z["chain_hi"]) == se.chain_hi):
        raise ValueError("checkpoint belongs to a different ensemble (grid or chain slice differ)")
    ctx.set_X(z["X0"], 0); ctx.set_X(z["X1"], 1); ctx.set_W(z["W0"], 0); ctx.set_W(z["W1"], 1)
    if "moments_count" in z:
        ctx.set_path_moments(z["moments_mean"], z["moments_m2"], int(z["moments_count"]))
    else:
        ctx.path_moments_reset()
    se.theta, se.theta_o = z["theta"].copy(), z["theta_o"].copy()
    sides = ((0, se.theta), (1, se.theta_o)) if se.two_sided else ((0, se.theta),)
    for side, th in sides:
        ctx.set_params(th, side=side, stores=3)
        if se.xbar is not None:
            ctx.set_aux_linearised(None, side=side, store=_lib.STORE_PP)
            ctx.set_aux_linearised(None, side=side, store=_lib.STORE_PPB)
    for be in layouts:
        ctx.set_ll(be.layout, z["ll0_%d" % be.layout], 0)
        ctx.set_ll(be.layout, z["ll1_%d" % be.layout], 1)
        if ("rho_%d" % be.layout) in z:
            ctx.set_rho_chains(be.layout, z["rho_%d" % be.layout])
            if ("rho_adapt_%d" % be.layout) in z:
                a = z["rho_adapt_%d" % be.layout]
                enable_rho_adaptation(be, **{k: (int(v) if k == "window" else float(v)) for k, v in zip(_ADAPT_KEYS, a)})
                ctx.set_rho_adaptation_state(be.layout, z["rho_s_%d" % be.layout], z["rho_nacc_%d" % be.layout], int(z["rho_calls_%d" % be.layout]))
            elif be.rho_adaptation is not None:
                disable_rho_adaptation(be)
        if be.ll_hist_len > 0 and ("acc_hist_%d" % be.layout) in z:
            acc = z["acc_hist_%d" % be.layout]
            for i in range(be.ll_hist_len):
                ctx.set_accepted(be.layout, i, acc[i])
                for s in (0, 1):
                    ctx.set_ll_history(be.layout, s, i, z["ll_hist%d_%d" % (s, be.layout)][i])
        ctx.recompute_guiding_term(be.layout, _lib.P_BOTH if se.two_sided else _lib.P_ONLY)
