"""ctypes binding of libdmt.so (include/dmt.h).  Fails loudly: no library or no GPU => exception, never a CPU path.

`Ctx` is a 1:1 numpy-facing wrapper of the C ABI (what the Julia glue in julia/DiffusionMCMCToolsB200.jl does with
ccall); the reference-shaped API (SamplingEnsemble / BlockEnsemble ...) is in host.py.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DMT_LIB") or os.path.join(_HERE, "libdmt.so")  # DMT_LIB: a tuning variant built by build.py --tag

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_bp = C.POINTER(C.c_uint8)
_vp = C.c_void_p

FHN, LV, LORENZ, PROK, JR, OU2 = range(6)
MODEL_NAMES = {FHN: "FitzHughNagumo", LV: "LotkaVolterra", LORENZ: "Lorenz", PROK: "Prokaryote", JR: "JansenRit", OU2: "OU2"}
ACCEPTED, PROPOSAL = 0, 1
STORE_PP, STORE_PPB = 0, 1
P_ONLY, PO_ONLY, P_BOTH = 1, 2, 3
SWAP_XX, SWAP_WW, SWAP_PP, SWAP_LL = 1, 2, 4, 8
K1_RK4, K1_TSIT5 = 0, 1


class DmtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libdmt error %d: %s" % (code, msg))
        self.code = code


class Config(C.Structure):
    _fields_ = [("model", C.c_int32), ("n_chains", C.c_int32), ("n_psets", C.c_int32), ("n_intervals", C.c_int32),
                ("obs_dim", C.c_int32), ("device", C.c_int32), ("two_sided_laws", C.c_int32), ("ll_hist_len", C.c_int32),
                ("n_layouts", C.c_int32), ("chain_offset", C.c_int32), ("seed", C.c_uint64), ("artificial_noise", C.c_double)]


# name -> (restype, argtypes); the list tests/test_abi.py checks against include/dmt.h
SIGNATURES = {
    "dmt_create": (C.c_int32, [C.POINTER(Config), _ip, _dp, _ip, C.POINTER(_vp)]),
    "dmt_destroy": (C.c_int32, [_vp]),
    "dmt_last_error": (C.c_char_p, [_vp]),
    "dmt_sync": (C.c_int32, [_vp]),
    "dmt_get_stream": (C.c_int32, [_vp, C.POINTER(_vp)]),
    "dmt_model_dims": (C.c_int32, [C.c_int32, _ip, _ip, _ip, _ip]),
    "dmt_version": (C.c_int32, []),
    "dmt_launch_count": (C.c_int32, [C.POINTER(C.c_uint64)]),
    "dmt_set_params": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _dp]),
    "dmt_set_aux": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _dp, _dp, _dp]),
    "dmt_set_aux_linearised": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _dp]),
    "dmt_set_obs": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, _dp, _dp, _dp]),
    "dmt_equalize_laws": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, _ip]),
    "dmt_set_blocks": (C.c_int32, [_vp, C.c_int32, C.c_int32, _ip, _ip, _dp, _bp, C.c_int32]),
    "dmt_set_rho": (C.c_int32, [_vp, C.c_int32, _dp]),
    "dmt_set_rho_chains": (C.c_int32, [_vp, C.c_int32, _dp]),
    "dmt_get_rho_chains": (C.c_int32, [_vp, C.c_int32, _dp]),
    "dmt_set_rho_adaptation": (C.c_int32, [_vp, C.c_int32, C.c_double, C.c_double, C.c_double, C.c_int32, C.c_double, C.c_double]),
    "dmt_adapt_rho": (C.c_int32, [_vp, C.c_int32]),
    "dmt_get_rho_adaptation_state": (C.c_int32, [_vp, C.c_int32, _dp, _ip, C.POINTER(C.c_uint64)]),
    "dmt_set_rho_adaptation_state": (C.c_int32, [_vp, C.c_int32, _dp, _ip, C.c_uint64]),
    "dmt_set_start": (C.c_int32, [_vp, _dp]),
    "dmt_init_paths": (C.c_int32, [_vp, C.c_int32, C.c_uint32, C.c_int32, _ip]),
    "dmt_set_X": (C.c_int32, [_vp, C.c_int32, _dp]),
    "dmt_get_X": (C.c_int32, [_vp, C.c_int32, _dp]),
    "dmt_set_W": (C.c_int32, [_vp, C.c_int32, _dp]),
    "dmt_get_W": (C.c_int32, [_vp, C.c_int32, _dp]),
    "dmt_set_artificial_obs": (C.c_int32, [_vp, C.c_int32]),
    "dmt_recompute_guiding_term": (C.c_int32, [_vp, C.c_int32, C.c_int32]),
    "dmt_find_W_for_X": (C.c_int32, [_vp, C.c_int32]),
    "dmt_loglikhd": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32]),
    "dmt_find_W_and_loglikhd": (C.c_int32, [_vp, C.c_int32]),
    "dmt_draw_proposal_path": (C.c_int32, [_vp, C.c_int32, C.c_uint32, _dp]),
    "dmt_find_W_loglikhd_draw": (C.c_int32, [_vp, C.c_int32, C.c_uint32, _dp]),
    "dmt_blocking_sweep": (C.c_int32, [_vp, C.c_int32, C.c_uint32]),
    "dmt_recompute_path": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "dmt_set_proposal_law": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32]),
    "dmt_accept_reject_path": (C.c_int32, [_vp, C.c_int32, C.c_uint32, _dp]),
    "dmt_swap": (C.c_int32, [_vp, C.c_int32, C.c_int32, _bp]),
    "dmt_swap_blocks": (C.c_int32, [_vp, C.c_int32, C.c_int32, _bp]),
    "dmt_save_ll": (C.c_int32, [_vp, C.c_int32, C.c_uint32]),
    "dmt_fetch_ll": (C.c_int32, [_vp, C.c_int32, C.c_int32, _dp, _dp]),
    "dmt_get_ll": (C.c_int32, [_vp, C.c_int32, C.c_int32, _dp]),
    "dmt_set_ll": (C.c_int32, [_vp, C.c_int32, C.c_int32, _dp]),
    "dmt_get_success": (C.c_int32, [_vp, C.c_int32, _bp]),
    "dmt_get_accept_history": (C.c_int32, [_vp, C.c_int32, C.c_uint32, C.c_uint32, _bp]),
    "dmt_get_ll_history": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_uint32, C.c_uint32, _dp]),
    "dmt_accept_counts": (C.c_int32, [_vp, C.c_int32, C.c_uint32, C.c_uint32, C.POINTER(C.c_int64)]),
    "dmt_get_last_accept": (C.c_int32, [_vp, C.c_int32, _bp]),
    "dmt_get_guiding_term": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, _dp, _dp, _dp]),
    "dmt_upload_guiding_term": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, _dp, _dp, _dp]),
    "dmt_enable_guiding_cache": (C.c_int32, [_vp, C.c_int32, C.c_int32]),
    "dmt_set_fwd_lanes": (C.c_int32, [_vp, C.c_int32]),
    "dmt_set_bwd_mode": (C.c_int32, [_vp, C.c_int32]),
    "dmt_set_bwd_solver": (C.c_int32, [_vp, C.c_int32, C.c_double, C.c_double]),
    "dmt_get_bwd_steps": (C.c_int32, [_vp, _ip, _ip]),
    "dmt_set_sweep_mode": (C.c_int32, [_vp, C.c_int32]),
    "dmt_set_lazy_noise": (C.c_int32, [_vp, C.c_int32]),
    "dmt_get_last_forward_kernel": (C.c_int32, [_vp, C.c_char_p, C.c_int32]),
    "dmt_get_X_chains": (C.c_int32, [_vp, C.c_int32, C.c_int32, _ip, _dp]),
    "dmt_get_W_chains": (C.c_int32, [_vp, C.c_int32, C.c_int32, _ip, _dp]),
    "dmt_path_moments_add": (C.c_int32, [_vp]),
    "dmt_path_moments_reset": (C.c_int32, [_vp]),
    "dmt_get_path_moments": (C.c_int32, [_vp, C.c_int32, _ip, _dp, _dp, C.POINTER(C.c_uint64)]),
    "dmt_set_path_moments": (C.c_int32, [_vp, _dp, _dp, C.c_uint64]),
    "dmt_get_pset_path_moments": (C.c_int32, [_vp, _dp, _dp, _dp]),
    "dmt_get_layout_guiding_term": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_int32, _dp, _dp, _dp]),
    "dmt_debug_normals": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, _dp]),
    "dmt_debug_exponentials": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, _dp]),
    "dmt_nccl_unique_id": (C.c_int32, [_bp]),
    "dmt_comm_init": (C.c_int32, [_vp, C.c_int32, C.c_int32, _bp]),
    "dmt_allreduce_stats": (C.c_int32, [_vp, C.c_int32, _dp]),
    "dmt_snapshot_paths_async": (C.c_int32, [_vp, C.c_int32, C.c_int32, _ip, _dp]),
    "dmt_snapshot_wait": (C.c_int32, [_vp]),
    "dmt_histories_async": (C.c_int32, [_vp, C.c_int32, C.c_uint32, C.c_uint32, _dp, _bp]),
    "dmt_set_accepted": (C.c_int32, [_vp, C.c_int32, C.c_uint32, _bp]),
    "dmt_set_ll_history": (C.c_int32, [_vp, C.c_int32, C.c_int32, C.c_uint32, _dp]),
    "dmt_p2p_export": (C.c_int32, [_vp, _bp]),
    "dmt_p2p_init": (C.c_int32, [_vp, C.c_int32, C.c_int32, _bp]),
    "dmt_p2p_disable": (C.c_int32, [_vp]),
}

_lib = None


def load():
    """dlopen libdmt.so; raises if the CUDA extension was not built (there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libdmt.so is missing: run `python diffusionmcmctools.jl_b200/build.py` "
                               "(the product has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(lib, name)
            f.restype = res
            f.argtypes = args
        _lib = lib
    return _lib


def launch_count():
    """kernels launched by libdmt in this process so far"""
    n = C.c_uint64(0)
    load().dmt_launch_count(C.byref(n))
    return int(n.value)


def model_dims(model):
    lib = load()
    d, dw, npar, cd = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
    if lib.dmt_model_dims(model, C.byref(d), C.byref(dw), C.byref(npar), C.byref(cd)):
        raise ValueError("unknown model id %r" % (model,))
    return d.value, dw.value, npar.value, bool(cd.value)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError("expected array of shape %s, got %s" % (tuple(shape), tuple(a.shape)))
    return a


def _p(a):
    return a.ctypes.data_as(_dp)


DEFAULT_FWD_LANES = 0  # applied to every new Ctx (the test-suite runs the GPU tests once per setting)


class Ctx:
    """One device-resident SamplingEnsemble (M chains on one GPU).  Thin wrapper of the C ABI; arrays are numpy, with
    the chain / pset index LAST (fastest), as include/dmt.h documents."""

    def __init__(self, model, n_pts, tt, n_chains, n_psets=None, obs_dim=1, device=0, two_sided_laws=False, ll_hist_len=0,
                 n_layouts=4, chain_offset=0, seed=0, artificial_noise=1e-11, pset_of_chain=None):
        self.lib = load()
        self.h = _vp()
        self.model = model
        self.d, self.dw, self.npar, self.constdiff = model_dims(model)
        self.n_pts = np.ascontiguousarray(n_pts, dtype=np.int32)
        self.K = int(self.n_pts.size)
        self.M = int(n_chains)
        self.P = int(n_psets if n_psets is not None else n_chains)
        self.m = int(obs_dim)
        self.NP = int(self.n_pts.sum())
        self.S = self.NP - self.K
        self.tt = _f64(tt, (self.NP,))
        self.pt0 = np.concatenate([[0], np.cumsum(self.n_pts)]).astype(np.int64)
        self.step0 = np.concatenate([[0], np.cumsum(self.n_pts - 1)]).astype(np.int64)
        self.n_layouts = n_layouts
        self.layout_nb = {}
        cfg = Config(model, self.M, self.P, self.K, self.m, device, int(two_sided_laws), ll_hist_len, n_layouts,
                     chain_offset, seed, artificial_noise)
        pp = None
        if pset_of_chain is not None:
            self._pset = np.ascontiguousarray(pset_of_chain, dtype=np.int32)
            pp = self._pset.ctypes.data_as(_ip)
        rc = self.lib.dmt_create(C.byref(cfg), self.n_pts.ctypes.data_as(_ip), _p(self.tt), pp, C.byref(self.h))
        if rc:
            raise DmtError(rc, (self.lib.dmt_last_error(None) or b"").decode())
        self.moments_count = 0  # updates in the path-moment accumulators (mirrors the library's count)
        if DEFAULT_FWD_LANES:
            self.set_fwd_lanes(DEFAULT_FWD_LANES)

    # -- plumbing
    def _ck(self, rc):
        if rc:
            raise DmtError(rc, (self.lib.dmt_last_error(self.h) or b"").decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.dmt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        self._ck(self.lib.dmt_sync(self.h))

    def stream(self):
        s = _vp()
        self._ck(self.lib.dmt_get_stream(self.h, C.byref(s)))
        return s.value or 0

    def _krange(self, k0, k1):
        k0 = 0 if k0 is None else k0
        k1 = self.K - 1 if k1 is None else k1
        return k0, k1

    # -- laws
    def set_params(self, theta, side=ACCEPTED, stores=3, k0=None, k1=None):
        k0, k1 = self._krange(k0, k1)
        th = _f64(theta)
        if th.ndim == 1:
            th = np.repeat(th[:, None], self.P, axis=1)
        th = _f64(th, (self.npar, self.P))
        self._ck(self.lib.dmt_set_params(self.h, side, stores, k0, k1, _p(th)))

    def _bc(self, a, shape_k, nk):
        """broadcast a per-interval array lacking the pset axis and/or the interval axis to [nk, ..., P]"""
        a = np.asarray(a, dtype=np.float64)
        if a.shape == tuple(shape_k):
            a = np.broadcast_to(a[None, ..., None], (nk,) + tuple(shape_k) + (self.P,))
        elif a.shape == (nk,) + tuple(shape_k):
            a = np.broadcast_to(a[..., None], (nk,) + tuple(shape_k) + (self.P,))
        return _f64(a, (nk,) + tuple(shape_k) + (self.P,))

    def set_aux(self, B, beta, atil, side=ACCEPTED, store=STORE_PP, k0=None, k1=None):
        k0, k1 = self._krange(k0, k1)
        nk, d = k1 - k0 + 1, self.d
        B = self._bc(B, (d, d), nk); beta = self._bc(beta, (d,), nk); atil = self._bc(atil, (d, d), nk)
        self._ck(self.lib.dmt_set_aux(self.h, side, store, k0, k1, _p(B), _p(beta), _p(atil)))

    def set_aux_linearised(self, xbar, side=ACCEPTED, store=STORE_PP, k0=None, k1=None):
        """xbar = None: re-linearise at the points uploaded last for this store (only theta changed)"""
        k0, k1 = self._krange(k0, k1)
        if xbar is None:
            self._ck(self.lib.dmt_set_aux_linearised(self.h, side, store, k0, k1, None))
            return
        xb = self._bc(xbar, (self.d,), k1 - k0 + 1)
        self._ck(self.lib.dmt_set_aux_linearised(self.h, side, store, k0, k1, _p(xb)))

    def set_obs(self, L, Sigma, v, side=ACCEPTED, k0=None, k1=None):
        k0, k1 = self._krange(k0, k1)
        nk, m, d = k1 - k0 + 1, self.m, self.d
        L = self._bc(L, (m, d), nk); Sigma = self._bc(Sigma, (m, m), nk); v = self._bc(v, (m,), nk)
        self._ck(self.lib.dmt_set_obs(self.h, side, k0, k1, _p(L), _p(Sigma), _p(v)))

    def equalize_laws(self, stores=3, k0=None, k1=None):
        """-> True when a proposal record differed from the accepted one (GP.equalize_*'s return value, src/biblock.jl:362-363)"""
        k0, k1 = self._krange(k0, k1)
        ch = C.c_int32(0)
        self._ck(self.lib.dmt_equalize_laws(self.h, stores, k0, k1, C.byref(ch)))
        return bool(ch.value)

    # -- layouts
    def set_blocks(self, layout, ranges, rho=0.0, last=None, ll_hist_len=-1):
        nb = len(ranges)
        i0 = np.ascontiguousarray([r[0] for r in ranges], dtype=np.int32)
        i1 = np.ascontiguousarray([r[1] for r in ranges], dtype=np.int32)
        rho = _f64(np.broadcast_to(np.asarray(rho, dtype=np.float64), (nb,)))
        lp = None
        if last is not None:
            last = np.ascontiguousarray(last, dtype=np.uint8)
            lp = last.ctypes.data_as(_bp)
        self._ck(self.lib.dmt_set_blocks(self.h, layout, nb, i0.ctypes.data_as(_ip), i1.ctypes.data_as(_ip), _p(rho), lp, ll_hist_len))
        self.layout_nb[layout] = nb

    def set_rho(self, layout, rho):
        rho = _f64(np.broadcast_to(np.asarray(rho, dtype=np.float64), (self.layout_nb[layout],)))
        self._ck(self.lib.dmt_set_rho(self.h, layout, _p(rho)))

    def set_rho_chains(self, layout, rho):
        """ρ of every (block, chain): anything that broadcasts to [n_blocks, M]"""
        shape = (self.layout_nb[layout], self.M)
        rho = _f64(np.broadcast_to(np.asarray(rho, dtype=np.float64), shape), shape)
        self._ck(self.lib.dmt_set_rho_chains(self.h, layout, _p(rho)))

    def get_rho_chains(self, layout):
        rho = np.empty((self.layout_nb[layout], self.M))
        self._ck(self.lib.dmt_get_rho_chains(self.h, layout, _p(rho)))
        return rho

    def set_rho_adaptation(self, layout, target, gamma0=1.0, decay=0.66, window=10, rho_min=0.0, rho_max=0.999):
        """target <= 0: freeze ρ (adaptation off); see include/dmt.h for the rule"""
        self._ck(self.lib.dmt_set_rho_adaptation(self.h, layout, float(target), float(gamma0), float(decay), int(window),
                                                 float(rho_min), float(rho_max)))

    def adapt_rho(self, layout):
        self._ck(self.lib.dmt_adapt_rho(self.h, layout))

    def get_rho_adaptation_state(self, layout):
        """-> (s [n_blocks, M], nacc [n_blocks, M] int32, calls)"""
        shape = (self.layout_nb[layout], self.M)
        s, nacc, calls = np.empty(shape), np.empty(shape, dtype=np.int32), C.c_uint64(0)
        self._ck(self.lib.dmt_get_rho_adaptation_state(self.h, layout, _p(s), nacc.ctypes.data_as(_ip), C.byref(calls)))
        return s, nacc, int(calls.value)

    def set_rho_adaptation_state(self, layout, s, nacc, calls):
        shape = (self.layout_nb[layout], self.M)
        s = _f64(s, shape)
        nacc = np.ascontiguousarray(nacc, dtype=np.int32)
        assert nacc.shape == shape
        self._ck(self.lib.dmt_set_rho_adaptation_state(self.h, layout, _p(s), nacc.ctypes.data_as(_ip), int(calls)))

    # -- paths
    def set_start(self, x0):
        x0 = np.asarray(x0, dtype=np.float64)
        if x0.ndim == 1:
            x0 = np.repeat(x0[:, None], self.M, axis=1)
        self._ck(self.lib.dmt_set_start(self.h, _p(_f64(x0, (self.d, self.M)))))

    def init_paths(self, layout=0, iter0=0, max_tries=100):
        nf = C.c_int32()
        self._ck(self.lib.dmt_init_paths(self.h, layout, iter0, max_tries, C.byref(nf)))
        return nf.value

    def set_X(self, X, side=ACCEPTED):
        self._ck(self.lib.dmt_set_X(self.h, side, _p(_f64(X, (self.NP, self.d, self.M)))))

    def get_X(self, side=ACCEPTED):
        X = np.empty((self.NP, self.d, self.M))
        self._ck(self.lib.dmt_get_X(self.h, side, _p(X)))
        return X

    def snapshot_paths_async(self, chains, out, side=ACCEPTED):
        """queue a copy of the paths of `chains` into out [NP, d, len(chains)] (float64, C-contiguous, ideally page-locked);
        read `out` after snapshot_wait()"""
        sel = np.ascontiguousarray(chains, dtype=np.int32)
        assert out.dtype == np.float64 and out.flags.c_contiguous and out.shape == (self.NP, self.d, sel.size)
        self._ck(self.lib.dmt_snapshot_paths_async(self.h, side, int(sel.size), sel.ctypes.data_as(_ip), _p(out)))

    def histories_async(self, layout, it0, it1, out_ll=None, out_acc=None):
        """queue a copy of ll_history rows it0..it1 into out_ll [n, 2, nb, M] (float64) and / or accpt_history into out_acc [n, nb, M]
        (uint8); C-contiguous, ideally page-locked; read after snapshot_wait()"""
        n, nb = it1 - it0 + 1, self.layout_nb[layout]
        if out_ll is not None:
            assert out_ll.dtype == np.float64 and out_ll.flags.c_contiguous and out_ll.shape == (n, 2, nb, self.M)
        if out_acc is not None:
            assert out_acc.dtype == np.uint8 and out_acc.flags.c_contiguous and out_acc.shape == (n, nb, self.M)
        self._ck(self.lib.dmt_histories_async(self.h, layout, it0, it1, _p(out_ll) if out_ll is not None else None,
                                              out_acc.ctypes.data_as(_bp) if out_acc is not None else None))

    def snapshot_wait(self):
        self._ck(self.lib.dmt_snapshot_wait(self.h))

    def get_X_chains(self, chains, side=ACCEPTED):
        """X [NP, d, len(chains)] of the listed recordings (bb.b.XX of a few recordings)"""
        sel = np.ascontiguousarray(chains, dtype=np.int32)
        X = np.empty((self.NP, self.d, sel.size))
        self._ck(self.lib.dmt_get_X_chains(self.h, side, int(sel.size), sel.ctypes.data_as(_ip), _p(X)))
        return X

    def get_W_chains(self, chains, side=ACCEPTED):
        sel = np.ascontiguousarray(chains, dtype=np.int32)
        W = np.empty((self.S, self.dw, sel.size))
        self._ck(self.lib.dmt_get_W_chains(self.h, side, int(sel.size), sel.ctypes.data_as(_ip), _p(W)))
        return W

    def set_W(self, W, side=ACCEPTED):
        self._ck(self.lib.dmt_set_W(self.h, side, _p(_f64(W, (self.S, self.dw, self.M)))))

    def get_W(self, side=ACCEPTED):
        W = np.empty((self.S, self.dw, self.M))
        self._ck(self.lib.dmt_get_W(self.h, side, _p(W)))
        return W

    # -- posterior path moments (per-chain Welford moments of the accepted paths, kept on the device)
    def path_moments_add(self):
        """accumulate the current accepted paths of all chains (one kernel launch)"""
        self._ck(self.lib.dmt_path_moments_add(self.h))
        self.moments_count += 1

    def path_moments_reset(self):
        self._ck(self.lib.dmt_path_moments_reset(self.h))
        self.moments_count = 0

    def get_path_moments(self, chains=None):
        """-> (mean [NP, d, n], m2 [NP, d, n], count) of the listed chains (None: all M); var = m2 / count"""
        sel = None if chains is None else np.ascontiguousarray(chains, dtype=np.int32)
        n = self.M if sel is None else int(sel.size)
        mean, m2, cnt = np.empty((self.NP, self.d, n)), np.empty((self.NP, self.d, n)), C.c_uint64(0)
        self._ck(self.lib.dmt_get_path_moments(self.h, n, None if sel is None else sel.ctypes.data_as(_ip), _p(mean), _p(m2), C.byref(cnt)))
        return mean, m2, int(cnt.value)

    def set_path_moments(self, mean, m2, count):
        """restore all M chains' moments (as get_path_moments() returned them)"""
        shape = (self.NP, self.d, self.M)
        self._ck(self.lib.dmt_set_path_moments(self.h, _p(_f64(mean, shape)), _p(_f64(m2, shape)), int(count)))
        self.moments_count = int(count)

    def get_pset_path_moments(self):
        """-> (mean, var, rhat), each [NP, d, P]: pooled over the chains of each parameter / data set (see include/dmt.h)"""
        out = [np.empty((self.NP, self.d, self.P)) for _ in range(3)]
        self._ck(self.lib.dmt_get_pset_path_moments(self.h, *(_p(a) for a in out)))
        return tuple(out)

    # -- hot path
    def set_artificial_obs(self, layout):
        self._ck(self.lib.dmt_set_artificial_obs(self.h, layout))

    def recompute_guiding_term(self, layout, which=P_BOTH):
        self._ck(self.lib.dmt_recompute_guiding_term(self.h, layout, which))

    def find_W_for_X(self, layout):
        self._ck(self.lib.dmt_find_W_for_X(self.h, layout))

    def loglikhd(self, layout, side=ACCEPTED, skip=0):
        self._ck(self.lib.dmt_loglikhd(self.h, layout, side, skip))

    def find_W_and_loglikhd(self, layout):
        self._ck(self.lib.dmt_find_W_and_loglikhd(self.h, layout))

    def draw_proposal_path(self, layout, it, Z=None):
        zp = None
        if Z is not None:
            Z = _f64(Z, (self.S, self.dw, self.M))
            zp = _p(Z)
        self._ck(self.lib.dmt_draw_proposal_path(self.h, layout, it, zp))

    def find_W_loglikhd_draw(self, layout, it, Z=None):
        zp = None
        if Z is not None:
            Z = _f64(Z, (self.S, self.dw, self.M))
            zp = _p(Z)
        self._ck(self.lib.dmt_find_W_loglikhd_draw(self.h, layout, it, zp))

    def blocking_sweep(self, layout, it):
        self._ck(self.lib.dmt_blocking_sweep(self.h, layout, it))

    def recompute_path(self, layout, law_side=PROPOSAL, noise_side=ACCEPTED, skip=0):
        self._ck(self.lib.dmt_recompute_path(self.h, layout, law_side, noise_side, skip))

    def set_proposal_law(self, layout, critical_change, skip=0):
        self._ck(self.lib.dmt_set_proposal_law(self.h, layout, int(bool(critical_change)), skip))

    def accept_reject_path(self, layout, it, E=None):
        ep = None
        if E is not None:
            E = _f64(E, (self.layout_nb[layout], self.M))
            ep = _p(E)
        self._ck(self.lib.dmt_accept_reject_path(self.h, layout, it, ep))

    def swap(self, layout, what, chain_mask=None):
        mp = None
        if chain_mask is not None:
            chain_mask = np.ascontiguousarray(chain_mask, dtype=np.uint8)
            assert chain_mask.shape == (self.M,)
            mp = chain_mask.ctypes.data_as(_bp)
        self._ck(self.lib.dmt_swap(self.h, layout, what, mp))

    def swap_blocks(self, layout, what, mask):
        """the swaps of dmt_swap for the (block, recording) pairs flagged in mask [n_blocks, M]"""
        mask = np.ascontiguousarray(mask, dtype=np.uint8)
        assert mask.shape == (self.layout_nb[layout], self.M)
        self._ck(self.lib.dmt_swap_blocks(self.h, layout, what, mask.ctypes.data_as(_bp)))

    def save_ll(self, layout, it):
        self._ck(self.lib.dmt_save_ll(self.h, layout, it))

    # -- read-back
    def fetch_ll(self, layout, side=ACCEPTED):
        tot = C.c_double()
        pb = np.empty(self.layout_nb[layout])
        self._ck(self.lib.dmt_fetch_ll(self.h, layout, side, C.byref(tot), _p(pb)))
        return tot.value, pb

    def get_ll(self, layout, side=ACCEPTED):
        ll = np.empty((self.layout_nb[layout], self.M))
        self._ck(self.lib.dmt_get_ll(self.h, layout, side, _p(ll)))
        return ll

    def set_ll(self, layout, ll, side=ACCEPTED):
        self._ck(self.lib.dmt_set_ll(self.h, layout, side, _p(_f64(ll, (self.layout_nb[layout], self.M)))))

    def get_success(self, layout):
        ok = np.empty((self.layout_nb[layout], self.M), dtype=np.uint8)
        self._ck(self.lib.dmt_get_success(self.h, layout, ok.ctypes.data_as(_bp)))
        return ok.astype(bool)

    def get_last_accept(self, layout):
        a = np.empty((self.layout_nb[layout], self.M), dtype=np.uint8)
        self._ck(self.lib.dmt_get_last_accept(self.h, layout, a.ctypes.data_as(_bp)))
        return a.astype(bool)

    def get_accept_history(self, layout, it0, it1):
        a = np.empty((it1 - it0 + 1, self.layout_nb[layout], self.M), dtype=np.uint8)
        self._ck(self.lib.dmt_get_accept_history(self.h, layout, it0, it1, a.ctypes.data_as(_bp)))
        return a.astype(bool)

    def set_accepted(self, layout, it, acc):
        a = np.ascontiguousarray(np.broadcast_to(np.asarray(acc), (self.layout_nb[layout], self.M)), dtype=np.uint8)
        self._ck(self.lib.dmt_set_accepted(self.h, layout, it, a.ctypes.data_as(_bp)))

    def set_ll_history(self, layout, side, it, ll):
        a = _f64(np.broadcast_to(np.asarray(ll, dtype=np.float64), (self.layout_nb[layout], self.M)), (self.layout_nb[layout], self.M))
        self._ck(self.lib.dmt_set_ll_history(self.h, layout, side, it, _p(a)))

    def get_ll_history(self, layout, side, it0, it1):
        a = np.empty((it1 - it0 + 1, self.layout_nb[layout], self.M))
        self._ck(self.lib.dmt_get_ll_history(self.h, layout, side, it0, it1, _p(a)))
        return a

    def accept_counts(self, layout, it0, it1):
        a = np.zeros(self.layout_nb[layout], dtype=np.int64)
        self._ck(self.lib.dmt_accept_counts(self.h, layout, it0, it1, a.ctypes.data_as(C.POINTER(C.c_int64))))
        return a

    def get_guiding_term(self, k, side=ACCEPTED, store=STORE_PP):
        n, d = int(self.n_pts[k]), self.d
        H = np.empty((n, d, d, self.P)); F = np.empty((n, d, self.P)); c = np.empty((n, self.P))
        self._ck(self.lib.dmt_get_guiding_term(self.h, side, store, k, _p(H), _p(F), _p(c)))
        return H, F, c

    def upload_guiding_term(self, k, H, F, c, side=ACCEPTED, store=STORE_PP):
        n, d = int(self.n_pts[k]), self.d
        H = _f64(H, (n, d, d, self.P)); F = _f64(F, (n, d, self.P)); c = _f64(c, (n, self.P))
        self._ck(self.lib.dmt_upload_guiding_term(self.h, side, store, k, _p(H), _p(F), _p(c)))

    def set_fwd_lanes(self, lanes):
        """lanes per (chain, block) in the forward kernel: 0 = automatic, or 1 / 2 / 4 / 8 (results are identical)"""
        self._ck(self.lib.dmt_set_fwd_lanes(self.h, int(lanes)))

    def set_sweep_mode(self, mode):
        """fused blocking-sweep pass: 0 = automatic, 1 = register-tile kernel, 2 = software-pipelined kernel, 3 = warp-specialised kernel, 5 = step-parallel kernel (or error)"""
        self._ck(self.lib.dmt_set_sweep_mode(self.h, int(mode)))

    def last_forward_kernel(self):
        """name / mapping of the forward kernel launched last (diagnostics)"""
        buf = C.create_string_buffer(96)
        self._ck(self.lib.dmt_get_last_forward_kernel(self.h, buf, 96))
        return buf.value.decode()

    def set_lazy_noise(self, enable=True):
        """blocking sweeps stop materialising W / W° (rebuilt from X on demand); see include/dmt.h"""
        self._ck(self.lib.dmt_set_lazy_noise(self.h, int(bool(enable))))

    def set_bwd_solver(self, solver, reltol=1e-3, abstol=1e-6):
        """K1_RK4 (default) or K1_TSIT5 (upstream's adaptive solver at OrdinaryDiffEq's default tolerances)"""
        self._ck(self.lib.dmt_set_bwd_solver(self.h, int(solver), float(reltol), float(abstol)))

    def get_bwd_steps(self):
        a, r = C.c_int32(0), C.c_int32(0)
        self._ck(self.lib.dmt_get_bwd_steps(self.h, C.byref(a), C.byref(r)))
        return a.value, r.value

    def set_bwd_mode(self, mode):
        """thread mapping of the backward filter: 0 = automatic, 1 = thread per parameter set, 2 = cooperative lanes"""
        self._ck(self.lib.dmt_set_bwd_mode(self.h, int(mode)))

    # -- guiding cache
    def enable_guiding_cache(self, layout, enable=True):
        self._ck(self.lib.dmt_enable_guiding_cache(self.h, layout, int(bool(enable))))

    def get_layout_guiding_term(self, layout, k, store=STORE_PP):
        n, d = int(self.n_pts[k]), self.d
        H = np.empty((n, d, d, self.P)); F = np.empty((n, d, self.P)); c = np.empty((n, self.P))
        self._ck(self.lib.dmt_get_layout_guiding_term(self.h, layout, store, k, _p(H), _p(F), _p(c)))
        return H, F, c

    # -- test hooks
    def debug_normals(self, chain0, tile0, it, n_chains, n_tiles, layout=0):
        out = np.empty((n_chains, n_tiles, 4 * self.dw))
        self._ck(self.lib.dmt_debug_normals(self.h, chain0, tile0, it, layout, n_chains, n_tiles, _p(out)))
        return out

    def debug_exponentials(self, chain0, it, layout, n_chains, n_blocks):
        out = np.empty((n_chains, n_blocks))
        self._ck(self.lib.dmt_debug_exponentials(self.h, chain0, it, layout, n_chains, n_blocks, _p(out)))
        return out

    # -- multi-GPU
    @staticmethod
    def nccl_unique_id():
        lib = load()
        buf = np.zeros(128, dtype=np.uint8)
        rc = lib.dmt_nccl_unique_id(buf.ctypes.data_as(_bp))
        if rc:
            raise DmtError(rc, (lib.dmt_last_error(None) or b"").decode())
        return buf

    def comm_init(self, n_ranks, rank, uid):
        uid = np.ascontiguousarray(uid, dtype=np.uint8)
        assert uid.size == 128
        self._ck(self.lib.dmt_comm_init(self.h, n_ranks, rank, uid.ctypes.data_as(_bp)))

    def p2p_export(self):
        h = np.zeros(64, dtype=np.uint8)
        self._ck(self.lib.dmt_p2p_export(self.h, h.ctypes.data_as(_bp)))
        return h

    def p2p_init(self, n_ranks, rank, handles):
        handles = np.ascontiguousarray(handles, dtype=np.uint8)
        assert handles.shape == (n_ranks, 64)
        self._ck(self.lib.dmt_p2p_init(self.h, n_ranks, rank, handles.ctypes.data_as(_bp)))

    def p2p_disable(self):
        self._ck(self.lib.dmt_p2p_disable(self.h))

    def allreduce_stats(self, layout):
        out = np.empty(2 + self.layout_nb[layout])
        self._ck(self.lib.dmt_allreduce_stats(self.h, layout, _p(out)))
        return out
