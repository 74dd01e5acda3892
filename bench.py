#!/usr/bin/env python
"""bench.py — guided path updates/s (chains x EM steps / s, FP64) of the blocking path update, BASELINE.json config C3:
Lorenz 3-D, the 4096-chain ensemble, 200 observation intervals x 100 EM steps, two staggered block layouts (10 / 11 blocks)
alternated, pCN rho = 0.9, every chain with its own data and guiding term (P = M).

With N GPUs the ensemble is SPLIT: one contiguous slice of 4096 / N chains per GPU (strong scaling, BASELINE.json north_star); the
weak-scaling rate (4096 chains on every GPU) is measured afterwards and reported as an extra key.

One sweep = exactly the tutorial loop body (/root/reference/docs/src/tutorials/block_collection/inference_with_blocking.md:52-58):
    set_obs! -> recompute_guiding_term!(P only) -> find_W_for_X! + loglikhd! + draw_proposal_path! -> accept_reject_proposal_path!
    -> (N > 1: all-reduce of ll sums / accept counts)
and advances every chain by S = 20,000 guided Euler-Maruyama steps.  One timed "step" = R consecutive sweeps (R stated in `config`,
chosen after the warm-up so that the K timed steps last >= 2.5 s: long enough for the clock sampler; with --dump-outputs, a fixed number
of sweeps per config instead, so that the dumped state does not depend on a measured time); units per step = R x M x S.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c3|c2|c4|c5] [--chains M_per_gpu] [--impl reference]
                    [--dump-outputs DIR]

After build(), bench.py writes nothing into the tree it runs from (which may be read-only): what it compiles goes to a temporary
directory.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # no __pycache__ in the tree for the modules only the benchmark imports

METRIC = "guided path updates/sec (chains x EM steps/s, FP64)"
UNIT = "guided EM steps/s"
TOTAL_CHAINS = {"c1": 1, "c2": 1024, "c3": 4096, "c4": 16384, "c5": 8192}
ALGO_BYTES = {  # SURVEY.md §8(d): per chain per EM step of draw_proposal_path! = 8(2 dw + d) [+ 8(d(d+1)/2 + d) when P = M]
    "c2": (48, 88), "c3": (72, 144), "c4": (96, 208), "c5": (64, 280), "c1": (32, 72),
}
MIN_TIMED_S = 2.5
# --dump-outputs: the dumped state depends on how many sweeps ran, so the timed region holds a fixed number of sweeps per config (the same
# on every rank) instead of one sized from a measured time: about MIN_TIMED_S of sweeps of the config's ensemble on one B200 at the
# sweep times measured in profiles/r02v_bench_c1.json, r02v_bench_c2.json, r02aw_bench_default.json, r02x_bench_c4.json and
# r02ae_bench_c5.json (0.31 / 1.54 / 3.44 / 16.3 / 225 ms; SM clock 1965 MHz, power limit not recorded)
DUMP_TIMED_SWEEPS = {"c1": 8000, "c2": 1600, "c3": 720, "c4": 150, "c5": 11}
DUMP_MAX_BYTES = 64 << 20
DUMP_SAMPLE_CHAINS = 32


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default="c3")
    ap.add_argument("--chains", type=int, default=None, help="chains PER GPU (default: the config's ensemble split over the GPUs)")
    ap.add_argument("--psets", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-chains", type=int, default=None, help="chains in the bounded CPU sample")
    ap.add_argument("--sweeps-per-step", type=int, default=0, help="R (0: chosen so that the timed region lasts >= %.1f s)" % MIN_TIMED_S)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the extra weak-scaling measurement")
    ap.add_argument("--no-uncached", action="store_true", help="skip the extra measurement with the full backward filter every sweep")
    ap.add_argument("--no-self-check", action="store_true")
    ap.add_argument("--one-call", action="store_true", help="blocking sweep through dmt_blocking_sweep (same launches; per-kernel timing is then not available)")
    ap.add_argument("--no-cache", action="store_true", help="blocking sweep with the full backward filter every sweep (no guiding cache)")
    ap.add_argument("--separate", action="store_true", help="blocking sweep with the three separate passes instead of the fused one")
    ap.add_argument("--sweep-mode", type=int, default=0, help="fused pass: 0 auto, 1 register-tile kernel, 2 software-pipelined, 3 / 4 warp-specialised (wide / compact), 5 step-parallel (4 lanes per (chain, block))")
    ap.add_argument("--fwd-lanes", type=int, default=0, help="lanes per (chain, block) in the forward kernel (0: automatic)")
    ap.add_argument("--eager-noise", action="store_true", help="the sweep stores W_acc / W° (default: lazy noise, rebuilt from X on demand)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy: stats, ll, ll_proposal, "
                         "accepted [n_blocks, M], and X, X_proposal [NP, d, n] of n <= %d chains drawn by np.random.default_rng(0); at "
                         "most %d MB.  Unless --sweeps-per-step is given, R is then a fixed number of sweeps per config so that runs "
                         "with the same arguments run the same sweeps" % (DUMP_SAMPLE_CHAINS, DUMP_MAX_BYTES >> 20))
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none")
    return a


def workload_config(cfg, M_total, prob):
    """the `config` object both arms print: names the BASELINE.json workload, no per-arm detail"""
    from dmt_b200 import _lib
    idx = {"c1": 0, "c2": 1, "c3": 2, "c4": 3, "c5": 4}[cfg]
    name = _lib.MODEL_NAMES[prob.model]
    lay = "/".join(str(len(r)) for r, _ in prob.layouts)
    return {"workload": "BASELINE.json configs[%d] (%s): %s %d-D, %d-chain ensemble, %d obs intervals x %d EM steps, block layouts %s, pCN rho=0.9"
                        % (idx, cfg.upper(), name, prob.d, M_total, prob.K, int(prob.n_pts[0] - 1), lay),
            "config_id": cfg, "total_chains": M_total, "steps_per_chain": prob.steps_per_chain}


# ------------------------------------------------------------------------------------------------ CPU arm (oracle port)
def native_oracle():
    """the OpenMP flavour of the oracle rebuilt for THIS host (-O3 -march=native) in a temporary directory when gcc is present; else the
    shipped generic build"""
    from oracle import orc
    src = os.path.join(ROOT, "oracle", "dmt_oracle.c")
    try:
        with tempfile.TemporaryDirectory() as tmp:   # the loaded library stays mapped after its file is removed
            out = os.path.join(tmp, "libdmt_oracle_omp_native.so")
            subprocess.run(["gcc", "-std=c99", "-O3", "-march=native", "-fopenmp", "-fPIC", "-shared", "-o", out, src, "-lm"], check=True, capture_output=True)
            return orc.load(path=out), "-O3 -march=native -fopenmp"
    except Exception:
        return orc.load(omp=True), "-O3 -fopenmp (generic x86-64)"


def cpu_arm(cfg_name, n_chains, steps, warm, threads=None):
    """Times the C restatement of the reference algorithm (oracle/, OpenMP over recordings) on a bounded sample of the same
    workload: `steps` timed sweeps over `n_chains` chains after `warm` untimed ones; the rate is units / MEDIAN sweep time.
    kind = "port": the Julia reference and its un-vendored numerical dependencies cannot run here."""
    import dmt_b200  # noqa: F401
    from dmt_b200 import configs
    from oracle import orc
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from harness import OracleEnsemble
    import ctypes as C
    threads = threads or os.cpu_count() or 1
    prob = configs.named_config(cfg_name, M=n_chains, seed=123)
    lib, flags = native_oracle()
    ora = OracleEnsemble(orc, lib, prob, seed=123)
    blocking = len(prob.layouts) > 1
    for P in ora.pairs:  # initial paths: whole-path guiding term, fresh noise, forced accept
        bb = P.biblock(0, prob.K - 1, True, 0.0)
        P.recompute_guiding_term(bb, 0)
        tries = 0
        while not P.draw_proposal_path(bb, seed=123, chain=tries, it=9999):
            tries += 1
        P.accept_reject(bb, float("inf"))
        P.loglikhd(bb, 0)
        if not blocking:
            for lay in ora.layouts:
                lay[ora.pairs.index(P)][0].ll[0] = bb.ll[0]
    arr_t = C.c_void_p * len(ora.pairs)
    handles = arr_t(*[P.h for P in ora.pairs])
    gt0 = orc.gtile0_of(prob.n_pts)
    flat = []
    for l, lay in enumerate(ora.layouts):
        nb = len(lay[0])
        blk = (orc.BiBlock * (nb * prob.M))()
        for c in range(prob.M):
            for b in range(nb):
                blk[c * nb + b] = lay[c][b]
        flat.append((blk, nb))
    nacc = C.c_int()

    def sweep(it):
        l = it % len(flat)
        blk, nb = flat[l]
        lib.orc_sweep_many(handles, blk, prob.M, nb, 123, 0, it, l, gt0.ctypes.data_as(C.POINTER(C.c_int)), int(blocking), threads, C.byref(nacc))
    for it in range(warm):
        sweep(it)
    times = []
    for it in range(warm, warm + steps):
        t0 = time.perf_counter()
        sweep(it)
        times.append(time.perf_counter() - t0)
    med = float(np.median(times))
    units = prob.M * prob.steps_per_chain
    sample = "%d of the ensemble's chains x %d timed sweeps (+%d warm-up) of config %s (%d EM steps per chain and sweep), %d OpenMP threads, gcc %s; rate from the median sweep time (min %.3f s, max %.3f s)" % (
        prob.M, steps, warm, cfg_name, prob.steps_per_chain, threads, flags, min(times), max(times))
    return {"value": units / med, "s_per_step": med, "threads": threads, "sample": sample, "total_s": float(sum(times)), "prob": prob}


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0=0.0, t1=1e300):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            if not (t0 <= ts <= t1):
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
                for nme, val in zip(names, r[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ GPU arm
class Runner:
    """one device context holding `M` chains of config `cfg` (global chain ids lo .. lo + M - 1) and the sweep loop over it"""

    def __init__(self, a, cfg, M, lo, local, rank, world, dev):
        import torch
        import torch.distributed as dist
        import dmt_b200
        from dmt_b200 import _lib, configs
        self.a, self.torch, self.dist, self._lib = a, torch, dist, _lib
        self.rank, self.world, self.dev, self.lo = rank, world, dev, lo
        self.prob = prob = configs.named_config(cfg, M=M, seed=0, chain_offset=lo, P=a.psets)
        self.blocking = len(prob.layouts) > 1
        self.nlay = nlay = len(prob.layouts)
        self.ctx = ctx = dmt_b200.Ctx(prob.model, prob.n_pts, prob.tt, prob.M, prob.P, obs_dim=prob.m, device=local, n_layouts=nlay + 1,
                                      chain_offset=lo, seed=2026, pset_of_chain=prob.pset_of_chain)
        configs.upload(prob, ctx)
        ctx.set_sweep_mode(a.sweep_mode)
        if a.fwd_lanes:
            ctx.set_fwd_lanes(a.fwd_lanes)
        self.fused = self.blocking and not a.separate   # find_W_for_X! + loglikhd! + draw_proposal_path! in one pass
        self.lazy = self.fused and not a.eager_noise and prob.P == prob.M
        whole = nlay
        ctx.set_blocks(whole, [(0, prob.K - 1)], 0.0)
        ctx.recompute_guiding_term(whole, _lib.P_ONLY)
        nfail = ctx.init_paths(whole, iter0=1 << 20, max_tries=1000)
        assert nfail == 0, "init_paths left %d failing chains" % nfail
        if not self.blocking:
            ctx.recompute_guiding_term(0, _lib.P_ONLY)
            ctx.loglikhd(0, 0, 0)
        if self.lazy:
            ctx.set_lazy_noise(True)
        self.cached = self.blocking and not a.no_cache
        if self.cached:  # smoothing: the laws stay fixed, only the blocks' frozen end points move => K1 through the guiding cache
            for l in range(nlay):
                ctx.enable_guiding_cache(l)
        self.allreduce_kind = "none"
        if world > 1:
            self._join_ranks()
        self.stream = torch.cuda.ExternalStream(ctx.stream(), device=dev)
        self.k1_each_step = (cfg == "c5")    # BASELINE C5: "each sweep = set_params -> K1 (P = M) -> K2" (backward-filter dominated)
        self.theta_host = np.repeat(prob.theta[:, None], prob.P, axis=1).copy()
        self.onecall = self.fused and a.one_call
        if self.onecall:
            self.names = ["sweep_fused", "accept", "stats"]
        elif self.fused:
            self.names = ["set_obs", "bwd_filter", "sweep_fused", "accept", "stats"]
        elif self.k1_each_step:
            self.names = ["set_params_aux", "bwd_filter", "draw", "accept", "stats"]
        else:
            self.names = (["set_obs", "bwd_filter", "invsolve_ll"] if self.blocking else []) + ["draw", "accept", "stats"]
        self.ev = {n: [] for n in self.names}

    def _join_ranks(self):
        """the small stats all-reduce as the library's own one-shot kernel over NVLink peer memory (dmt_p2p_init); if any rank cannot
        map its peers (IPC not permitted), every rank falls back to the NCCL communicator inside libdmt"""
        torch, dist, ctx, dev, world, rank = self.torch, self.dist, self.ctx, self.dev, self.world, self.rank
        ok = torch.ones(1, device=dev)
        if os.environ.get("DMT_NO_P2P"):
            ok.zero_()
        else:
            try:
                mine = torch.from_numpy(ctx.p2p_export().copy()).to(dev)
            except Exception:
                mine = torch.zeros(64, dtype=torch.uint8, device=dev)
                ok.zero_()
            allh = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(allh, mine)
            if ok.item():
                try:
                    ctx.p2p_init(world, rank, np.stack([h.cpu().numpy() for h in allh]))
                except Exception:
                    ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if ok.item():
            self.allreduce_kind = "p2p kernel (NVLink peer memory)"
        else:
            ctx.p2p_disable()
            uid = torch.from_numpy(ctx.nccl_unique_id() if rank == 0 else np.zeros(128, np.uint8)).to(dev)
            dist.broadcast(uid, 0)
            ctx.comm_init(world, rank, uid.cpu().numpy())
            self.allreduce_kind = "ncclAllReduce"

    def sweep(self, it, timed, E=None):
        ctx, _lib, torch = self.ctx, self._lib, self.torch
        l = it % self.nlay
        marks = []

        def mark():
            if timed:
                e = torch.cuda.Event(enable_timing=True); e.record(self.stream); marks.append(e)
        mark()
        if self.onecall:
            ctx.blocking_sweep(l, it); mark()   # set_obs!, recompute_guiding_term!(P only), find_W_for_X!, loglikhd!, draw_proposal_path!
        elif self.blocking:
            ctx.set_artificial_obs(l); mark()
            ctx.recompute_guiding_term(l, _lib.P_ONLY); mark()
            if self.fused:
                ctx.find_W_loglikhd_draw(l, it); mark()
            else:
                ctx.find_W_and_loglikhd(l); mark()
        if self.k1_each_step:  # new parameters, aux laws re-linearised on the device, K1, then the path update
            ctx.set_params(self.theta_host, side=0, stores=1)
            ctx.set_aux_linearised(None, side=0, store=_lib.STORE_PP); mark()
            ctx.recompute_guiding_term(l, _lib.P_ONLY); mark()
        if not self.fused:
            ctx.draw_proposal_path(l, it); mark()
        ctx.accept_reject_path(l, it, E); mark()   # E: host-drawn Exp(1) (the reference's rand(Exponential(1.0)), src/biblock.jl:122) or device Philox
        stats = ctx.allreduce_stats(l); mark()     # [sum ll, sum ll°, accept counts...] summed over the ranks when N > 1
        if timed:
            for n, e0, e1 in zip(self.names, marks[:-1], marks[1:]):
                self.ev[n].append((e0, e1))
        return stats

    def barrier(self):
        self.ctx.sync(); self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.ctx.sync(); self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed_run(self, it0, n_steps, R, timed_kernels=True, E_np=None, readback=False):
        """n_steps steps of R sweeps between two events on the library's stream -> (device ms, wall s [both max over ranks], last stats, it)"""
        torch = self.torch
        self.barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        t0w = time.perf_counter()
        e0.record(self.stream)
        last, it = None, it0
        for _ in range(n_steps):
            for _ in range(R):
                l = it % self.nlay
                last = self.sweep(it, timed_kernels, None if E_np is None else E_np[l])
                if readback:
                    self.ctx.get_ll(l, 0); self.ctx.get_last_accept(l)
                it += 1
        e1.record(self.stream)
        self.barrier()
        wall = time.perf_counter() - t0w
        return self.max_over_ranks(e0.elapsed_time(e1)), self.max_over_ranks(wall), last, it

    def kernel_ms(self):
        return {n: float(np.mean([a.elapsed_time(b) for a, b in self.ev[n]])) for n in self.names if self.ev[n]}


def self_check(run, it):
    """(1) the all-reduced sum of ll equals the sum over ranks of the per-(block, chain) values each rank holds; (2) three of rank 0's
    chains replayed for one sweep on the CPU oracle (a CHECKER, outside every timed region): ll, ll°, X° and the decisions."""
    torch, dist, ctx, prob = run.torch, run.dist, run.ctx, run.prob
    l = it % run.nlay
    stats = run.sweep(it, False)
    loc = np.array([ctx.get_ll(l, 0).sum(), ctx.get_ll(l, 1).sum(), float(ctx.get_last_accept(l).sum())])
    t = torch.from_numpy(loc).to(run.dev)
    if run.world > 1:
        dist.all_reduce(t)
    glob = t.cpu().numpy()
    fin = np.isfinite(glob[:2])
    rel = float(np.max(np.abs(glob[:2][fin] - stats[:2][fin]) / np.maximum(1.0, np.abs(glob[:2][fin])))) if fin.any() else 0.0
    out = {"allreduce_vs_gathered_rel_diff": rel, "accept_count_equal": bool(abs(glob[2] - stats[2:].sum()) < 0.5),
           "allreduce_ok": bool(rel < 1e-9 and abs(glob[2] - stats[2:].sum()) < 0.5)}
    if run.rank == 0 and run.blocking and not run.k1_each_step:
        try:
            import copy
            from oracle import orc
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            from harness import OracleEnsemble, rel_err
            olib = orc.load()
            chains = sorted({0, prob.M // 2, prob.M - 1})
            sub = copy.copy(prob)
            sub.M = sub.P = len(chains)
            sub.v, sub.xbar, sub.x0 = prob.v[:, :, chains].copy(), prob.xbar[:, :, chains].copy(), prob.x0[:, chains].copy()
            gids = [run.lo + c for c in chains]
            ora = OracleEnsemble(orc, olib, sub, seed=2026, chain_ids=gids)
            X = ctx.get_X_chains(chains, 0)
            for s in (0, 1):
                ora.set_X(s, X)
            it2 = it + 1
            l2 = it2 % run.nlay
            ctx.blocking_sweep(l2, it2)
            ora.set_artificial_obs(l2); ora.recompute_guiding_term(l2); ora.find_W_for_X(l2); ora.loglikhd(l2); ora.draw(l2, it2)
            e = max(rel_err(ctx.get_ll(l2, 0)[:, chains], ora.ll(l2, 0)), rel_err(ctx.get_ll(l2, 1)[:, chains], ora.ll(l2, 1)),
                    rel_err(ctx.get_X_chains(chains, 1), ora.X(1)))
            ctx.accept_reject_path(l2, it2)
            acc_o, _ = ora.accept(l2, it2)
            same = bool(np.array_equal(ctx.get_last_accept(l2)[:, chains], acc_o))
            out["oracle_replay"] = {"global_chains": gids, "max_rel_err": e, "decisions_equal": same, "ok": bool(e < 1e-9 and same)}
        except Exception as ex:  # the bench number does not depend on the checker; say what happened
            out["oracle_replay"] = {"ok": False, "error": repr(ex)}
    if run.world > 1:  # every rank took part in the collective part above; keep them in step
        dist.barrier()
    return out


def dump_last_step(run, l, stats, out_dir):
    """what the last timed sweep (layout l) left for its caller: the all-reduced stats, per-(block, chain) ll / ll° and decisions,
    and the accepted / proposed paths of a fixed sample of chains"""
    ctx, prob = run.ctx, run.prob
    out = {"stats": np.asarray(stats, dtype=np.float64), "ll": ctx.get_ll(l, 0), "ll_proposal": ctx.get_ll(l, 1),
           "accepted": ctx.get_last_accept(l).astype(np.float32)}
    fixed = sum(v.nbytes for v in out.values())
    per_chain = 2 * 8 * ctx.NP * prob.d
    n = min(prob.M, DUMP_SAMPLE_CHAINS, max(0, (DUMP_MAX_BYTES - fixed) // per_chain))
    if n == 0:
        raise ValueError("--dump-outputs: the per-chain outputs of %d chains exceed %d MB" % (prob.M, DUMP_MAX_BYTES >> 20))
    chains = np.sort(np.random.default_rng(0).choice(prob.M, n, replace=False))
    out["X"], out["X_proposal"] = ctx.get_X_chains(chains, 0), ctx.get_X_chains(chains, 1)
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def gpu_arm(a):
    import torch
    import torch.distributed as dist
    import dmt_b200  # noqa: F401
    from dmt_b200 import _lib, host

    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    M_total = TOTAL_CHAINS[a.config]
    if a.chains:   # explicit chains per GPU: weak scaling
        scaling, M, lo, M_job = "weak", a.chains, rank * a.chains, a.chains * world
    else:          # the config's ensemble, one contiguous slice per GPU
        lo, hi = host.shard_slice(M_total, rank, world)
        scaling, M, M_job = "strong", hi - lo, M_total
    run = Runner(a, a.config, M, lo, local, rank, world, dev)
    prob, ctx = run.prob, run.ctx
    blocking, fused, lazy = run.blocking, run.fused, run.lazy

    sampler = ClockSampler(local)
    sampler.start()  # nvidia-smi takes a moment to start: launch it before the warm-up, keep only the timed window
    it = 0
    R = max(1, a.sweeps_per_step)
    for _ in range(max(a.warmup, 3)):   # warm-up steps (cover the guiding-cache build on both layouts)
        for _ in range(max(R, run.nlay)):
            run.sweep(it, False); it += 1
    if a.sweeps_per_step <= 0 and a.dump_outputs:
        R = max(1, int(math.ceil(DUMP_TIMED_SWEEPS[a.config] / a.steps)))
    elif a.sweeps_per_step <= 0:        # estimate the sweep time, then fix R for the timed region
        ms_est, _, _, it = run.timed_run(it, 1, 2 * run.nlay, timed_kernels=False)
        per_sweep = ms_est / (2 * run.nlay) * 1e-3
        R = int(run.max_over_ranks(max(1, int(math.ceil(MIN_TIMED_S / (a.steps * per_sweep))))))
    n0 = _lib.launch_count()
    t_wall0 = time.time()
    ms_total, _, last, it = run.timed_run(it, a.steps, R)
    t_wall1 = time.time()
    launches = _lib.launch_count() - n0
    clocks = sampler.stop(t_wall0, t_wall1)
    if a.dump_outputs and rank == 0:
        dump_last_step(run, (it - 1) % run.nlay, last, a.dump_outputs)
    units_per_step = R * M_job * prob.steps_per_chain
    value = units_per_step * a.steps / (ms_total * 1e-3)
    ms_per_sweep = ms_total / (a.steps * R)
    kern_ms = run.kernel_ms()
    fwd_kernel_name = run.ctx.last_forward_kernel()

    # ---- roofline of the dominant kernel
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    d, dw = prob.d, prob.dw
    nh = d * (d + 1) // 2
    g_bytes = 8 * (nh + d) if prob.P == prob.M else 0
    bsh, bper = ALGO_BYTES[a.config]
    bpu = bper if prob.P == prob.M else bsh
    kname, kop = "draw", "OP_DRAW"
    if fused:
        # fused pass: reads X_acc and H,F; writes X° (+ W_acc, W° unless the noise is lazy); the accepted noise stays in registers
        bpu = 8 * (2 * d + (0 if lazy else 2 * dw)) + g_bytes
        kname, kop = "sweep_fused", "OP_SWEEP"
    units_per_launch = prob.M * prob.steps_per_chain
    algo_bytes = bpu * units_per_launch
    achieved = algo_bytes / (kern_ms[kname] * 1e-3) / 1e9 if kname in kern_ms else None
    kernel_name = "%s [%s]" % (fwd_kernel_name, _lib.MODEL_NAMES[prob.model])   # as reported by the library (dmt_get_last_forward_kernel)
    roofline = {"kernel": kernel_name, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak if achieved else None, "traffic": None,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                "algorithmic_bytes_per_unit": bpu, "units_per_launch": units_per_launch, "launch_ms": kern_ms.get(kname)}
    try:  # dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel, from the committed `ncu --set full` capture
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        ent = tr.get(roofline["kernel"])
        if ent and ent.get("units_per_launch") == roofline["units_per_launch"]:
            roofline["traffic"] = ent["dram_bytes_per_launch"]
            roofline["traffic_source"] = ent["source"]
    except Exception:
        pass
    if blocking:
        # whole sweep on the bytes the ALGORITHM needs: the fused pass (bpu); a run whose laws change pays the backward filter's H,F
        # write on top (8(d(d+1)/2 + d) B per step).  The cache's own F0 / Psi reads are NOT counted as useful bytes.
        need = bpu if fused else (8 * (d + dw) + g_bytes) + bpu
        roofline["step"] = {"needed_bytes_per_unit": need, "ms_per_sweep": ms_per_sweep,
                            "achieved": need * units_per_launch / (ms_per_sweep * 1e-3) / 1e9,
                            "frac": need * units_per_launch / (ms_per_sweep * 1e-3) / 1e9 / peak,
                            "k1": "guiding cache (F = F0 + Psi v)" if run.cached else "full backward filter"}

    # ---- end to end through the C ABI with HOST buffers: every sweep the accept step's Exp(1) draws come from pinned host memory
    # (H2D inside dmt_accept_reject_path, as rand(Exponential(1.0)) in the reference) and the per-(block, chain) ll and accept flags
    # are read back (D2H); paths stay on the device (the tutorials read them every 400th iteration)
    e2e = None
    if not a.no_e2e:
        nb_l = [len(r) for r, _ in prob.layouts]
        rng = np.random.default_rng(7)
        E_pinned = [torch.empty((nb, prob.M), dtype=torch.float64, pin_memory=True) for nb in nb_l]
        for t in E_pinned:
            t.copy_(torch.from_numpy(rng.exponential(size=tuple(t.shape))))
        n_e2e = max(3, a.steps // 2)
        _, wall, _, it = run.timed_run(it, n_e2e, R, timed_kernels=False, E_np=[t.numpy() for t in E_pinned], readback=True)
        e2e = {"value": units_per_step * n_e2e / wall, "unit": UNIT,
               "h2d_bytes_per_step": int(R * np.mean(nb_l) * prob.M * 8), "d2h_bytes_per_step": int(R * (np.mean(nb_l) * prob.M * 9 + 8 * (2 + np.mean(nb_l)))),
               "steps": n_e2e, "timed_s": wall,
               "note": "per GPU and sweep: host-drawn E (pinned) -> dmt_accept_reject_path, dmt_get_ll + dmt_get_last_accept + stats read back; wall clock between barriers, max over ranks"}

    # ---- the same sweep with the FULL backward filter (what any run with changing theta pays): K1 ms, rate, fraction on needed bytes
    if run.cached and not a.no_uncached:
        for l in range(run.nlay):
            ctx.enable_guiding_cache(l, False)
        run.cached = False
        for n in run.names:
            run.ev[n] = []
        for _ in range(run.nlay):
            run.sweep(it, False); it += 1
        n_unc = 3 * run.nlay
        ms_u, _, _, it = run.timed_run(it, 1, n_unc)
        ku = run.kernel_ms()
        need_u = bpu + 8 * (nh + d)
        roofline["uncached"] = {
            "ms_per_sweep": ms_u / n_unc, "value": n_unc * M_job * prob.steps_per_chain / (ms_u * 1e-3), "k1_ms": ku.get("bwd_filter"),
            "needed_bytes_per_unit": need_u, "frac": need_u * units_per_launch / (ms_u / n_unc * 1e-3) / 1e9 / peak,
            "k1_write_frac": 8 * (nh + d) * units_per_launch / (ku["bwd_filter"] * 1e-3) / 1e9 / peak if ku.get("bwd_filter") else None,
            "k1_bound": "FP64 pipe (RK4 on the Riccati system), not HBM", "sweeps": n_unc}

    check = None if a.no_self_check else self_check(run, it)

    cfg = workload_config(a.config, M_job, prob)
    cfg.update({"chains_per_gpu": prob.M, "parameter_sets_per_gpu": prob.P, "sweeps_per_step": R,
                "step": ("%d blocking sweep(s), layouts alternating" % R) if blocking else ("%d x (draw + accept)" % R),
                "noise": "lazy (W rebuilt from X on demand, dmt_set_lazy_noise)" if lazy else "eager (W_acc, W° stored every sweep)",
                "l2": "per-GPU inputs (paths %.2f GB + guiding term %.2f GB) exceed the 126 MB L2; nothing is reused between sweeps"
                      % (2 * 8 * ctx.S * (d + dw) * prob.M / 1e9, 8 * ctx.S * (nh + d) * prob.P / 1e9),
                "stats_allreduce": run.allreduce_kind})
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg, "roofline": roofline, "ms_per_sweep": ms_per_sweep, "timed_region_s": ms_total * 1e-3, "kernel_ms": kern_ms,
        "gpu_launches": int(launches), "clocks": clocks,
        "last_stats": {"sum_ll": float(last[0]), "sum_ll_prop": float(last[1]), "accept_frac": float(np.sum(last[2:]) / (len(last[2:]) * M_job))},
    }
    if e2e:
        out["e2e"] = e2e
    if check:
        out["self_check"] = check

    # ---- N > 1: the weak-scaling rate as an extra (the config's full ensemble on EVERY GPU)
    ctx.close()
    if world > 1 and scaling == "strong" and not a.no_weak:
        wrun = Runner(a, a.config, M_total, rank * M_total, local, rank, world, dev)
        itw = 0
        for _ in range(3 * wrun.nlay):
            wrun.sweep(itw, False); itw += 1
        ms_est, _, _, itw = wrun.timed_run(itw, 1, 2 * wrun.nlay, timed_kernels=False)
        nw = int(wrun.max_over_ranks(max(2 * wrun.nlay, math.ceil(1.0 / (ms_est / (2 * wrun.nlay) * 1e-3)))))
        ms_w, _, _, itw = wrun.timed_run(itw, 1, nw, timed_kernels=False)
        out["weak_scaling"] = {"value": nw * M_total * world * wrun.prob.steps_per_chain / (ms_w * 1e-3), "unit": UNIT, "chains_per_gpu": M_total,
                               "ms_per_sweep": ms_w / nw, "sweeps": nw}
        wrun.ctx.close()

    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        nch = a.cpu_chains or min(512, 16 * (os.cpu_count() or 1))
        r = cpu_arm(a.config, nch, steps=5, warm=1)
        out["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["threads"], "kind": "port", "sample": r["sample"],
                               "note": "C restatement of the reference algorithm (oracle/), not the Julia package: Julia is not installed"}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(out))


def reference_arm(a):
    """the reference's CPU implementation of the path on the box's host cores: K timed steps (one sweep over the bounded sample each)
    after W warm-up steps; rank 0 alone works"""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    nch = a.cpu_chains or min(512, 16 * (os.cpu_count() or 1))
    M_total = TOTAL_CHAINS[a.config]
    r = cpu_arm(a.config, nch, steps=max(1, a.steps), warm=max(0, a.warmup))
    cfg = workload_config(a.config, M_total, r["prob"])
    cfg.update({"sweeps_per_step": 1, "step": "1 blocking sweep over the bounded sample" if len(r["prob"].layouts) > 1 else "draw + accept over the bounded sample"})
    cb = {"value": r["value"], "unit": UNIT, "cores": r["threads"], "kind": "port", "sample": r["sample"]}
    out = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": max(1, a.steps), "warmup": max(0, a.warmup),
           "ms_per_step": r["s_per_step"] * 1e3, "timed_region_s": r["total_s"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic", "config": cfg, "cpu_baseline": cb,
           "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
           "note": "reference arm = C restatement of the reference algorithm (oracle/, OpenMP over recordings) on the host cores; the Julia reference cannot run in this image (no Julia, un-vendored dependencies)"}
    print(json.dumps(out))


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)
