"""Cost of the posterior path moments (dmt_path_moments_add) on the C3 ensemble: 4096 Lorenz chains, 200 intervals of 100 steps,
two staggered block layouts, K1 through the guiding cache, lazy noise — the configuration bench.py measures.

Reports, on the library's stream (dmt_get_stream) with CUDA events:
  - the time of one dmt_path_moments_add over a window of >= 2.5 s, its rate on the algorithmic bytes
    (40 d B per point: X read 8 d, mean / m2 read 16 d and written 16 d) and the fraction of 6545.3 GB/s (the copy peak);
  - the blocking-sweep rate (dmt_blocking_sweep + dmt_accept_reject_path) with no accumulation, with an update after every sweep
    and with one every 10 sweeps, the three runs alternating.
The card's name, power limit and maximum SM clock (read-only nvidia-smi query) go beside the numbers.  One JSON line is printed and
written to <out>/path_moments_bench.json; nothing is written into the repository.

    python scripts/path_moments_bench.py --out <dir> [--chains 4096] [--window 2.5] [--sweeps 300] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.dont_write_bytecode = True

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

COPY_PEAK_GBS = 6545.3


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        name, plim, mx = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit_w": float(plim), "sm_max_mhz": float(mx)}
    except Exception as e:  # the numbers are still printed, flagged as without card information
        return {"name": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory for the JSON line")
    ap.add_argument("--chains", type=int, default=4096)
    ap.add_argument("--window", type=float, default=2.5, help="seconds of dmt_path_moments_add in the timed window (minimum)")
    ap.add_argument("--sweeps", type=int, default=300, help="sweeps per sweep-rate run")
    ap.add_argument("--reps", type=int, default=3, help="rounds of the three alternating sweep-rate runs")
    a = ap.parse_args()

    import torch
    import dmt_b200
    from dmt_b200 import _lib, configs
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the GPU and has nothing to fall back to")

    prob = configs.named_config("c3", M=a.chains, seed=0)
    nlay = len(prob.layouts)
    ctx = dmt_b200.Ctx(prob.model, prob.n_pts, prob.tt, prob.M, prob.P, obs_dim=prob.m, n_layouts=nlay + 1, seed=2026,
                       pset_of_chain=prob.pset_of_chain)
    configs.upload(prob, ctx)
    ctx.set_blocks(nlay, [(0, prob.K - 1)], 0.0)
    ctx.recompute_guiding_term(nlay, _lib.P_ONLY)
    assert ctx.init_paths(nlay, iter0=1 << 20, max_tries=1000) == 0
    ctx.set_lazy_noise(True)
    for l in range(nlay):
        ctx.enable_guiding_cache(l)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=0)
    M, d, S, K = prob.M, prob.d, prob.steps_per_chain, prob.K
    bytes_per_update = 40 * d * (S + K) * M
    steps_per_sweep = S * M

    it = 0

    def sweeps(n, every):
        nonlocal it
        for _ in range(n):
            l = it % nlay
            ctx.blocking_sweep(l, it)
            ctx.accept_reject_path(l, it)
            if every and it % every == 0:
                ctx.path_moments_add()
            it += 1

    def timed(fn):
        ctx.sync(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e-3

    # warm-up: sweeps (guiding caches built), the first update (allocation, n == 1 branch) and steady-state updates
    sweeps(20, 0)
    ctx.path_moments_add()
    est = timed(lambda: [ctx.path_moments_add() for _ in range(20)]) / 20
    n_add = max(20, int(np.ceil(a.window / est)))
    t_add = timed(lambda: [ctx.path_moments_add() for _ in range(n_add)])
    add_s = t_add / n_add
    gbs = bytes_per_update / add_s / 1e9

    # sweep rates, the three variants alternating
    variants = {"none": 0, "every_sweep": 1, "every_10": 10}
    sweeps(20, 1)
    runs = {k: [] for k in variants}
    for _ in range(a.reps):
        for k, every in variants.items():
            ctx.path_moments_reset()
            t = timed(lambda: sweeps(a.sweeps, every))
            runs[k].append(steps_per_sweep * a.sweeps / t)
    rate = {k: float(np.median(v)) for k, v in runs.items()}
    ctx.close()

    res = {
        "what": "dmt_path_moments_add on C3 (Lorenz, %d chains, %d intervals, %d steps per chain; 2 staggered layouts, cached K1, lazy noise)"
                % (M, K, S),
        "card": card(),
        "moments_add_ms": add_s * 1e3,
        "moments_add_window_s": t_add, "moments_add_launches_timed": n_add,
        "algorithmic_bytes_per_update": bytes_per_update,
        "moments_add_GBps": gbs,
        "fraction_of_copy_peak": gbs / COPY_PEAK_GBS, "copy_peak_GBps": COPY_PEAK_GBS,
        "sweep_steps_per_s": rate,
        "sweep_steps_per_s_all_runs": runs,
        "sweep_ms": {k: steps_per_sweep / v * 1e3 for k, v in rate.items()},
        "sweep_note": "blocking_sweep + accept_reject_path per sweep, %d sweeps per run, %d alternating rounds, median" % (a.sweeps, a.reps),
        "time": time.strftime("%Y-%m-%d %H:%M:%S"),
    }
    line = json.dumps(res)
    print(line)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "path_moments_bench.json"), "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
