// sweep_kernel.cuh — the blocking sweep's fused forward pass (K5 + K4 + K3 + K2 + K4), software-pipelined.
//
// Same arithmetic as fwd_kernel<MD, OP_SWEEP> (fwd_kernel.cuh) and the same reference calls
//   find_W_for_X!(b); loglikhd!(b); draw_proposal_path!(bb)   (/root/reference/docs/src/tutorials/block_collection/inference_with_blocking.md:55-57,
//   /root/reference/src/block.jl:120-152, /root/reference/src/biblock.jl:80-106),
// but a different memory schedule.  Round 1 measured (profiles/r01_tuning.md) that with ~2.4 warps per scheduler the register-tile
// kernel ADDS its memory time and its issue time per 4-step tile (4.4 us + 2.2 us per tile round and SM): every warp issues its 12
// sector loads and then has nothing to run until they land.  Here every input of tile t+1 is already in flight while tile t is
// computed, with NO extra registers for the widest stream:
//   * H, F (d(d+1)/2 + d sectors per lane and tile) and the tile's dt / sqrt(dt) travel global -> shared through the TMA unit
//     (cp.async.bulk, one mbarrier per stage, two stages per warp): with one parameter set per chain in chain order a warp's sectors of
//     one component are 1 KiB contiguous, so lane 0 issues d(d+1)/2 + d + 2 bulk copies per tile and the step loop reads the guiding
//     term in place from shared memory;
//   * the accepted path X (d sectors; per-chain buffer parity, so not contiguous across lanes) is double-buffered in registers;
//   * the per-interval auxiliary-law record (B, beta) lives in shared memory, one column per lane.
// One warp per CTA: a warp owns its ring and its barriers, nothing is shared between warps, and the grid balances at warp granularity.
//
// LAZYW: the sweep does not materialise W_acc and W°.  In the blocking loop find_W_for_X! overwrites b.WW at the start of EVERY sweep
// (inference_with_blocking.md:52-58), so neither array is ever read; dmt_get_W / draws without K5 rebuild W from X on demand
// (dmt_api.cu, ensure_W).  120 instead of 168 B per step.
#pragma once
#include "fwd_kernel.cuh"
#include <type_traits>

namespace dmt {

// compile-time loop: the body receives std::integral_constant<int, I>
template <int N, int I = 0, class F> __device__ __forceinline__ void static_for(F &&f) {
    if constexpr (I < N) {
        f(std::integral_constant<int, I>{});
        static_for<N, I + 1>(f);
    }
}

// One lane of a converged warp, chosen by the hardware (elect.sync).  With `if (lane == 0)` ptxas cannot know that a single lane is active and
// wraps EVERY bulk copy — a uniform-datapath instruction — in its own elect-one loop (R2UR ... ELECT ... BRA.U.ANY, ~12 instructions per copy,
// 11 copies per tile); behind elect.sync the operands are uniform by construction.
__device__ __forceinline__ bool elect_one_lane() {
    uint32_t pred;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
    return pred != 0;
}
template <class MD> constexpr int sweep_pipe_minb() { return MD::D <= 3 ? 10 : 1; } // 10 warps per SM at <= 200 registers: C3 in one wave

template <class MD> __host__ __device__ constexpr size_t sweep_pipe_smem() { // one warp's ring, law record and barriers; a multiple of 128 bytes
    constexpr int D = MD::D, NG = D * (D + 1) / 2 + D;
    return ((size_t)2 * (NG * 128 + 8) * 8 + (size_t)(D * D + D) * 32 * 8 + 2 * 8 + 127) / 128 * 128;
}

// Which warp runs which interval of which (32-chain group, block) unit.
// Without `task`: one unit per warp, blockIdx = (chain group, block), its intervals in order.
// With `task` the grid is persistent.  A task is one interval of one unit; tickets are dealt interval-major: ticket t is chain
// group t % G of entry task[t / G], an entry being (block b, interval j of the block) packed as b + 64 j, every block's first interval
// first, then every block's second, and so on.  A warp takes a ticket whenever it has issued the loads of its current task's last
// tile, runs the task, and hands the chains' state on to whichever warp holds the unit's next interval.
// Every wait ends, also when not all warps are resident (another job on the GPU): a warp waits only for the previous interval of its
// unit, whose ticket is smaller.  A ticket is taken only by a running warp, so tickets below one that was taken are all held by
// running warps, and a warp runs its tasks in ticket order.  By induction on the ticket: the task with ticket t starts once the
// holder's previous task (smaller ticket) and the unit's previous interval (smaller ticket) are done, then runs without waiting.
struct PipeSched {
    const int *task;    // [entries] b + 64 j, round-major; null: one unit per warp
    int n_tasks;        // entries x chain groups
    unsigned *ticket;   // [1 + units]: the ticket counter, then the intervals each unit has completed; zero at launch
    double *hand;       // [D + 3][units][32]: xo, ll, llo, ok of every chain at the end of its unit's last completed interval
};

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned *p, unsigned v) { asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }

// One lane per (chain, block), 32 chains per warp, WPC independent warps per CTA (4: two CTAs per SM put exactly two warps on every
// scheduler).  Unit u = block * G + chain group, G = ceil(M / 32).
template <class MD, bool LAZYW, int WPC>
__global__ void __launch_bounds__(32 * WPC, WPC == 1 ? sweep_pipe_minb<MD>() : 2)
    sweep_pipe_kernel(const DevCtx cx, const LayoutDev ly, const FwdArgs fa, const PipeSched sc) {
    constexpr int D = MD::D, DW = MD::DW, NPAR = MD::NPAR, NH = D * (D + 1) / 2, NG = NH + D, NAUX = D * D + D + NH;
    constexpr int STAGE = NG * 128 + 8; // doubles per stage: [component][lane][4] then dt[4], sqrt(dt)[4]
    extern __shared__ __align__(128) unsigned char sw_smem[];
    const int lane = threadIdx.x & 31;
    double *ring = reinterpret_cast<double *>(sw_smem + (threadIdx.x >> 5) * sweep_pipe_smem<MD>());
    double *cst = ring + 2 * STAGE;                                  // [D*D + D][32]: B (row-major), beta of the current interval
    uint64_t *bars = reinterpret_cast<uint64_t *>(cst + (D * D + D) * 32);
    const size_t M = cx.M, P = cx.P;
    const int G = (cx.M + 31) >> 5;
    const size_t gstr = P * 4;
    const bool tickets = sc.task != nullptr;

    if (lane == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncwarp();

    // ---- prefetch cursor: the tile after the one being computed, of task (un, kn); the task of each stage in (tu, tk)
    int un, kn;
    bool more = true;
    auto take_ticket = [&]() { // the next task, or more = false
        unsigned t = 0;
        if (lane == 0) t = atomicAdd(sc.ticket, 1u);
        t = __shfl_sync(0xffffffffu, t, 0);
        if (t >= (unsigned)sc.n_tasks) { more = false; return; }
        const int e = (int)(t / (unsigned)G), en = sc.task[e], bn = en & 63;
        un = bn * G + (int)(t - (unsigned)e * G);
        kn = ly.i0[bn] + (en >> 6);
    };
    if (tickets) take_ticket();
    else {
        un = blockIdx.y * G + blockIdx.x;
        kn = ly.i0[blockIdx.y];
    }
    int qn = 0, ntl_n = 0, t0_n = 0, n_prod = 0, tu[2] = {0, 0}, tk[2] = {0, 0};
    uint32_t chunk_n = 0;
    const double *gp_n = nullptr, *xin_n = nullptr;
    auto start_cursor = [&]() { // (un, kn) -> the addresses of its tile 0
        const int bn = un / G, c0n = (un - bn * G) * 32, cn = min(c0n + lane, cx.M - 1);
        ntl_n = (cx.nsteps[kn] + 3) >> 2;
        t0_n = cx.tile0[kn];
        chunk_n = 32u * (uint32_t)min(32, cx.M - c0n);
        gp_n = g_tile_of<NG>(cx, ly, kn, ly.i1[bn], ly.last[bn] != 0, 0, c0n).base; // warp-uniform: the chunk of the warp's first chain
        xin_n = cx.X + (size_t)cx.parX[(size_t)kn * M + cn] * cx.Xbuf + ((size_t)t0_n * D * M + cn) * 4;
    };
    if (more) start_cursor();
    double xnx[D][4];
    auto prefetch = [&]() { // issue every load of tile (kn, qn), then advance the cursor
        if (!more) return;
        if (elect_one_lane()) {
            uint64_t *bar = &bars[n_prod & 1];
            double *dst = ring + (size_t)(n_prod & 1) * STAGE;
            mbar_expect_tx(bar, NG * chunk_n + 64u);
#pragma unroll
            for (int a = 0; a < NG; a++) bulk_g2s(dst + a * 128, gp_n + ((size_t)qn * NG + a) * gstr, chunk_n, bar);
            bulk_g2s(dst + NG * 128, cx.dt + (size_t)(t0_n + qn) * 4, 32u, bar);
            bulk_g2s(dst + NG * 128 + 4, cx.sqdt + (size_t)(t0_n + qn) * 4, 32u, bar);
        }
#pragma unroll
        for (int i = 0; i < D; i++) ld256(xin_n + ((size_t)qn * D + i) * M * 4, xnx[i]);
        if (n_prod & 1) { tu[1] = un; tk[1] = kn; } else { tu[0] = un; tk[0] = kn; }
        n_prod++;
        if (++qn == ntl_n) {
            qn = 0;
            if (tickets) take_ticket();
            else if (++kn > ly.i1[blockIdx.y]) more = false;
            if (more) start_cursor();
        }
    };
    prefetch();

    double xo[D], ll = 0.0, llo = 0.0;
    bool ok = true;
    int n_cons = 0;
    while (n_cons < n_prod) { // one task: interval k of unit u, from the tile the next stage holds
        const int u = (n_cons & 1) ? tu[1] : tu[0], k = (n_cons & 1) ? tk[1] : tk[0];
        const int b = u / G, c0 = (u - b * G) * 32;
        const int c_raw = c0 + lane;
        const int c = min(c_raw, cx.M - 1); // lanes beyond the ensemble shadow the last chain and never store
        const bool live = c_raw < cx.M;
        const int ps = c;                   // launch condition: one parameter set per chain, in chain order
        const int i0 = ly.i0[b], i1 = ly.i1[b];
        const bool last = ly.last[b] != 0;
        const double rho = layout_rho(ly, b, c, M), crho = sqrt(1.0 - rho * rho); // per task: a persistent warp changes block
        const GTile<NG> gt = g_tile_of<NG>(cx, ly, k, i1, last, 0, ps);
        double th[NPAR];
        {
            const double *tp = cx.theta[gt.slot][gt.store] + (size_t)k * NPAR * P + ps;
#pragma unroll
            for (int i = 0; i < NPAR; i++) th[i] = tp[(size_t)i * P];
        }
        const typename MD::Par par(th);
        {   // B, beta of this interval's auxiliary law -> this lane's column of the shared record
            const double *ap = cx.aux[gt.slot][gt.store] + (size_t)k * NAUX * P + ps;
#pragma unroll
            for (int i = 0; i < D * D + D; i++) cst[i * 32 + lane] = ap[(size_t)i * P];
        }
        double at[NH];
        if (!MD::CONSTDIFF) {
            const double *ap = cx.aux[gt.slot][gt.store] + (size_t)k * NAUX * P + ps;
#pragma unroll
            for (int i = 0; i < NH; i++) at[i] = ap[(size_t)(D * D + D + i) * P];
        }
        const int nst = cx.nsteps[k], t0 = cx.tile0[k];
        const uint8_t pw = cx.parW[(size_t)k * M + c], px = cx.parX[(size_t)k * M + c];
        double *Wacc = cx.W + (size_t)pw * cx.Wbuf + ((size_t)t0 * DW * M + c) * 4;
        double *Wprop = cx.W + (size_t)(1 ^ pw) * cx.Wbuf + ((size_t)t0 * DW * M + c) * 4;
        double *Xout = cx.X + (size_t)(1 ^ px) * cx.Xbuf + ((size_t)t0 * D * M + c) * 4;
        double x[D]; // interval k starts at ITS OWN XX[k].x[1]; the block's y1 = XX[1].x[1] at k = i0  (src/biblock.jl:96, src/block.jl:177)
#pragma unroll
        for (int i = 0; i < D; i++) x[i] = cx.X0[(size_t)px * cx.X0buf + ((size_t)k * D + i) * M + c];
        if (k == i0) {
#pragma unroll
            for (int i = 0; i < D; i++) xo[i] = x[i];
            ok = true;
        }
        const int ntl = (nst + 3) >> 2;
        for (int q = 0; q < ntl; ++q) {
            double xt[D][4];
#pragma unroll
            for (int i = 0; i < D; i++)
#pragma unroll
                for (int s = 0; s < 4; s++) xt[i][s] = xnx[i][s];
            prefetch(); // tile t+1: its stage was drained at the end of tile t-1 (the __syncwarp below)
            if (q == ntl - 1 && n_prod == n_cons + 2) { // the next task's law records and start point: pull them into L2 one tile ahead, so
                                                        // that the dependent loads at the interval boundary do not pay a DRAM round trip each
                const int u1 = (n_prod & 1) ? tu[0] : tu[1], k1 = (n_prod & 1) ? tk[0] : tk[1]; // the stage issued last
                const int b1 = u1 / G, c1 = min((u1 - b1 * G) * 32 + lane, cx.M - 1), ps1 = c1;
                const int store1 = (k1 == ly.i1[b1] && !ly.last[b1]) ? 1 : 0;
                const int slot1 = cx.parP[store1][(size_t)k1 * P + ps1];
                const double *tp = cx.theta[slot1][store1] + (size_t)k1 * NPAR * P + ps1;
#pragma unroll
                for (int i = 0; i < NPAR; i++) prefetch_l2(tp + (size_t)i * P);
                const double *ap = cx.aux[slot1][store1] + (size_t)k1 * NAUX * P + ps1;
#pragma unroll
                for (int i = 0; i < (MD::CONSTDIFF ? D * D + D : NAUX); i++) prefetch_l2(ap + (size_t)i * P);
#pragma unroll
                for (int i = 0; i < D; i++) {
                    prefetch_l2(cx.X0 + ((size_t)k1 * D + i) * M + c1);
                    prefetch_l2(cx.X0 + cx.X0buf + ((size_t)k1 * D + i) * M + c1);
                }
                prefetch_l2(cx.parX + (size_t)k1 * M + c1);
                prefetch_l2(cx.parW + (size_t)k1 * M + c1);
            }
            // the tile's normals BEFORE the wait for its data: the generator runs while the sectors are still in flight
            // (measured, profiles/r02_tuning.md: 2.44 ms against 2.61-3.08 ms with the normals generated inside the step loop)
            double z[4 * DW];
            tile_normals<DW>(cx.seed, cx.chain_offset + (uint32_t)c, (uint32_t)(t0 + q), fa.iter, (uint32_t)ly.id, z);
            if (q == 0) {
                if (tickets && k > i0) { // the state at the end of interval k - 1, from the warp that ran it
                    const unsigned *done = sc.ticket + 1 + u;
                    while (ld_acquire_gpu(done) < (unsigned)(k - i0)) __nanosleep(100);
                    const double *h = sc.hand + (size_t)u * 32 + lane;
                    const size_t hs = (size_t)G * ly.nb * 32;
#pragma unroll
                    for (int i = 0; i < D; i++) xo[i] = __ldcg(h + i * hs);
                    ll = __ldcg(h + D * hs);
                    llo = __ldcg(h + (D + 1) * hs);
                    ok = __ldcg(h + (D + 2) * hs) != 0.0;
                    __syncwarp();
                }
                if (live) { // XX°[k].x[1] = y1
                    double *x0p = cx.X0 + (size_t)(1 ^ px) * cx.X0buf + (size_t)k * D * M + c;
#pragma unroll
                    for (int i = 0; i < D; i++) x0p[(size_t)i * M] = xo[i];
                }
            }

            mbar_wait(&bars[n_cons & 1], (uint32_t)(n_cons >> 1) & 1u);
            const double *st = ring + (size_t)(n_cons & 1) * STAGE;
            const double *sg = st + lane * 4;
            n_cons++;
            if (k == i0 && q == 0) { // loglikhd_obs(PP[1], y1) = -c - y'Hy/2 + F'y  (src/block.jl:178)
                double s0 = -*gt.c0;
#pragma unroll
                for (int i = 0; i < D; i++) {
                    double hx = 0.0;
#pragma unroll
                    for (int j = 0; j < D; j++) hx = fma(sg[sidx<D>(i, j) * 128], x[j], hx);
                    s0 += x[i] * (sg[(NH + i) * 128] - 0.5 * hx);
                }
                ll = s0;
                llo = s0; // same law, same start point
            }
            double w[LAZYW ? 1 : DW][4], wo[LAZYW ? 1 : DW][4], xot[D][4];
            // One EM step of the tile.  FULL (every step of the tile exists — always, on grids whose intervals hold a multiple of 4
            // steps): no branch at all, so the four steps and the generator calls they consume form ONE basic block that ptxas can
            // interleave; a failed proposal keeps computing (its state is unspecified anyway) and is marked at the end.
            auto step = [&](auto s_c, auto full_c) {
                constexpr int s = decltype(s_c)::value;
                constexpr bool FULL = decltype(full_c)::value;
                const int i = 4 * q + s;
                if (FULL || i < nst) {
                    double Hs[NH], F[D], Bm[D * D], beta[D], gd[D], G = 0.0;
#pragma unroll
                    for (int a = 0; a < NH; a++) Hs[a] = sg[a * 128 + s];
#pragma unroll
                    for (int a = 0; a < D; a++) F[a] = sg[(NH + a) * 128 + s];
#pragma unroll
                    for (int a = 0; a < D * D; a++) Bm[a] = cst[a * 32 + lane];
#pragma unroll
                    for (int a = 0; a < D; a++) beta[a] = cst[(D * D + a) * 32 + lane];
                    const double dt = st[NG * 128 + s], sq = st[NG * 128 + 4 + s];
                    const typename MD::Diff df(par, x);
                    guided_terms<MD, true>(par, df, Bm, beta, at, Hs, F, x, gd, G);
                    ll = fma(G, dt, ll);
                    double xn[D], res[D], dwv[DW];
#pragma unroll
                    for (int a = 0; a < D; a++) xn[a] = xt[a][s];
#pragma unroll
                    for (int a = 0; a < D; a++) res[a] = xn[a] - x[a] - gd[a] * dt; // K5: dW = sigma^+ (x' - x - (b + a r) dt)   (A.5)
                    df.inv_sig(res, dwv);
#pragma unroll
                    for (int a = 0; a < D; a++) x[a] = xn[a];
                    double dwo[DW];
                    static_for<DW>([&](auto j_c) { // K3: dW° = rho dW + sqrt(1-rho^2) sqrt(dt) xi   (A.2)
                        constexpr int j = decltype(j_c)::value;
                        const double xi = z[s * DW + j];
                        dwo[j] = rho * dwv[j] + crho * sq * xi;
                        if (!LAZYW) { w[j][s] = dwv[j]; wo[j][s] = dwo[j]; }
                    });
                    if (FULL || ok) { // K2 + K4 on the proposal, from the noise just refreshed
                        double swo[D], gdo[D], Go = 0.0, xon[D];
                        const typename MD::Diff dfo(par, xo);
                        guided_terms<MD, true>(par, dfo, Bm, beta, at, Hs, F, xo, gdo, Go);
                        llo = fma(Go, dt, llo);
                        dfo.sig_mul(dwo, swo);
#pragma unroll
                        for (int a = 0; a < D; a++) xon[a] = fma(gdo[a], dt, xo[a]) + swo[a];
                        bool fin = dfo.ok();
#pragma unroll
                        for (int a = 0; a < D; a++) fin = fin && isfinite(xon[a]);
                        ok = ok && fin && MD::bound_ok(par, xon); // src/block.jl:181 (ll° := -Inf once, after the loop)
#pragma unroll
                        for (int a = 0; a < D; a++) { xot[a][s] = xon[a]; xo[a] = xon[a]; }
                    } else {
#pragma unroll
                        for (int a = 0; a < D; a++) xot[a][s] = 0.0;
                    }
                } else {
#pragma unroll
                    for (int a = 0; a < D; a++) xot[a][s] = 0.0;
                    if (!LAZYW) {
#pragma unroll
                        for (int j = 0; j < DW; j++) { w[j][s] = 0.0; wo[j][s] = 0.0; }
                    }
                }
            };
            if (4 * q + 4 <= nst) static_for<4>([&](auto s_c) { step(s_c, std::true_type{}); });
            else static_for<4>([&](auto s_c) { step(s_c, std::false_type{}); });
            if (live) {
                if (!LAZYW) {
#pragma unroll
                    for (int j = 0; j < DW; j++) st256(Wacc + ((size_t)q * DW + j) * M * 4, w[j]);
#pragma unroll
                    for (int j = 0; j < DW; j++) st256(Wprop + ((size_t)q * DW + j) * M * 4, wo[j]);
                }
#pragma unroll
                for (int i = 0; i < D; i++) st256(Xout + ((size_t)q * D + i) * M * 4, xot[i]);
            }
            __syncwarp(); // every lane is done with this stage (and with cst when the interval ends): the next prefetch may refill it
        }
        if (k == i1) {
            if (live) {
                ly.ll[(size_t)b * M + c] = ll;
                ly.ll[((size_t)ly.nb + b) * M + c] = ok ? llo : -INFINITY;
                ly.ok[(size_t)b * M + c] = ok ? 1 : 0;
            }
        } else if (tickets) { // hand the state on: the stores, then the release of the unit's progress word
            double *h = sc.hand + (size_t)u * 32 + lane;
            const size_t hs = (size_t)G * ly.nb * 32;
#pragma unroll
            for (int i = 0; i < D; i++) __stcg(h + i * hs, xo[i]);
            __stcg(h + D * hs, ll);
            __stcg(h + (D + 1) * hs, llo);
            __stcg(h + (D + 2) * hs, ok ? 1.0 : 0.0);
            __syncwarp();
            if (lane == 0) st_release_gpu(sc.ticket + 1 + u, (unsigned)(k - i0 + 1));
        }
    }
}

} // namespace dmt
