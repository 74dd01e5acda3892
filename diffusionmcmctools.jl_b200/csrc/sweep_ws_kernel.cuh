// sweep_ws_kernel.cuh — the blocking sweep's fused forward pass, warp-specialised with mbarrier rings.
//
// Same arithmetic and reference calls as sweep_pipe_kernel / fwd_kernel<MD, OP_SWEEP>
//   find_W_for_X!(b); loglikhd!(b); draw_proposal_path!(bb)   (/root/reference/docs/src/tutorials/block_collection/inference_with_blocking.md:55-57,
//   /root/reference/src/block.jl:120-152, /root/reference/src/biblock.jl:80-106).
//
// Why: of the ~1,700 instructions one lane spends on a 4-step tile only the proposal's Euler-Maruyama RECURSION is sequential in time
// (x°[i+1] needs x°[i]): ~45 instructions per step.  The generator (Philox + Box-Muller, ~960 per tile), the inverse solve K5 and the
// accepted path's likelihood (~330: every step's x[i], x[i+1] are already in memory) and even the PROPOSAL's likelihood (~350: an
// integral over a path that exists once the recursion has passed) are independent across steps.  One-thread-per-(chain, block) kernels
// serialise all of it behind the recursion: when the ensemble is split over 8 GPUs (BASELINE.json north_star: 512 chains x 10 blocks
// per GPU = 160 warps for 592 warp schedulers) the sweep is bound by ONE warp's latency per tile (~6,700 cycles, profiles/r02_tuning.md).
//
// Here a CTA owns one group of 32 chains of one block and its warps form a pipeline over the block's tiles, coupled by shared-memory
// rings with full/empty mbarriers (no block-wide barrier inside the loop, every role runs as far ahead as its ring allows):
//   T  (1 warp, lane 0)  H, F, dt, sqrt(dt) of tile j: global -> shared by TMA bulk copies                    -> G ring (NSG stages)
//   R  (NR <= 6 warps)   the tile's 4 DW normals; warp r evaluates Philox / Box-Muller calls r, r + NR, ...   -> Z ring
//   A  (4 warps)         K5: dW from X, the accepted path's likelihood, the pCN refresh
//                        dW° = rho dW + sqrt(1 - rho^2) sqrt(dt) xi  (A.2), and H, F re-laid out for P             -> D ring
//   P  (1 warp)          the recursion x° += (b + a (F - H x°)) dt + sigma dW°  (A.3) and nothing else; stores X° (W°) -> X ring
//   L  (4 warps)         the proposal's likelihood (A.4) and its failure flags from the X ring, behind P
// P and R map one lane to one chain.  A and L have no recursion to respect, so they map one lane to one (chain, STEP): a warp covers
// 8 chains x the tile's 4 steps, and lane l reads element l of each 1 KiB guiding-term chunk [chain][4 steps] — conflict-free
// shared-memory access where the lane-per-chain mapping has a 4-way bank conflict (32-byte lane stride).  The Z / D / X rings are
// stored [row][36] (row = step x component, 4 pad words): both the lane-per-chain and the (chain, step) accesses are conflict-free.
// Every loop body is kept small on purpose: with one warp per role nothing hides an instruction fetch, and the first version of this
// kernel (fully unrolled tiles, 69 KB of SASS) spent 40 % of its stall samples on "no instruction" (L0 i-cache 6 KB, L1.5 32 KB).
// Measured (profiles/r02_tuning.md, scripts/ws_trace_summary.py on a -DDMT_WS_TRACE build): one CTA walks a block at ~1,900 cycles per
// tile whatever the ensemble size, and at 16 warps x 128 registers only one CTA fits an SM, so the pass takes ceil(units / 148) rounds of
// ~0.5 ms (C3's 20-interval blocks): it beats the one-thread-per-(chain, block) kernels up to ~3 rounds (<= 1,400 chains per GPU at 10
// blocks) and loses to them on a full GPU, where they hide the same latencies with 8-10 independent warps per SM.
// Sums of ll / ll° over a chain's 4 step-lanes are taken in a fixed order at the end: results are deterministic and equal to the other
// kernels' up to FP64 rounding (a different summation / FMA contraction order); the random stream is bit-identical.
#pragma once
#include "sweep_kernel.cuh"
#ifdef DMT_WS_TRACE
#include <cstdio>
#endif

namespace dmt {

// 16 warps (P, T, up to 6 R, 4 A, 4 L): 16 warps x 128 registers fill an SM's register file — one CTA per SM.  NR generator warps,
// NSG stages of the G ring, NSR slots of each of the Z, D and X rings.
template <int NR_, int NSG_, int NSR_> struct WsShape {
    static constexpr int NR = NR_, NA = 4, NL = 4, NSG = NSG_, NSZ = NSR_, NSD = NSR_, NSX = NSR_;
    static constexpr int WARPS = 16, THREADS = WARPS * 32;
    static constexpr int NBAR = 2 * (NSG + NSZ + NSD + NSX);
    static_assert(NR >= 1 && NR <= 6, "generator warps: up to 6");
};
constexpr int WS_RS = 36; // row stride of the Z / D / X rings in doubles
// step stride of the transposed guiding term inside a D-ring slot: >= NG rows, and = 4 (mod 16) so that the (chain, step) writers
// (half-warp = 4 chains x 4 steps) hit 16 different bank pairs
__host__ __device__ constexpr int ws_gt_stride(int NG) { int v = NG * WS_RS; while (v % 16 != 4) v += 4; return v; }
// Warp -> role.  Warp w issues on scheduler w % 4.  The recursion warp P shares its scheduler only with the lightest warps (the TMA
// lane and two L warps); the generator warps, which saturate the FP64 pipe of their scheduler, are spread over the other three.
enum { WS_P = 0, WS_T = 1, WS_R = 2, WS_A = 3, WS_L = 4 };
__device__ __forceinline__ void ws_role_of(int warp, int &role, int &id) {
    // w:      15 14 13 12 11 10  9  8  7  6  5  4  3  2  1  0      (one hex digit per warp; no table in local memory)
    // role:    A  L  L  L  A  A  A  L  R  R  R  T  R  R  R  P
    // id:      3  3  2  1  2  1  0  0  5  4  3  0  2  1  0  0
    role = (int)((0x3444333422212220ull >> (4 * warp)) & 0xfull);
    id = (int)((0x3321210054302100ull >> (4 * warp)) & 0xfull);
}

template <class MD, class SH> constexpr size_t sweep_ws_smem() {
    constexpr int D = MD::D, DW = MD::DW, NG = D * (D + 1) / 2 + D;
    return (size_t)SH::NSG * (NG * 128 + 8) * 8 + (size_t)SH::NSZ * (4 * DW) * WS_RS * 8 +
           (size_t)SH::NSD * ((4 * DW) * WS_RS + 4 * ws_gt_stride(NG)) * 8 + (size_t)SH::NSX * 5 * D * WS_RS * 8 + (size_t)3 * 32 * 8 + SH::NBAR * 8 +
           (size_t)(D * D + D) * 32 * 8;
}

__device__ __forceinline__ void mbar_arrive(uint64_t *b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory"); }

#ifdef DMT_WS_TRACE // (debug build: per-role time stamps of some tiles of CTA (0,0), printed at the end)
#define WS_TR_DECL long long tr_[48][3]; const bool tr_on = blockIdx.x == 0 && blockIdx.y == 0 && lane == 0;
#define WS_TR(j, i) if (tr_on && (j) >= 100 && (j) < 148) tr_[(j) - 100][i] = clock64();
#define WS_TR_DUMP(name) if (tr_on) for (int j_ = 0; j_ < 48 && j_ + 100 < T; j_++) printf("TR %s %d %d %lld %lld %lld\n", name, warp, j_ + 100, tr_[j_][0], tr_[j_][1], tr_[j_][2]);
#else
#define WS_TR_DECL
#define WS_TR(j, i)
#define WS_TR_DUMP(name)
#endif
struct WsCursor { // (interval, tile inside it) of a tile of the block
    int k, q, ntl, t0;
};

template <class MD, bool LAZYW, class SH>
__global__ void __launch_bounds__(SH::THREADS, 1) sweep_ws_kernel(const DevCtx cx, const LayoutDev ly, const FwdArgs fa) {
    constexpr int NR = SH::NR, NA = SH::NA, NL = SH::NL, NSG = SH::NSG, NSZ = SH::NSZ, NSD = SH::NSD, NSX = SH::NSX, RS = WS_RS;
    constexpr int D = MD::D, DW = MD::DW, NPAR = MD::NPAR, NH = D * (D + 1) / 2, NG = NH + D, NAUX = D * D + D + NH;
    constexpr int STAGE = NG * 128 + 8, NZ = 4 * DW, ZS = NZ * RS, XS = 5 * D * RS, SS = ws_gt_stride(NG), DS = ZS + 4 * SS;
    extern __shared__ __align__(128) unsigned char ws_smem[];
    double *gring = reinterpret_cast<double *>(ws_smem);          // [NSG][STAGE]
    double *zring = gring + (size_t)NSG * STAGE;                   // [NSZ][4][DW][RS]  standard normals, row n = step * DW + coordinate
    double *dring = zring + (size_t)NSZ * ZS;                      // [NSD] { [4][DW][RS] refreshed noise dW° ; [4][SS] H, F per step, row = component }
    double *xring = dring + (size_t)NSD * DS;                      // [NSX][D][5][RS]   x° before step 0 and after steps 0..3
    double *part = xring + (size_t)NSX * XS;                       // [3][32]           ll, ll°, success per chain
    uint64_t *bars = reinterpret_cast<uint64_t *>(part + 3 * 32);
    uint64_t *full_g = bars, *empty_g = full_g + NSG, *full_z = empty_g + NSG, *empty_z = full_z + NSZ;
    uint64_t *full_d = empty_z + NSZ, *empty_d = full_d + NSD, *full_x = empty_d + NSD, *empty_x = full_x + NSX;
    double *alaw = reinterpret_cast<double *>(empty_x + NSX);    // [D*D + D][32]: B, beta of the A warps' chains for the current interval

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int role, w_id;
    ws_role_of(warp, role, w_id);
    const int c0 = blockIdx.x * 32, b = blockIdx.y;
    if (c0 >= cx.M) return;
    const size_t M = cx.M, P = cx.P;
    const int i0 = ly.i0[b], i1 = ly.i1[b];
    const bool last = ly.last[b] != 0;
    const uint32_t chunk_bytes = 32u * (uint32_t)min(32, cx.M - c0);
    const size_t gstr = P * 4;

    if (threadIdx.x == 0) { // every warp of a role visits every tile, so each barrier simply counts the role's warps
        for (int s = 0; s < NSG; s++) { mbar_init(&full_g[s], 1); mbar_init(&empty_g[s], NA + NL); }
        for (int s = 0; s < NSZ; s++) { mbar_init(&full_z[s], NR); mbar_init(&empty_z[s], NA); }
        for (int s = 0; s < NSD; s++) { mbar_init(&full_d[s], NA); mbar_init(&empty_d[s], 1); }
        for (int s = 0; s < NSX; s++) { mbar_init(&full_x[s], 1); mbar_init(&empty_x[s], NL); }
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    int T = 0; // tiles of this block
    for (int k = i0; k <= i1; k++) T += (cx.nsteps[k] + 3) >> 2;

    auto cur_init = [&]() { WsCursor u; u.k = i0; u.q = 0; u.ntl = (cx.nsteps[i0] + 3) >> 2; u.t0 = cx.tile0[i0]; return u; };
    auto cur_next = [&](WsCursor &u) {
        if (++u.q == u.ntl) {
            u.q = 0;
            if (++u.k <= i1) { u.ntl = (cx.nsteps[u.k] + 3) >> 2; u.t0 = cx.tile0[u.k]; }
        }
    };
    // ring protocol: the producers of item j wait until the slot's previous occupant (item j - N) has been released, the consumers until
    // item j has landed.  (mbarrier waits name a phase by its PARITY: legal because every waiter visits every item of its ring in order.)
    auto wait_full = [&](uint64_t *bar, int j, int N) { mbar_wait(&bar[j % N], (uint32_t)(j / N) & 1u); };
    auto wait_empty = [&](uint64_t *bar, int j, int N) { if (j >= N) mbar_wait(&bar[j % N], (uint32_t)(j / N - 1) & 1u); };
    auto signal = [&](uint64_t *bar, int j, int N) { __syncwarp(); if (lane == 0) mbar_arrive(&bar[j % N]); };
    auto law_of = [&](int k, int ps, int &slot, int &store) {
        store = (k == i1 && !last) ? 1 : 0;
        slot = cx.parP[store][(size_t)k * P + ps];
    };

    if (role == WS_P) {
        // ================================================================== P: the proposal's recursion, one lane per chain
        const int c = min(c0 + lane, cx.M - 1); // lanes beyond the ensemble shadow the last chain and never store
        const bool live = c0 + lane < cx.M;
        const int ps = c;                       // launch condition: one parameter set per chain, in chain order
        WsCursor u = cur_init();
        double xo[D];
        {
            const int sl = cx.parX[(size_t)i0 * M + c];
#pragma unroll
            for (int i = 0; i < D; i++) xo[i] = cx.X0[sl * cx.X0buf + ((size_t)i0 * D + i) * M + c];
        }
        double thn[NPAR];
        uint8_t px = 0, pw = 0, pxn = 0, pwn = 0;
        auto fetch = [&](int k, double *t, uint8_t &x_, uint8_t &w_) { // theta and buffer parities of interval k
            int slot, store;
            law_of(k, ps, slot, store);
            const double *tp = cx.theta[slot][store] + (size_t)k * NPAR * P + ps;
#pragma unroll
            for (int i = 0; i < NPAR; i++) t[i] = tp[(size_t)i * P];
            x_ = cx.parX[(size_t)k * M + c];
            w_ = cx.parW[(size_t)k * M + c];
        };
        fetch(i0, thn, pxn, pwn);
        typename MD::Par par(thn);
        int k_loaded = -1, nst = 0;
        WS_TR_DECL
        for (int j = 0; j < T; j++) {
            WS_TR(j, 0)
            if (u.k != k_loaded) { // a new interval: its record was fetched one interval ago
                par = typename MD::Par(thn);
                px = pxn; pw = pwn;
                if (u.k < i1) fetch(u.k + 1, thn, pxn, pwn);
                nst = cx.nsteps[u.k];
                if (live) { // XX°[k].x[1] = the proposal's current state
                    double *x0p = cx.X0 + (size_t)(1 ^ px) * cx.X0buf + (size_t)u.k * D * M + c;
#pragma unroll
                    for (int i = 0; i < D; i++) x0p[(size_t)i * M] = xo[i];
                }
                k_loaded = u.k;
            }
            wait_empty(empty_x, j, NSX);
            double *xs = xring + (size_t)(j % NSX) * XS + lane;
#pragma unroll
            for (int a = 0; a < D; a++) xs[(a * 5) * RS] = xo[a];
            wait_full(full_d, j, NSD);
            const double *dwi = dring + (size_t)(j % NSD) * DS + lane; // dW°, then the guiding term transposed by A (conflict-free here)
            const double *gt = dwi + ZS;
            const double *dtp = cx.dt + (size_t)(u.t0 + u.q) * 4;
            WS_TR(j, 1)
            double wo[LAZYW ? 1 : DW][4];
            auto step = [&](auto s_c) {
                constexpr int s = decltype(s_c)::value;
                double Hs[NH], F[D], dwo[DW], swo[D], gdo[D], Gd = 0.0;
#pragma unroll
                for (int a = 0; a < NH; a++) Hs[a] = gt[s * SS + a * RS];
#pragma unroll
                for (int a = 0; a < D; a++) F[a] = gt[s * SS + (NH + a) * RS];
                const double dt = __ldg(dtp + s);
#pragma unroll
                for (int jj = 0; jj < DW; jj++) {
                    dwo[jj] = dwi[(s * DW + jj) * RS];
                    if (!LAZYW) wo[jj][s] = dwo[jj];
                }
                const typename MD::Diff dfo(par, xo);
                guided_terms<MD, false>(par, dfo, nullptr, nullptr, nullptr, Hs, F, xo, gdo, Gd);
                dfo.sig_mul(dwo, swo);
#pragma unroll
                for (int a = 0; a < D; a++) {
                    xo[a] = fma(gdo[a], dt, xo[a]) + swo[a];
                    xs[(a * 5 + 1 + s) * RS] = xo[a];
                }
            };
            if (4 * u.q + 4 <= nst) { // a full tile (always, on grids whose intervals hold a multiple of 4 steps): one basic block, loads hoisted
                static_for<4>([&](auto s_c) { step(s_c); });
            } else {
                static_for<4>([&](auto s_c) {
                    constexpr int s = decltype(s_c)::value;
                    if (4 * u.q + s < nst) step(s_c);
                    else {
#pragma unroll
                        for (int a = 0; a < D; a++) xs[(a * 5 + 1 + s) * RS] = xo[a];
                        if (!LAZYW) {
#pragma unroll
                            for (int jj = 0; jj < DW; jj++) wo[jj][s] = 0.0;
                        }
                    }
                });
            }
            // the tile of X° for the store, read back from the ring (this lane's own words) before the slot is handed to L; steps past the
            // end of the interval are stored as zeros like everywhere else
            double xot[D][4];
#pragma unroll
            for (int a = 0; a < D; a++)
#pragma unroll
                for (int s = 0; s < 4; s++) xot[a][s] = (4 * u.q + s < nst) ? xs[(a * 5 + 1 + s) * RS] : 0.0;
            signal(full_x, j, NSX);
            signal(empty_d, j, NSD);
            WS_TR(j, 2)
            if (live) {
                if (!LAZYW) {
                    double *Wprop = cx.W + (size_t)(1 ^ pw) * cx.Wbuf + ((size_t)u.t0 * DW * M + c) * 4;
#pragma unroll
                    for (int jj = 0; jj < DW; jj++) st256(Wprop + ((size_t)u.q * DW + jj) * M * 4, wo[jj]);
                }
                double *Xout = cx.X + (size_t)(1 ^ px) * cx.Xbuf + ((size_t)u.t0 * D * M + c) * 4;
#pragma unroll
                for (int i = 0; i < D; i++) st256(Xout + ((size_t)u.q * D + i) * M * 4, xot[i]);
            }
            cur_next(u);
        }
        WS_TR_DUMP("P")
    } else if (role == WS_T) {
        // ================================================================== T: TMA producer of the G ring
        if (lane == 0) {
            WsCursor u = cur_init();
            const double *gp = g_tile_of<NG>(cx, ly, i0, i1, last, 0, c0).base;
            int k_cur = i0;
            for (int j = 0; j < T; j++) {
                if (u.k != k_cur) { gp = g_tile_of<NG>(cx, ly, u.k, i1, last, 0, c0).base; k_cur = u.k; }
                wait_empty(empty_g, j, NSG);
                uint64_t *bar = &full_g[j % NSG];
                double *dst = gring + (size_t)(j % NSG) * STAGE;
                mbar_expect_tx(bar, NG * chunk_bytes + 64u);
#pragma unroll 1
                for (int a = 0; a < NG; a++) bulk_g2s(dst + a * 128, gp + ((size_t)u.q * NG + a) * gstr, chunk_bytes, bar);
                bulk_g2s(dst + NG * 128, cx.dt + (size_t)(u.t0 + u.q) * 4, 32u, bar);
                bulk_g2s(dst + NG * 128 + 4, cx.sqdt + (size_t)(u.t0 + u.q) * 4, 32u, bar);
                cur_next(u);
            }
        }
    } else if (role == WS_R) {
        // ================================================================== R: the tile's normals, one lane per chain
        const int r = w_id;
        if (r < NR) {
        const int c = min(c0 + lane, cx.M - 1);
        WsCursor u = cur_init();
        WS_TR_DECL
        for (int j = 0; j < T; j++) {
            WS_TR(j, 0)
            wait_empty(empty_z, j, NSZ);
            WS_TR(j, 1)
            double *zo = zring + (size_t)(j % NSZ) * ZS + lane;
#pragma unroll 1
            for (int call = r; call < 2 * DW; call += NR) {
                u32x4 ctr = {cx.chain_offset + (uint32_t)c, (uint32_t)(u.t0 + u.q), fa.iter, ctr_word3(STREAM_PCN, (uint32_t)ly.id, (uint32_t)call)};
                double z0, z1;
                box_muller(philox4x32_10(ctr, (uint32_t)cx.seed, (uint32_t)(cx.seed >> 32)), z0, z1);
                zo[(2 * call) * RS] = z0;
                zo[(2 * call + 1) * RS] = z1;
            }
            signal(full_z, j, NSZ);
            WS_TR(j, 2)
            cur_next(u);
        }
        WS_TR_DUMP("R")
        }
    } else {
        // ================================================================== A and L: one lane per (chain, step), 8 chains per warp
        const bool is_A = role == WS_A;
        const int s = lane & 3;                      // this lane's step inside every tile
        const int cl = 8 * w_id + (lane >> 2);       // chain slot inside the CTA's group of 32
        const int c = min(c0 + cl, cx.M - 1);
        const bool live = c0 + cl < cx.M;
        WsCursor u = cur_init();
        // the law record of interval k for this lane's chain; the next interval's record goes into L2 now, so that the switch costs L2
        // hits instead of DRAM round trips
        double th[NPAR], Bm[D * D], beta[D], at[NH];
        auto load_law = [&](int k) {
            int slot, store;
            law_of(k, c, slot, store);
            const double *tp = cx.theta[slot][store] + (size_t)k * NPAR * P + c;
#pragma unroll
            for (int i = 0; i < NPAR; i++) th[i] = tp[(size_t)i * P];
            const double *ap = cx.aux[slot][store] + (size_t)k * NAUX * P + c;
#pragma unroll
            for (int i = 0; i < D * D; i++) Bm[i] = ap[(size_t)i * P];
#pragma unroll
            for (int i = 0; i < D; i++) beta[i] = ap[(size_t)(D * D + i) * P];
            if (!MD::CONSTDIFF) {
#pragma unroll
                for (int i = 0; i < NH; i++) at[i] = ap[(size_t)(D * D + D + i) * P];
            }
            if (k < i1 && s == 0) {
                int slot1, store1;
                law_of(k + 1, c, slot1, store1);
                const double *tp1 = cx.theta[slot1][store1] + (size_t)(k + 1) * NPAR * P + c;
                const double *ap1 = cx.aux[slot1][store1] + (size_t)(k + 1) * NAUX * P + c;
#pragma unroll
                for (int i = 0; i < NPAR; i++) prefetch_l2(tp1 + (size_t)i * P);
#pragma unroll
                for (int i = 0; i < (MD::CONSTDIFF ? D * D + D : NAUX); i++) prefetch_l2(ap1 + (size_t)i * P);
                if (is_A) {
#pragma unroll
                    for (int i = 0; i < D; i++) {
                        prefetch_l2(cx.X0 + ((size_t)(k + 1) * D + i) * M + c);
                        prefetch_l2(cx.X0 + cx.X0buf + ((size_t)(k + 1) * D + i) * M + c);
                    }
                }
            }
        };
        // loglikhd_obs(PP[1], y1) = -c - y'Hy/2 + F'y at the block's first point (src/block.jl:178)
        auto start_term = [&](const double *Hs, const double *F, const double *y) {
            const GTile<NG> gt = g_tile_of<NG>(cx, ly, i0, i1, last, 0, c);
            double s0 = -*gt.c0;
#pragma unroll
            for (int i = 0; i < D; i++) {
                double hx = 0.0;
#pragma unroll
                for (int jj = 0; jj < D; jj++) hx = fma(Hs[sidx<D>(i, jj)], y[jj], hx);
                s0 += y[i] * (F[i] - 0.5 * hx);
            }
            return s0;
        };
        load_law(i0);
        typename MD::Par par(th);
        int k_loaded = i0, nst = cx.nsteps[i0];
        double acc = 0.0; // this lane's share of ll (A) / ll° (L)
        if (is_A) {
            // ---------------------------------------------------------------- A: K5, the accepted path's likelihood, the pCN refresh
            const double rho = layout_rho(ly, b, c, M), crho = sqrt(1.0 - rho * rho);
            // X two tiles ahead in registers: the tile's value at this lane's step
            WsCursor xc = cur_init();
            int jx = 0;
            double xa[D], x1[D], carry[D];
            // (the buffer parity of the prefetch cursor's interval is kept in a register and the NEXT interval's is fetched when an interval
            // is entered: a warp issues in order, so a parity load in front of every tile's X loads would stall it for an L2 round trip)
            int kx = i0;
            uint8_t pxx = cx.parX[(size_t)i0 * M + c], pxx_next = i0 < i1 ? cx.parX[(size_t)(i0 + 1) * M + c] : 0;
            auto load_x = [&](double (&xv)[D]) {
                if (jx >= T) return;
                if (xc.k != kx) {
                    kx = xc.k;
                    pxx = pxx_next;
                    if (kx < i1) pxx_next = cx.parX[(size_t)(kx + 1) * M + c];
                }
                const uint8_t px = pxx;
                const double *xin = cx.X + (size_t)px * cx.Xbuf + (((size_t)xc.t0 + xc.q) * D * M + c) * 4 + s;
#pragma unroll
                for (int i = 0; i < D; i++) xv[i] = __ldg(xin + (size_t)i * M * 4);
                jx++;
                cur_next(xc);
            };
#pragma unroll
            for (int i = 0; i < D; i++) carry[i] = 0.0;
            load_x(xa); load_x(x1);
            uint8_t pw = cx.parW[(size_t)i0 * M + c];
            // B and beta live in shared memory (one column per chain), not in registers: this warp holds the X prefetch in flight, and a
            // spill reload behind those loads costs a DRAM round trip per tile (same scoreboard; 60 % of this warp's stall samples once)
            auto stash_law = [&]() {
                __syncwarp();
                if (s == 0) {
#pragma unroll
                    for (int i = 0; i < D * D; i++) alaw[i * 32 + cl] = Bm[i];
#pragma unroll
                    for (int i = 0; i < D; i++) alaw[(D * D + i) * 32 + cl] = beta[i];
                }
                __syncwarp();
            };
            stash_law();
            WS_TR_DECL
            for (int j = 0; j < T; j++) {
                WS_TR(j, 0)
                if (u.k != k_loaded) {
                    load_law(u.k);
                    par = typename MD::Par(th);
                    stash_law();
                    pw = cx.parW[(size_t)u.k * M + c];
                    nst = cx.nsteps[u.k];
                    k_loaded = u.k;
                }
                if (u.q == 0) { // the interval's own first point XX[k].x[1] (in L2 since the previous interval's load_law)
                    const uint8_t px = cx.parX[(size_t)u.k * M + c];
#pragma unroll
                    for (int i = 0; i < D; i++) carry[i] = cx.X0[(size_t)px * cx.X0buf + ((size_t)u.k * D + i) * M + c];
                }
                const bool on = 4 * u.q + s < nst;
                wait_full(full_g, j, NSG);
                const double *st = gring + (size_t)(j % NSG) * STAGE;
                const double *sg = st + w_id * 32 + lane; // element (chain slot cl, step s) of every component's chunk
                const double dt = st[NG * 128 + s], sq = st[NG * 128 + 4 + s];
                double Hs[NH], F[D], xb[D], gd[D], G = 0.0, res[D], dwv[DW];
#pragma unroll
                for (int a = 0; a < NH; a++) Hs[a] = sg[a * 128];
#pragma unroll
                for (int a = 0; a < D; a++) F[a] = sg[(NH + a) * 128];
                // the left point of this lane's step: the value one step earlier (one lane down); across tiles the carry; at an interval start
                // the interval's own first point
#pragma unroll
                for (int a = 0; a < D; a++) {
                    const double up = __shfl_up_sync(0xffffffffu, xa[a], 1);
                    xb[a] = s > 0 ? up : carry[a];
                    carry[a] = __shfl_sync(0xffffffffu, xa[a], lane | 3);
                }
                const typename MD::Diff df(par, xb);
                {
                    double Bs[D * D], bs[D];
#pragma unroll
                    for (int i = 0; i < D * D; i++) Bs[i] = alaw[i * 32 + cl];
#pragma unroll
                    for (int i = 0; i < D; i++) bs[i] = alaw[(D * D + i) * 32 + cl];
                    guided_terms<MD, true>(par, df, Bs, bs, at, Hs, F, xb, gd, G);
                }
                if (j == 0 && s == 0) acc = start_term(Hs, F, xb);
                if (on) acc = fma(G, dt, acc);
#pragma unroll
                for (int a = 0; a < D; a++) res[a] = xa[a] - xb[a] - gd[a] * dt; // K5: dW = sigma^+ (x' - x - (b + a r) dt)   (A.5)
                df.inv_sig(res, dwv);
                if (!LAZYW && live) {
                    double *Wacc = cx.W + (size_t)pw * cx.Wbuf + (((size_t)u.t0 + u.q) * DW * M + c) * 4 + s;
#pragma unroll
                    for (int jj = 0; jj < DW; jj++) Wacc[(size_t)jj * M * 4] = on ? dwv[jj] : 0.0;
                }
                // rotate the X prefetch registers and fetch the tile two ahead
#pragma unroll
                for (int a = 0; a < D; a++) xa[a] = x1[a];
                load_x(x1);
                // K3: dW° = rho dW + sqrt(1 - rho^2) sqrt(dt) xi   (A.2)
                WS_TR(j, 1)
                wait_empty(empty_d, j, NSD);
                double *dwo = dring + (size_t)(j % NSD) * DS;
                {   // the guiding term of this (chain, step) for P: row = component, one column per chain, one block per step
                    double *gt = dwo + ZS + s * SS + cl;
#pragma unroll
                    for (int a = 0; a < NH; a++) gt[a * RS] = Hs[a];
#pragma unroll
                    for (int a = 0; a < D; a++) gt[(NH + a) * RS] = F[a];
                }
                wait_full(full_z, j, NSZ);
                const double *zi = zring + (size_t)(j % NSZ) * ZS;
#pragma unroll
                for (int jj = 0; jj < DW; jj++) {
                    const int n = (s * DW + jj) * RS + cl;
                    dwo[n] = on ? rho * dwv[jj] + crho * sq * zi[n] : 0.0;
                }
                signal(full_d, j, NSD);
                signal(empty_z, j, NSZ);
                signal(empty_g, j, NSG);
                WS_TR(j, 2)
                cur_next(u);
            }
            WS_TR_DUMP("A")
        } else {
            // ---------------------------------------------------------------- L: the proposal's likelihood and failure flags
            bool ok = true;
            WS_TR_DECL
            for (int j = 0; j < T; j++) {
                WS_TR(j, 0)
                if (u.k != k_loaded) {
                    load_law(u.k);
                    par = typename MD::Par(th);
                    nst = cx.nsteps[u.k];
                    k_loaded = u.k;
                }
                const bool on = 4 * u.q + s < nst;
                wait_full(full_g, j, NSG); // (landed long ago: P has been through this tile)
                const double *st = gring + (size_t)(j % NSG) * STAGE;
                const double *sg = st + w_id * 32 + lane;
                const double dt = st[NG * 128 + s];
                wait_full(full_x, j, NSX);
                const double *xs = xring + (size_t)(j % NSX) * XS + cl;
                double Hs[NH], F[D], xb[D], xn[D], gdo[D], Go = 0.0;
#pragma unroll
                for (int a = 0; a < NH; a++) Hs[a] = sg[a * 128];
#pragma unroll
                for (int a = 0; a < D; a++) F[a] = sg[(NH + a) * 128];
#pragma unroll
                for (int a = 0; a < D; a++) { xb[a] = xs[(a * 5 + s) * RS]; xn[a] = xs[(a * 5 + s + 1) * RS]; }
                signal(empty_x, j, NSX);
                signal(empty_g, j, NSG);
                WS_TR(j, 1)
                const typename MD::Diff dfo(par, xb);
                guided_terms<MD, true>(par, dfo, Bm, beta, at, Hs, F, xb, gdo, Go);
                if (j == 0 && s == 0) acc = start_term(Hs, F, xb); // the same start term as the accepted path: same law, same start point
                if (on) {
                    acc = fma(Go, dt, acc);
                    bool fin = dfo.ok();
#pragma unroll
                    for (int a = 0; a < D; a++) fin = fin && isfinite(xn[a]);
                    ok = ok && fin && MD::bound_ok(par, xn); // src/block.jl:181 (ll° := -Inf once, after the loop)
                }
                WS_TR(j, 2)
                cur_next(u);
            }
            WS_TR_DUMP("L")
            const unsigned bad = __ballot_sync(0xffffffffu, !ok);
            if (s == 0) part[64 + cl] = ((bad >> (lane & ~3)) & 0xfu) ? 0.0 : 1.0;
        }
        // the chain's sum over its 4 step-lanes, in a fixed order
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
        if (s == 0) part[(is_A ? 0 : 32) + cl] = acc;
    }
    __syncthreads();
    if (warp == 0 && c0 + lane < cx.M) {
        const int c = c0 + lane;
        const bool ok = part[64 + lane] != 0.0;
        ly.ll[(size_t)b * M + c] = part[lane];
        ly.ll[((size_t)ly.nb + b) * M + c] = ok ? part[32 + lane] : -INFINITY;
        ly.ok[(size_t)b * M + c] = ok ? 1 : 0;
    }
}

} // namespace dmt
