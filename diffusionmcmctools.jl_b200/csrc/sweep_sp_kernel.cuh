// sweep_sp_kernel.cuh — the blocking sweep's fused forward pass (K5 + K4 + K3 + K2 + K4), STEP-PARALLEL: four lanes per (chain, block).
//
// Same arithmetic and the same reference calls as fwd_kernel<MD, OP_SWEEP> and sweep_pipe_kernel
//   find_W_for_X!(b); loglikhd!(b); draw_proposal_path!(bb)   (/root/reference/docs/src/tutorials/block_collection/inference_with_blocking.md:55-57,
//   /root/reference/src/block.jl:120-152, /root/reference/src/biblock.jl:80-106),
// for ensembles too small to fill the GPU (the 4096-chain ensemble split over 4 or 8 GPUs: 1024 / 512 chains x 10 blocks).  There the
// one-thread-per-(chain, block) kernels are bound by ONE warp's latency per 4-step tile (~4,000 cycles, profiles/r02_tuning.md §4), and of the
// tile's work only the proposal's recursion x°(s) -> x°(s+1) is sequential in time.  So lane s of a 4-lane group owns STEP s of every tile:
//   * its loads are the 8-byte elements [..][chain][s] of the tile's sectors (the group reads whole 32-byte sectors together), double-buffered
//     in registers one tile ahead (14 doubles for Lorenz);
//   * the generator's 2 DW Philox + Box–Muller calls are split over the four lanes (tile_normals_coop, philox.cuh: the same random stream);
//   * inverse solve, accepted-path likelihood and pCN refresh of step s run in lane s, all four steps at once (the accepted path is known);
//   * the proposal's recursion runs as four rounds: every lane evaluates the guided Euler–Maruyama step from the group's current x° with ITS
//     step's H, F, dt, dW°, and the group adopts lane u's result in round u (shuffle broadcast); lane u keeps its left point and evaluates
//     the integrand of ll° after the rounds, in parallel with the other three;
//   * ll and ll° are per-lane partial sums, added in a fixed order at the end of the block (not the serial order: results agree with the other
//     kernels to rounding, not bit for bit — the tests compare at 1e-11).
// A warp holds 8 chains; everything is warp-uniform (lanes beyond the ensemble shadow the last chain and never store).
#pragma once
#include "fwd_kernel.cuh"
#include <type_traits>

namespace dmt {

__device__ __forceinline__ double ld64s(const double *p) { // streaming 8-byte element of a sector that the lane group reads together
    double v;
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double shfl4(double v, int src) { return __shfl_sync(0xffffffffu, v, src, 4); }
// v[s] for a lane-dependent s in 0..3 as two levels of selects (a chain of `s == 0 ? .. : s == 1 ? ..` became three divergent branch
// regions per tile: 8 % of the stall samples, profiles/r02an_summary.md)
__device__ __forceinline__ double sel4(int s, double a, double b, double c, double d) {
    const bool b0 = (s & 1) != 0, b1 = (s & 2) != 0;
    const int lo0 = b0 ? __double2loint(b) : __double2loint(a), hi0 = b0 ? __double2hiint(b) : __double2hiint(a);
    const int lo1 = b0 ? __double2loint(d) : __double2loint(c), hi1 = b0 ? __double2hiint(d) : __double2hiint(c);
    return __hiloint2double(b1 ? hi1 : hi0, b1 ? lo1 : lo0);
}

template <class MD, bool LAZYW>
__global__ void __launch_bounds__(32) sweep_sp_kernel(const DevCtx cx, const LayoutDev ly, const FwdArgs fa) {
    constexpr int D = MD::D, DW = MD::DW, NPAR = MD::NPAR, NH = D * (D + 1) / 2, NG = NH + D, NAUX = D * D + D + NH;
    const int lane = threadIdx.x, s = lane & 3; // s: the step of every tile this lane owns
    const int c_raw = blockIdx.x * 8 + (lane >> 2), b = blockIdx.y;
    const int c = min(c_raw, cx.M - 1);
    const bool live = c_raw < cx.M; // this lane's chain exists (every lane of a live group stores its own step)
    const size_t M = cx.M, P = cx.P;
    const int ps = cx.pset[c];
    const int i0 = ly.i0[b], i1 = ly.i1[b];
    const bool last = ly.last[b] != 0;
    const double rho = layout_rho(ly, b, c, M), crho = sqrt(1.0 - rho * rho); // the four lanes of a chain share it
    const size_t gstr = P * 4;

    // ---- prefetch cursor (the tile after the one being computed) and its register buffer
    int kn = i0, qn = 0, ntl_n = (cx.nsteps[i0] + 3) >> 2, t0_n = cx.tile0[i0];
    const double *gp_n = g_tile_of<NG>(cx, ly, i0, i1, last, 0, ps).base + s;
    const double *xin_n = cx.X + (size_t)cx.parX[(size_t)i0 * M + c] * cx.Xbuf + ((size_t)t0_n * D * M + c) * 4 + s;
    bool more = true;
    double gN[NG], xN[D], dtN = 0.0, sqN = 0.0;
    auto prefetch = [&]() {
        if (!more) return;
#pragma unroll
        for (int a = 0; a < NG; a++) gN[a] = ld64s(gp_n + ((size_t)qn * NG + a) * gstr);
#pragma unroll
        for (int i = 0; i < D; i++) xN[i] = ld64s(xin_n + ((size_t)qn * D + i) * M * 4);
        dtN = __ldg(cx.dt + (size_t)(t0_n + qn) * 4 + s);
        sqN = __ldg(cx.sqdt + (size_t)(t0_n + qn) * 4 + s);
        if (++qn == ntl_n) {
            qn = 0;
            if (++kn <= i1) {
                ntl_n = (cx.nsteps[kn] + 3) >> 2;
                t0_n = cx.tile0[kn];
                gp_n = g_tile_of<NG>(cx, ly, kn, i1, last, 0, ps).base + s;
                xin_n = cx.X + (size_t)cx.parX[(size_t)kn * M + c] * cx.Xbuf + ((size_t)t0_n * D * M + c) * 4 + s;
            } else more = false;
        }
    };
    prefetch();

    double xa[D], xo[D]; // xa: accepted path at the END of the previous tile (the left point of step 0); xo: the proposal, same for the group
    {   // y1 = XX[1].x[1] of the block  (src/biblock.jl:96, src/block.jl:177)
        const int sl = cx.parX[(size_t)i0 * M + c];
#pragma unroll
        for (int i = 0; i < D; i++) { xa[i] = cx.X0[sl * cx.X0buf + ((size_t)i0 * D + i) * M + c]; xo[i] = xa[i]; }
    }
    double ll = 0.0, llo = 0.0; // this lane's partial sums
    bool ok = true;
    {   // loglikhd_obs(PP[1], y1) = -c - y'Hy/2 + F'y  (src/block.jl:178): lane 0 holds H, F at the block's first grid point (the prefetched tile 0)
        double s0 = -*g_tile_of<NG>(cx, ly, i0, i1, last, 0, ps).c0;
#pragma unroll
        for (int i = 0; i < D; i++) {
            double hx = 0.0;
#pragma unroll
            for (int j = 0; j < D; j++) hx = fma(gN[sidx<D>(i, j)], xa[j], hx);
            s0 += xa[i] * (gN[NH + i] - 0.5 * hx);
        }
        ll = s == 0 ? s0 : 0.0;
        llo = ll; // same law, same start point
    }

    for (int k = i0; k <= i1; ++k) {
        const GTile<NG> gt = g_tile_of<NG>(cx, ly, k, i1, last, 0, ps);
        double th[NPAR];
        {
            const double *tp = cx.theta[gt.slot][gt.store] + (size_t)k * NPAR * P + ps;
#pragma unroll
            for (int i = 0; i < NPAR; i++) th[i] = tp[(size_t)i * P];
        }
        const typename MD::Par par(th);
        double Bm[D * D], beta[D], at[NH];
        {
            const double *ap = cx.aux[gt.slot][gt.store] + (size_t)k * NAUX * P + ps;
#pragma unroll
            for (int i = 0; i < D * D; i++) Bm[i] = ap[(size_t)i * P];
#pragma unroll
            for (int i = 0; i < D; i++) beta[i] = ap[(size_t)(D * D + i) * P];
            if (!MD::CONSTDIFF) {
#pragma unroll
                for (int i = 0; i < NH; i++) at[i] = ap[(size_t)(D * D + D + i) * P];
            }
        }
        const int nst = cx.nsteps[k], t0 = cx.tile0[k];
        const uint8_t pw = cx.parW[(size_t)k * M + c], px = cx.parX[(size_t)k * M + c];
        double *Wacc = cx.W + (size_t)pw * cx.Wbuf + ((size_t)t0 * DW * M + c) * 4 + s;
        double *Wprop = cx.W + (size_t)(1 ^ pw) * cx.Wbuf + ((size_t)t0 * DW * M + c) * 4 + s;
        double *Xout = cx.X + (size_t)(1 ^ px) * cx.Xbuf + ((size_t)t0 * D * M + c) * 4 + s;
        if (k > i0) { // an existing path: interval k starts at ITS OWN XX[k].x[1]
#pragma unroll
            for (int i = 0; i < D; i++) xa[i] = cx.X0[(size_t)px * cx.X0buf + ((size_t)k * D + i) * M + c];
        }
        if (live && s == 0) { // XX°[k].x[1] = y1
            double *x0p = cx.X0 + (size_t)(1 ^ px) * cx.X0buf + (size_t)k * D * M + c;
#pragma unroll
            for (int i = 0; i < D; i++) x0p[(size_t)i * M] = xo[i];
        }
        const int ntl = (nst + 3) >> 2;
        for (int q = 0; q < ntl; ++q) {
            double g[NG], xt[D];
#pragma unroll
            for (int a = 0; a < NG; a++) g[a] = gN[a];
#pragma unroll
            for (int i = 0; i < D; i++) xt[i] = xN[i];
            const double dt = dtN, sq = sqN;
            prefetch();

            // ---- the tile's normals: the group's four lanes split the 2 DW generator calls; this lane keeps the DW of its step
            double zs[DW];
            {
                double z[4 * DW];
                tile_normals_coop<DW, 4>(cx.seed, cx.chain_offset + (uint32_t)c, (uint32_t)(t0 + q), fa.iter, (uint32_t)ly.id, s, z);
#pragma unroll
                for (int j = 0; j < DW; j++) zs[j] = sel4(s, z[j], z[DW + j], z[2 * DW + j], z[3 * DW + j]);
            }
            const bool mine = 4 * q + s < nst; // this lane's step exists (false only in the padding of an interval's last tile)
            const double *Hs = g, *F = g + NH;

            // ---- the accepted path's left point of step s: the right point of step s-1 (lane s-1; lane 0: the previous tile's last point)
            double xl[D];
#pragma unroll
            for (int i = 0; i < D; i++) {
                const double up = __shfl_up_sync(0xffffffffu, xt[i], 1, 4);
                xl[i] = s == 0 ? xa[i] : up;
            }
#pragma unroll
            for (int i = 0; i < D; i++) xa[i] = shfl4(xt[i], 3); // (padding steps of a last tile: unused, the next interval reloads xa)

            // ---- K4 on the accepted path, K5, K3 — step s, all four steps of the tile at once
            double dwo[DW];
            {
                double gd[D], G = 0.0, res[D], dwv[DW];
                const typename MD::Diff df(par, xl);
                guided_terms<MD, true>(par, df, Bm, beta, at, Hs, F, xl, gd, G);
                ll = mine ? fma(G, dt, ll) : ll;
#pragma unroll
                for (int a = 0; a < D; a++) res[a] = xt[a] - xl[a] - gd[a] * dt; // K5: dW = sigma^+ (x' - x - (b + a r) dt)   (A.5)
                df.inv_sig(res, dwv);
#pragma unroll
                for (int j = 0; j < DW; j++) { // K3: dW° = rho dW + sqrt(1-rho^2) sqrt(dt) xi   (A.2)
                    const double wj = rho * dwv[j] + crho * sq * zs[j];
                    dwo[j] = mine ? wj : 0.0;
                    dwv[j] = mine ? dwv[j] : 0.0;
                }
                if (!LAZYW && live) {
#pragma unroll
                    for (int j = 0; j < DW; j++) {
                        Wacc[((size_t)q * DW + j) * M * 4] = dwv[j];
                        Wprop[((size_t)q * DW + j) * M * 4] = dwo[j];
                    }
                }
            }

            // ---- K2 on the proposal: four rounds, the group adopts lane u's step in round u (no likelihood integrand in the rounds: the lane
            //      that owns the step keeps the left point and evaluates it afterwards, all four lanes at once)
            double xmine[D], xleft[D];
#pragma unroll
            for (int a = 0; a < D; a++) { xmine[a] = 0.0; xleft[a] = xo[a]; }
            auto rounds = [&](auto full_c) { // FULL (every step of the tile exists): the four rounds form one basic block
                constexpr bool FULL = decltype(full_c)::value;
#pragma unroll
                for (int u = 0; u < 4; u++) {
                if (FULL || 4 * q + u < nst) { // warp-uniform: every chain shares the time grid
                    double gdo[D], Gu = 0.0, swo[D], xon[D];
                    const typename MD::Diff dfo(par, xo);
                    guided_terms<MD, false>(par, dfo, Bm, beta, at, Hs, F, xo, gdo, Gu);
                    dfo.sig_mul(dwo, swo);
#pragma unroll
                    for (int a = 0; a < D; a++) xon[a] = fma(gdo[a], dt, xo[a]) + swo[a];
                    bool fin = dfo.ok();
#pragma unroll
                    for (int a = 0; a < D; a++) fin = fin && isfinite(xon[a]);
                    fin = fin && MD::bound_ok(par, xon); // src/block.jl:181 (ll° := -Inf once, after the loop)
                    const bool own = s == u;             // selects, not a divergent branch
                    ok = own ? (ok && fin) : ok;
#pragma unroll
                    for (int a = 0; a < D; a++) {
                        xmine[a] = own ? xon[a] : xmine[a];
                        xleft[a] = own ? xo[a] : xleft[a];
                    }
#pragma unroll
                    for (int a = 0; a < D; a++) xo[a] = shfl4(xon[a], u);
                }
            }
            };
            if (4 * q + 4 <= nst) rounds(std::true_type{});
            else rounds(std::false_type{});
            {   // K4 on the proposal, step s
                double gdo[D], Go = 0.0;
                const typename MD::Diff dfo(par, xleft);
                guided_terms<MD, true>(par, dfo, Bm, beta, at, Hs, F, xleft, gdo, Go);
                llo = mine ? fma(Go, dt, llo) : llo;
            }
            if (live) {
#pragma unroll
                for (int i = 0; i < D; i++) Xout[((size_t)q * D + i) * M * 4] = xmine[i];
            }
        }
    }
    // ---- the block's ll, ll°, success: the four lanes' partial results in a fixed order
    ll += __shfl_xor_sync(0xffffffffu, ll, 1, 4);
    ll += __shfl_xor_sync(0xffffffffu, ll, 2, 4);
    llo += __shfl_xor_sync(0xffffffffu, llo, 1, 4);
    llo += __shfl_xor_sync(0xffffffffu, llo, 2, 4);
    int oki = ok ? 1 : 0;
    oki &= __shfl_xor_sync(0xffffffffu, oki, 1, 4);
    oki &= __shfl_xor_sync(0xffffffffu, oki, 2, 4);
    if (live && s == 0) {
        ly.ll[(size_t)b * M + c] = ll;
        ly.ll[((size_t)ly.nb + b) * M + c] = oki ? llo : -INFINITY;
        ly.ok[(size_t)b * M + c] = oki ? 1 : 0;
    }
}

} // namespace dmt
