// fwd_kernel.cuh — the forward kernel (K2/K3/K4/K5).
//
// Memory discipline (measured with scripts/stream_pattern.cu on B200, profiles/r01_stream_pattern.txt): the
// [tile][component][chain][4] layout streams at 7.0 TB/s when EVERY SECTOR CROSSES L2 EXACTLY ONCE, i.e. one 256-bit
// LDG/STG per lane per sector.  Anything that touches a sector twice at L2 loses: cp.async in 16-byte pieces caps at
// 4.6 TB/s, prefetch.global.L2 followed by the demand load costs a second L2 access (5.3-5.7 vs 6.9 TB/s at equal thread
// count).  So the tile's sectors are loaded straight into registers at the top of the tile, all at once (up to
// d(d+1)/2 + 2d + dw independent 256-bit loads in flight per lane), and the refreshed noise is streamed out before the
// recursion starts so the stores overlap the arithmetic.
#pragma once
#include "kernels.cuh"

namespace dmt {

// ---- TMA bulk copy + mbarrier (sm_90+): the warp-contiguous 1 KiB chunk of one component of one tile, global -> shared
// (sweep_kernel.cuh, sweep_ws_kernel.cuh)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *b, int cnt) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(cnt)); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *b) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
                 "r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *b, uint32_t parity) {
    asm volatile("{\n.reg .pred p;\nWAIT_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}" ::"r"(smem_u32(b)),
                 "r"(parity) : "memory");
}

template <int NG> struct GTile { // where the guiding term of interval k lives for this thread's pset / law side
    const double *base;          // tile 0, component 0, this pset
    const double *c0;            // c at the interval start, this pset
    int store, slot, gt0;        // gt0: first tile of the interval in its store
};
template <int NG>
__device__ __forceinline__ GTile<NG> g_tile_of(const DevCtx &cx, const LayoutDev &ly, int k, int i1, bool last, int law_side, int ps) {
    GTile<NG> t;
    t.store = (k == i1 && !last) ? 1 : 0; // P_last comes from PPb (src/block.jl:68)
    t.slot = law_side ^ cx.parP[t.store][(size_t)k * cx.P + ps];
    const int gt0 = t.store ? cx.ppb_tile0[k] : cx.tile0[k];
    t.gt0 = gt0;
    const bool priv = (law_side == 0) && (ly.Gl[t.store] != nullptr); // layout-private (cached) accepted-law guiding term
    t.base = (priv ? ly.Gl[t.store] : cx.G[t.slot][t.store]) + ((size_t)gt0 * NG * cx.P + ps) * 4;
    t.c0 = (priv ? ly.c0l[t.store] : cx.c0[t.slot][t.store]) + (size_t)k * cx.P + ps;
    return t;
}

// Register budget (profiles/r01_tuning.md): with <= 45k (chain, block) threads per GPU the kernel is latency bound, and having
// EVERY CTA resident in one wave matters more than avoiding spills: d <= 3 models are capped at 168 registers
// (6 CTAs of 64 threads per SM), the wider ones keep the full budget.
// The cooperative instantiations (G > 1) only run when the GPU is far from full: no cap, no spills.
template <class MD, int G = 1> constexpr int fwd_minb() { return G > 1 ? 1 : (DMT_FWD_MINB > 0 ? DMT_FWD_MINB : (MD::D <= 3 ? 6 : 1)); }
// One thread = one (chain, block).  grid = (ceil(M/TPB), n_blocks).  Replaces, per OP:
//   OP_DRAW        draw_proposal_path!(bb)            src/biblock.jl:80-106   (pCN + guided EM + ll, fused; K3+K2+K4)
//   OP_RECOMPUTE   recompute_path!(b°, b.WW; skip)    src/block.jl:161-187    (K2+K4)
//   OP_LOGLIK      loglikhd!(b)                       src/block.jl:140-152    (K4)
//   OP_INVSOLVE    find_W_for_X!(b)                   src/block.jl:120-131    (K5)
//   OP_INVSOLVE_LL both of the above in one pass over X
//   OP_INIT        init_paths! / draw_proposal_path!(u::SamplingUnit)  src/sampling_unit.jl:83-87,118-120 (fresh noise, in place)
//   OP_SWEEP       find_W_for_X!(b); loglikhd!(b); draw_proposal_path!(bb) of the blocking sweep
//                  (docs/src/tutorials/block_collection/inference_with_blocking.md:55-57) in ONE pass over the tiles: the
//                  accepted noise recovered by K5 feeds the pCN refresh in registers (168 instead of 264 B per step).
//
// G > 1 (ensembles too small to fill the GPU: thread count x G still fits one wave): G adjacent lanes share one
// (chain, block).  The normals of a tile — 2 DW independent Philox + Box-Muller calls, most of the tile's instructions — are
// split over the G lanes and all-gathered with shuffles; everything else is computed redundantly by the G lanes from the same
// loads (one sector request per group, no extra traffic) and lane 0 of the group stores.  The random stream and every
// result are bit-identical to G = 1.
template <class MD, int OP, int TPB, int G = 1>
__global__ void __launch_bounds__(TPB, fwd_minb<MD, G>()) fwd_kernel(const DevCtx cx, const LayoutDev ly, const FwdArgs fa) {
    constexpr int D = MD::D, DW = MD::DW, NPAR = MD::NPAR, NH = D * (D + 1) / 2, NG = NH + D, NAUX = D * D + D + NH;
    constexpr bool SWEEP = (OP == OP_SWEEP);
    constexpr bool READS_X = (OP == OP_LOGLIK || OP == OP_INVSOLVE || OP == OP_INVSOLVE_LL || SWEEP);
    constexpr bool WRITES_X = (OP == OP_DRAW || OP == OP_RECOMPUTE || OP == OP_INIT);
    constexpr bool READS_W = (OP == OP_DRAW || OP == OP_RECOMPUTE);
    constexpr bool WRITES_W = (OP == OP_DRAW || OP == OP_INIT || OP == OP_INVSOLVE || OP == OP_INVSOLVE_LL || SWEEP);
    constexpr bool INV = (OP == OP_INVSOLVE || OP == OP_INVSOLVE_LL || SWEEP);
    constexpr bool WANT_LL = (OP != OP_INVSOLVE);
    constexpr bool RNG = (OP == OP_DRAW || OP == OP_INIT || SWEEP);

    static_assert(G == 1 || G == 2 || G == 4 || G == 8, "lanes per chain");
    constexpr bool UNI = G > 1;                        // warp-uniform control flow: lanes idle instead of leaving
    const int t_raw = blockIdx.x * TPB + threadIdx.x;
    const int c_raw = t_raw / G, sub = t_raw % G;
    const int b = blockIdx.y;
    if (!UNI && c_raw >= cx.M) return;
    if (UNI && ((t_raw & ~31) / G) >= cx.M) return;    // the whole warp lies beyond the ensemble (uniform exit)
    const int c = UNI ? min(c_raw, cx.M - 1) : c_raw;  // lanes without a chain shadow the last one and never store
    const size_t M = cx.M, P = cx.P;
    bool live = c_raw < cx.M && sub == 0;
    if (OP == OP_INIT && ly.ok[(size_t)b * M + c]) { // retry only the chains that failed so far
        if (!UNI) return;
        live = false;
    }
    const int ps = cx.pset[c];
    const int i0 = ly.i0[b], i1 = ly.i1[b];
    const bool last = ly.last[b] != 0;

    const int law_side = (OP == OP_RECOMPUTE || OP == OP_LOGLIK) ? fa.law_side : 0;
    const int xin_side = law_side;
    const int xout_side = (OP == OP_DRAW || SWEEP) ? 1 : law_side;
    const int win_side = (OP == OP_RECOMPUTE) ? fa.w_side : 0;
    const int wout_side = (OP == OP_DRAW) ? 1 : 0; // SWEEP writes both: accepted in place, proposal to the other buffer
    const int ll_side = (OP == OP_DRAW) ? 1 : law_side;
    const double rho = (OP == OP_DRAW || SWEEP) ? layout_rho(ly, b, c, M) : 0.0;
    const double crho = (OP == OP_DRAW || SWEEP) ? sqrt(1.0 - rho * rho) : 1.0;
    const int skip = fa.skip;
    const size_t gstr = P * 4; // doubles between components of one tile

    double x[D], xo[SWEEP ? D : 1]; // x: the path that is read or written; xo (SWEEP): the proposal path
    {   // y1 = XX[1].x[1] of the block  (src/biblock.jl:96, src/block.jl:177)
        const int sl = xin_side ^ cx.parX[(size_t)i0 * M + c];
#pragma unroll
        for (int i = 0; i < D; i++) x[i] = cx.X0[sl * cx.X0buf + ((size_t)i0 * D + i) * M + c];
        if (SWEEP) {
#pragma unroll
            for (int i = 0; i < D; i++) xo[i] = x[i];
        }
    }
    double ll = 0.0, llo = 0.0;
    bool ok = true;

    for (int k = i0; k <= i1 && (ok || SWEEP || UNI); ++k) {
        const GTile<NG> gt = g_tile_of<NG>(cx, ly, k, i1, last, law_side, ps);
        const int store = gt.store, slotL = gt.slot;
        const double *Gp = gt.base;
        double th[NPAR];
        {
            const double *tp = cx.theta[slotL][store] + (size_t)k * NPAR * P + ps;
#pragma unroll
            for (int i = 0; i < NPAR; i++) th[i] = tp[(size_t)i * P];
        }
        const typename MD::Par par(th);
        double Bm[D * D], beta[D], at[NH];
        if (WANT_LL) {
            const double *ap = cx.aux[slotL][store] + (size_t)k * NAUX * P + ps;
#pragma unroll
            for (int i = 0; i < D * D; i++) Bm[i] = ap[(size_t)i * P];
#pragma unroll
            for (int i = 0; i < D; i++) beta[i] = ap[(size_t)(D * D + i) * P];
            if (!MD::CONSTDIFF) {
#pragma unroll
                for (int i = 0; i < NH; i++) at[i] = ap[(size_t)(D * D + D + i) * P];
            }
        }
        const int nst = cx.nsteps[k];
        const int t0 = cx.tile0[k];
        const uint8_t pw = cx.parW[(size_t)k * M + c], px = cx.parX[(size_t)k * M + c];
        const double *Win = cx.W + (size_t)(win_side ^ pw) * cx.Wbuf + ((size_t)t0 * DW * M + c) * 4;
        double *Wout = cx.W + (size_t)(wout_side ^ pw) * cx.Wbuf + ((size_t)t0 * DW * M + c) * 4;
        double *Wprop = cx.W + (size_t)(1 ^ pw) * cx.Wbuf + ((size_t)t0 * DW * M + c) * 4; // SWEEP only
        const double *Xin = cx.X + (size_t)(xin_side ^ px) * cx.Xbuf + ((size_t)t0 * D * M + c) * 4;
        double *Xout = cx.X + (size_t)(xout_side ^ px) * cx.Xbuf + ((size_t)t0 * D * M + c) * 4;
        if (READS_X && k > i0) { // an existing path: interval k starts at ITS OWN XX[k].x[1]
#pragma unroll
            for (int i = 0; i < D; i++) x[i] = cx.X0[(size_t)(xin_side ^ px) * cx.X0buf + ((size_t)k * D + i) * M + c];
        }
        if ((WRITES_X || SWEEP) && live) { // XX°[k].x[1] = y1
            double *x0p = cx.X0 + (size_t)(xout_side ^ px) * cx.X0buf + (size_t)k * D * M + c;
#pragma unroll
            for (int i = 0; i < D; i++) x0p[(size_t)i * M] = SWEEP ? xo[i] : x[i];
        }

        const int ntl = (nst + 3) >> 2;
        for (int q = 0; q < ntl; ++q) {
            double g[NG][4], w[DW][4], xt[D][4], dt4[4], sq4[4];
            double wo[SWEEP ? DW : 1][4], xot[SWEEP ? D : 1][4], z[RNG ? 4 * DW : 1];
            // ---- every sector of the tile, once, straight into registers
            if (READS_W) {
#pragma unroll
                for (int j = 0; j < DW; j++) ld256(Win + ((size_t)q * DW + j) * M * 4, w[j]);
            }
#pragma unroll
            for (int a = 0; a < NG; a++) ld256(Gp + ((size_t)q * NG + a) * gstr, g[a]);
            if (READS_X) {
#pragma unroll
                for (int i = 0; i < D; i++) ld256(Xin + ((size_t)q * D + i) * M * 4, xt[i]);
            }
            ld256u(cx.dt + (size_t)(t0 + q) * 4, dt4);
            if (RNG) ld256u(cx.sqdt + (size_t)(t0 + q) * 4, sq4);

            if (RNG) { // xi ~ N(0, I): independent of everything loaded above, runs while the sectors are in flight
                if (fa.Z) {
#pragma unroll
                    for (int s = 0; s < 4; s++)
#pragma unroll
                        for (int j = 0; j < DW; j++) {
                            const int i = 4 * q + s;
                            z[s * DW + j] = (i < nst) ? fa.Z[((size_t)(cx.step0[k] + i) * DW + j) * M + c] : 0.0;
                        }
                } else {
                    if (G > 1) tile_normals_coop<DW, G>(cx.seed, cx.chain_offset + (uint32_t)c, (uint32_t)(t0 + q), fa.iter, (uint32_t)ly.id, sub, z);
                    else tile_normals<DW>(cx.seed, cx.chain_offset + (uint32_t)c, (uint32_t)(t0 + q), fa.iter, (uint32_t)ly.id, z);
                }
                if (!SWEEP) { // K3: dW° = rho dW + sqrt(1-rho^2) sqrt(dt) xi   (A.2)
#pragma unroll
                    for (int s = 0; s < 4; s++)
#pragma unroll
                        for (int j = 0; j < DW; j++) {
                            if (OP == OP_DRAW) w[j][s] = rho * w[j][s] + crho * sq4[s] * z[s * DW + j];
                            else w[j][s] = sq4[s] * z[s * DW + j];
                        }
                    if (live) {
#pragma unroll
                        for (int j = 0; j < DW; j++) st256(Wout + ((size_t)q * DW + j) * M * 4, w[j]); // final: stream out now
                    }
                }
            }

            if (WANT_LL && k == i0 && q == 0) { // loglikhd_obs(PP[1], y1) = -c - y'Hy/2 + F'y  (src/block.jl:178)
                double s0 = -*gt.c0;
#pragma unroll
                for (int i = 0; i < D; i++) {
                    double hx = 0.0;
#pragma unroll
                    for (int j = 0; j < D; j++) hx = fma(g[sidx<D>(i, j)][0], x[j], hx);
                    s0 += x[i] * (g[NH + i][0] - 0.5 * hx);
                }
                ll = s0;
                llo = s0; // same law, same start point
            }
#pragma unroll
            for (int s = 0; s < 4; s++) {
                const int i = 4 * q + s;
                if (i < nst && (ok || SWEEP)) {
                    double Hs[NH], F[D], gd[D], G = 0.0;
#pragma unroll
                    for (int a = 0; a < NH; a++) Hs[a] = g[a][s];
#pragma unroll
                    for (int a = 0; a < D; a++) F[a] = g[NH + a][s];
                    const typename MD::Diff df(par, x);
                    guided_terms<MD, WANT_LL>(par, df, Bm, beta, at, Hs, F, x, gd, G);
                    if (WANT_LL && i < nst - skip) ll = fma(G, dt4[s], ll);
                    double xn[D];
                    if (WRITES_X) { // K2: x' = x + (b + a r) dt + sigma dW   (A.3)
                        double dwv[DW], sw[D];
#pragma unroll
                        for (int j = 0; j < DW; j++) dwv[j] = w[j][s];
                        df.sig_mul(dwv, sw);
#pragma unroll
                        for (int a = 0; a < D; a++) xn[a] = fma(gd[a], dt4[s], x[a]) + sw[a];
                        bool fin = df.ok();
#pragma unroll
                        for (int a = 0; a < D; a++) fin = fin && isfinite(xn[a]);
                        if (!(fin && MD::bound_ok(par, xn))) { ok = false; ll = -INFINITY; } // src/block.jl:181
#pragma unroll
                        for (int a = 0; a < D; a++) xt[a][s] = xn[a];
                    } else {
#pragma unroll
                        for (int a = 0; a < D; a++) xn[a] = xt[a][s];
                        if (INV) { // K5: dW = sigma^+ (x' - x - (b + a r) dt)   (A.5)
                            double res[D], dwv[DW];
#pragma unroll
                            for (int a = 0; a < D; a++) res[a] = xn[a] - x[a] - gd[a] * dt4[s];
                            df.inv_sig(res, dwv);
#pragma unroll
                            for (int j = 0; j < DW; j++) w[j][s] = dwv[j];
                        }
                    }
#pragma unroll
                    for (int a = 0; a < D; a++) x[a] = xn[a];
                    if (SWEEP) { // the proposal: pCN from the noise just recovered, then the guided step from xo
                        double dwo[DW], swo[D], gdo[D], Go = 0.0;
#pragma unroll
                        for (int j = 0; j < DW; j++) { dwo[j] = rho * w[j][s] + crho * sq4[s] * z[s * DW + j]; wo[j][s] = dwo[j]; }
                        if (ok) {
                            const typename MD::Diff dfo(par, xo);
                            guided_terms<MD, true>(par, dfo, Bm, beta, at, Hs, F, xo, gdo, Go);
                            llo = fma(Go, dt4[s], llo);
                            dfo.sig_mul(dwo, swo);
                            double xon[D];
#pragma unroll
                            for (int a = 0; a < D; a++) xon[a] = fma(gdo[a], dt4[s], xo[a]) + swo[a];
                            bool fin = dfo.ok();
#pragma unroll
                            for (int a = 0; a < D; a++) fin = fin && isfinite(xon[a]);
                            if (!(fin && MD::bound_ok(par, xon))) { ok = false; llo = -INFINITY; }
#pragma unroll
                            for (int a = 0; a < D; a++) { xot[a][s] = xon[a]; xo[a] = xon[a]; }
                        } else {
#pragma unroll
                            for (int a = 0; a < D; a++) xot[a][s] = 0.0;
                        }
                    }
                } else {
                    if (WRITES_X) {
#pragma unroll
                        for (int a = 0; a < D; a++) xt[a][s] = 0.0;
                    }
                    if (WRITES_W && !RNG) {
#pragma unroll
                        for (int j = 0; j < DW; j++) w[j][s] = 0.0;
                    }
                    if (SWEEP) {
#pragma unroll
                        for (int j = 0; j < DW; j++) { w[j][s] = 0.0; wo[j][s] = 0.0; }
#pragma unroll
                        for (int a = 0; a < D; a++) xot[a][s] = 0.0;
                    }
                }
            }
            const bool keep_w = !SWEEP || !fa.lazy_w; // lazy noise (dmt_set_lazy_noise): the blocking sweep never reads what it would store here
            if (WRITES_W && (!RNG || SWEEP) && live && keep_w) {
#pragma unroll
                for (int j = 0; j < DW; j++) st256(Wout + ((size_t)q * DW + j) * M * 4, w[j]);
            }
            if (SWEEP && live) {
                if (keep_w) {
#pragma unroll
                    for (int j = 0; j < DW; j++) st256(Wprop + ((size_t)q * DW + j) * M * 4, wo[j]);
                }
#pragma unroll
                for (int i = 0; i < D; i++) st256(Xout + ((size_t)q * D + i) * M * 4, xot[i]);
            }
            if (WRITES_X && live) {
#pragma unroll
                for (int i = 0; i < D; i++) st256(Xout + ((size_t)q * D + i) * M * 4, xt[i]);
            }
            if (!ok && !SWEEP && !UNI) break;
        }
    }
    if (WANT_LL && live) ly.ll[((size_t)ll_side * ly.nb + b) * M + c] = ll;
    if (SWEEP && live) ly.ll[((size_t)ly.nb + b) * M + c] = llo;
    if ((WRITES_X || SWEEP) && live) ly.ok[(size_t)b * M + c] = ok ? 1 : 0;
}

} // namespace dmt
