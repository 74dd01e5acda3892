// moments_kernel.cuh — posterior summaries of the accepted paths, kept on the device (dmt_path_moments_add / dmt_get_path_moments /
// dmt_get_pset_path_moments).  The tutorials keep a copy of the accepted path every few hundred iterations and look at the mean
// and the spread of the copies (docs/src/tutorials/biblock/smoothing.md:55); here every chain carries running Welford moments of
// its accepted path instead, updated where the paths live.
//
// The accumulators use the X layout exactly (kernels.cuh, DESIGN.md §3), without the accepted / proposal buffer pair:
//   A   [NT][D][M][4]   moment of the state after step 4*tile+s
//   A0  [K ][D][M]      moment of the first point of every interval
// so the update moves whole 32-byte sectors, one lane per sector per component, like cache_apply_kernel.  Padded tile slots
// (n_k - 1 not a multiple of 4) hold whatever the padded X slots hold; they are never returned.
#pragma once
#include "kernels.cuh"

namespace dmt {

// 256-bit load of a sector this kernel also writes: no .nc (the read-only path may not be used for data written by the kernel)
__device__ __forceinline__ void ld256rw(const double *p, double *v) {
    asm volatile("ld.global.L1::no_allocate.L2::evict_first.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]) : "l"(p));
}

// One Welford step, every operation rounded on its own (no FMA contraction), so that a float64 NumPy restatement
//   delta = x - mean; mean' = mean + delta * w; m2' = m2 + delta * (x - mean')
// reproduces it bit for bit.  w = 1 / n is computed on the host in double.
__device__ __forceinline__ void welford(double x, double &mean, double &m2, double w) {
    const double delta = __dsub_rn(x, mean);
    mean = __dadd_rn(mean, __dmul_rn(delta, w));
    m2 = __dadd_rn(m2, __dmul_rn(delta, __dsub_rn(x, mean)));
}

// The whole update in one launch.  Grid (chains / blockDim, rows): rows 0..NT-1 are tiles (D 256-bit sectors per chain), rows
// NT..NT+K-1 the first points of the intervals (D doubles per chain); grid.y strides over the rows if there are more than 65535.
// The accepted buffer of chain c on the interval that owns the row is resolved through parX, as xfer_X_kernel / gather_X_kernel do.
// first == 1 (n == 1): mean := x, m2 := 0 without reading the accumulators (so they need no initialisation).
template <int D>
__global__ void __launch_bounds__(128) path_moments_kernel(const DevCtx cx, double *mean, double *m2, double *mean0, double *m20, double w,
                                                           int first) {
    const size_t M = cx.M;
    const size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= M) return;
    for (int row = blockIdx.y; row < cx.NT + cx.K; row += gridDim.y) {
        if (row < cx.NT) {
            const int t = row, k = cx.k_of_tile[t];
            const double *xp = cx.X + (size_t)cx.parX[(size_t)k * M + c] * cx.Xbuf;
            double x[D][4], mu[D][4], s[D][4];
            // all loads of the row first: the stores below are ordered after them (st256 clobbers memory)
#pragma unroll
            for (int i = 0; i < D; i++) {
                const size_t o = (((size_t)t * D + i) * M + c) * 4;
                ld256(xp + o, x[i]);
                if (!first) { ld256rw(mean + o, mu[i]); ld256rw(m2 + o, s[i]); }
            }
#pragma unroll
            for (int i = 0; i < D; i++) {
                const size_t o = (((size_t)t * D + i) * M + c) * 4;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    if (first) { mu[i][j] = x[i][j]; s[i][j] = 0.0; }
                    else welford(x[i][j], mu[i][j], s[i][j], w);
                }
                st256(mean + o, mu[i]);
                st256(m2 + o, s[i]);
            }
        } else {
            const int k = row - cx.NT;
            const double *xp = cx.X0 + (size_t)cx.parX[(size_t)k * M + c] * cx.X0buf;
#pragma unroll
            for (int i = 0; i < D; i++) {
                const size_t o = ((size_t)k * D + i) * M + c;
                const double x = xp[o];
                double mu = x, s = 0.0;
                if (!first) {
                    mu = mean0[o]; s = m20[o];
                    welford(x, mu, s, w);
                }
                mean0[o] = mu;
                m20[o] = s;
            }
        }
    }
}

// accumulator layout <-> natural [point][dim][n] (the point axis of dmt_get_X).  dir 0: gather the chains sel[0..n) (sel == null:
// chain s for s < n) into nat; dir 1: scatter nat into the accumulators of chains 0..n-1.  Grid (ceil(n / blockDim), K).
__global__ void moments_xfer_kernel(const DevCtx cx, int D, double *A, double *A0, const int *sel, int n, double *nat, int dir) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x, k = blockIdx.y;
    if (s >= n) return;
    const size_t M = cx.M;
    const int c = sel ? sel[s] : s;
    const int nst = cx.nsteps[k], p0 = cx.pt0[k], t0 = cx.tile0[k];
    for (int i = 0; i < D; i++) {
        double *a0 = A0 + ((size_t)k * D + i) * M + c;
        double *np0 = nat + ((size_t)p0 * D + i) * n + s;
        if (dir) *a0 = *np0; else *np0 = *a0;
        for (int j = 0; j < nst; j++) {
            double *ap = A + (((size_t)(t0 + (j >> 2)) * D + i) * M + c) * 4 + (j & 3);
            double *np = nat + ((size_t)(p0 + j + 1) * D + i) * n + s;
            if (dir) *ap = *np; else *np = *ap;
        }
    }
}

// Per-pset pooling of the per-chain moments.  Thread (j, i, q) of block row k: point j of interval k, component i, pset q; output
// [NP][D][P] at point pt0[k] + j.  The chains of q are chains[cs[q] .. cs[q+1]) in ascending order (CSR built on the host).  Every sum
// runs in one fixed order — four interleaved partial sums over the list, combined as (s0 + s1) + (s2 + s3) — so the result is bitwise
// reproducible for a given (M, pset map).  n = number of updates (>= 1), as a double.
__device__ __forceinline__ const double *moment_ptr(const DevCtx &cx, int D, const double *A, const double *A0, int k, int j, int i, int c) {
    const size_t M = cx.M;
    if (j == 0) return A0 + ((size_t)k * D + i) * M + c;
    const int st = j - 1;
    return A + (((size_t)(cx.tile0[k] + (st >> 2)) * D + i) * M + c) * 4 + (st & 3);
}
__global__ void pset_moments_kernel(const DevCtx cx, int D, const double *mean, const double *m2, const double *mean0, const double *m20,
                                    const int *cs, const int *chains, double n, double *out_mean, double *out_var, double *out_rhat) {
    const int k = blockIdx.y;
    const int nk = cx.nsteps[k] + 1;
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x, P = cx.P;
    if (e >= (size_t)nk * D * P) return;
    const int q = (int)(e % P), i = (int)((e / P) % D), j = (int)(e / (P * D));
    const int c0 = cs[q], m = cs[q + 1] - c0;
    const int *ch = chains + c0;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0, b0 = 0.0, b1 = 0.0, b2 = 0.0, b3 = 0.0;
#define MU(r) (*moment_ptr(cx, D, mean, mean0, k, j, i, ch[r]))
#define M2(r) (*moment_ptr(cx, D, m2, m20, k, j, i, ch[r]))
    int r = 0;
    for (; r + 4 <= m; r += 4) { // sums of mu_c and m2_c
        a0 += MU(r); a1 += MU(r + 1); a2 += MU(r + 2); a3 += MU(r + 3);
        b0 += M2(r); b1 += M2(r + 1); b2 += M2(r + 2); b3 += M2(r + 3);
    }
    if (r < m) { a0 += MU(r); b0 += M2(r); }
    if (r + 1 < m) { a1 += MU(r + 1); b1 += M2(r + 1); }
    if (r + 2 < m) { a2 += MU(r + 2); b2 += M2(r + 2); }
    const double mbar = ((a0 + a1) + (a2 + a3)) / m, sm2 = (b0 + b1) + (b2 + b3);
    a0 = a1 = a2 = a3 = 0.0;
    for (r = 0; r + 4 <= m; r += 4) { // sum of (mu_c - mbar)^2
        const double d0 = MU(r) - mbar, d1 = MU(r + 1) - mbar, d2 = MU(r + 2) - mbar, d3 = MU(r + 3) - mbar;
        a0 += d0 * d0; a1 += d1 * d1; a2 += d2 * d2; a3 += d3 * d3;
    }
    if (r < m) { const double dv = MU(r) - mbar; a0 += dv * dv; }
    if (r + 1 < m) { const double dv = MU(r + 1) - mbar; a1 += dv * dv; }
    if (r + 2 < m) { const double dv = MU(r + 2) - mbar; a2 += dv * dv; }
#undef MU
#undef M2
    const double sdev = (a0 + a1) + (a2 + a3);
    const size_t o = (((size_t)cx.pt0[k] + j) * D + i) * P + q;
    out_mean[o] = mbar;
    out_var[o] = (sm2 / n + sdev) / m; // variance of all n m draws
    // Gelman-Rubin: W within-chain, B between-chain variance; undefined (NaN) for m < 2, n < 2 or W == 0 (e.g. the known start point)
    const double W = sm2 / (m * (n - 1.0)), B = n * sdev / (m - 1);
    const double vplus = ((n - 1.0) / n) * W + B / n;
    out_rhat[o] = (m < 2 || n < 2.0 || W == 0.0) ? __longlong_as_double(0x7ff8000000000000ULL) : sqrt(vplus / W);
}

} // namespace dmt
