// philox.cuh — counter-based Philox4x32-10 (Salmon, Moraes, Dror, Shaw 2011) and the FP64 normal / exponential
// transforms for the pCN refresh (K3) and the Metropolis test (K6).
// Replaces `Wnr`-driven sampling inside GP.rand! (/root/reference/src/biblock.jl:95-98) and
// rand(Exponential(1.0)) (/root/reference/src/biblock.jl:122).  Counter layout (documented in DESIGN.md §4; the test oracle restates it):
//   pCN   : ctr = (global chain, global tile, iteration, STREAM_PCN<<24 | layout<<8 | call), call = 0 .. 2*DW-1
//   accept: ctr = (global chain, block,       iteration, STREAM_ACC<<24 | layout<<8)
// The LAYOUT ID is part of both counters: the reference loop runs every layout's sweep with the SAME iteration index
// (`for i; for B in blocks; draw_proposal_path!(B); accept_reject_proposal_path!(B, i)`,
// /root/reference/docs/src/tutorials/biblock/smoothing_with_blocking.md:32-59), and the innovations of two sweeps must be independent.
//   key   = (seed lo, seed hi)
// One call -> 128 bits -> two 53-bit uniforms -> one Box–Muller pair.  Z never touches HBM.
#pragma once
#include <stdint.h>
#ifndef DMT_LIBDEVICE_MATH
#define DMT_LIBDEVICE_MATH 0 // 1: libdevice log/sqrt/sincospi (reference for the custom versions in fastmath.cuh)
#endif
#include "fastmath.cuh"

namespace dmt {

constexpr uint32_t STREAM_PCN = 3u, STREAM_ACC = 4u;

struct u32x4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ u32x4 philox4x32_10(u32x4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
#ifdef __CUDA_ARCH__
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
#else
        uint64_t p0 = (uint64_t)0xD2511F53u * c.x, p1 = (uint64_t)0xCD9E8D57u * c.z;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
#endif
        u32x4 n;
        n.x = hi1 ^ c.y ^ k0; n.y = lo1; n.z = hi0 ^ c.w ^ k1; n.w = lo0;
        c = n;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c;
}

// two N(0,1) from one Philox block: u1 in (0,1], u2 in [0,1)
__device__ __forceinline__ void box_muller(u32x4 o, double &z0, double &z1) {
    uint64_t w0 = ((uint64_t)o.y << 32) | o.x, w1 = ((uint64_t)o.w << 32) | o.z;
    double u1 = (double)((w0 >> 11) + 1ull) * 0x1.0p-53;
    double u2 = (double)(w1 >> 11) * 0x1.0p-53;
#if DMT_LIBDEVICE_MATH
    double r = sqrt(-2.0 * log(u1));
    double s, c;
    sincospi(2.0 * u2, &s, &c);
#else
    double r = sqrt_nonneg(-2.0 * log_pos_normal(u1));
    double s, c;
    sincospi_02(u2 + u2, s, c);
#endif
    z0 = r * c;
    z1 = r * s;
}

__host__ __device__ __forceinline__ uint32_t ctr_word3(uint32_t stream, uint32_t layout, uint32_t call) { return (stream << 24) | (layout << 8) | call; }

// 4*DW standard normals of one tile (4 EM steps): normal n = slot*DW + j lives in call n/2 (even: cos, odd: sin)
template <int DW>
__device__ __forceinline__ void tile_normals(uint64_t seed, uint32_t chain, uint32_t gtile, uint32_t iter, uint32_t layout, double *z) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int call = 0; call < 2 * DW; call++) {
        u32x4 c = {chain, gtile, iter, ctr_word3(STREAM_PCN, layout, (uint32_t)call)};
        box_muller(philox4x32_10(c, k0, k1), z[2 * call], z[2 * call + 1]);
    }
}

// the same 4*DW normals, produced by G adjacent lanes together: lane `sub` of the group evaluates calls sub, sub+G, ... and the
// group all-gathers the pairs with shuffles (every lane of the warp must call this)
template <int DW, int G>
__device__ __forceinline__ void tile_normals_coop(uint64_t seed, uint32_t chain, uint32_t gtile, uint32_t iter, uint32_t layout, int sub, double *z) {
    constexpr int NC = 2 * DW, PER = (NC + G - 1) / G;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    double zl[2 * PER];
#pragma unroll
    for (int p = 0; p < PER; p++) {
        const int call = min(sub + p * G, NC - 1); // (a lane past the end repeats the last call; its result is not gathered)
        u32x4 c = {chain, gtile, iter, ctr_word3(STREAM_PCN, layout, (uint32_t)call)};
        box_muller(philox4x32_10(c, k0, k1), zl[2 * p], zl[2 * p + 1]);
    }
#pragma unroll
    for (int call = 0; call < NC; call++) {
        z[2 * call] = __shfl_sync(0xffffffffu, zl[2 * (call / G)], call % G, G);
        z[2 * call + 1] = __shfl_sync(0xffffffffu, zl[2 * (call / G) + 1], call % G, G);
    }
}

__device__ __forceinline__ double accept_exponential(uint64_t seed, uint32_t chain, uint32_t block, uint32_t iter, uint32_t layout) {
    u32x4 c = {chain, block, iter, ctr_word3(STREAM_ACC, layout, 0u)};
    u32x4 o = philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    uint64_t w0 = ((uint64_t)o.y << 32) | o.x;
#if DMT_LIBDEVICE_MATH
    return -log((double)((w0 >> 11) + 1ull) * 0x1.0p-53);
#else
    return -log_pos_normal((double)((w0 >> 11) + 1ull) * 0x1.0p-53);
#endif
}

} // namespace dmt
