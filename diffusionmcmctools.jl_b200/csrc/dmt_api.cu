// dmt_api.cu — the C ABI of include/dmt.h: context management, uploads, kernel launches.
// No torch types, no CPU fallback: every compute entry point launches sm_100a kernels or fails.
#include "../../include/dmt.h"
#include "kernels.cuh"
#include "fwd_kernel.cuh"
#include "sweep_kernel.cuh"
#include "sweep_ws_kernel.cuh"
#include "sweep_sp_kernel.cuh"
#include "tsit5_kernel.cuh"
#include "moments_kernel.cuh"

#include <algorithm>
#include <atomic>
#include <nvtx3/nvToolsExt.h> // header-only: ranges are emitted when DMT_NVTX=1 and a profiler is attached
#include <cmath>
#include <cstdio>
#include <cstring>
#include <dlfcn.h>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

using namespace dmt;

// tuning builds may compile a single model (-DDMT_ONLY_MODEL=2) to cut nvcc time; the shipped library has all six
#ifdef DMT_ONLY_MODEL
#define DMT_FOR_MODELS(X) X(DMT_ONLY_MODEL)
#else
#define DMT_FOR_MODELS(X) X(M_FHN) X(M_LV) X(M_LORENZ) X(M_PROK) X(M_JR) X(M_OU2)
#endif

namespace {

struct DmtError : std::runtime_error {
    int code;
    DmtError(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

#define CK(call)                                                                                                   \
    do {                                                                                                           \
        cudaError_t e_ = (call);                                                                                   \
        if (e_ != cudaSuccess)                                                                                     \
            throw DmtError(DMT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                      \
    } while (0)
#define REQUIRE(cond, code, msg)                                                                                   \
    do {                                                                                                           \
        if (!(cond)) throw DmtError(code, msg);                                                                    \
    } while (0)

std::string g_create_error;
std::atomic<unsigned long long> g_launches{0}; // kernels launched by this library in this process, all contexts (dmt_launch_count)

struct ModelDims { int D, DW, NPAR; bool constdiff; };
bool model_dims(int model, ModelDims &md) {
    switch (model) {
    case M_FHN: md = {Model<M_FHN>::D, Model<M_FHN>::DW, Model<M_FHN>::NPAR, Model<M_FHN>::CONSTDIFF}; return true;
    case M_LV: md = {Model<M_LV>::D, Model<M_LV>::DW, Model<M_LV>::NPAR, Model<M_LV>::CONSTDIFF}; return true;
    case M_LORENZ: md = {Model<M_LORENZ>::D, Model<M_LORENZ>::DW, Model<M_LORENZ>::NPAR, Model<M_LORENZ>::CONSTDIFF}; return true;
    case M_PROK: md = {Model<M_PROK>::D, Model<M_PROK>::DW, Model<M_PROK>::NPAR, Model<M_PROK>::CONSTDIFF}; return true;
    case M_JR: md = {Model<M_JR>::D, Model<M_JR>::DW, Model<M_JR>::NPAR, Model<M_JR>::CONSTDIFF}; return true;
    case M_OU2: md = {Model<M_OU2>::D, Model<M_OU2>::DW, Model<M_OU2>::NPAR, Model<M_OU2>::CONSTDIFF}; return true;
    }
    return false;
}

// Ordering rule: every copy and fill goes on the context's stream (ctx->stream), in order with the kernels that use the memory.
// Only the asynchronous read-backs (dmt_snapshot_paths_async, dmt_histories_async) run on copy_stream, behind an event.  The
// context's stream is non-blocking: nothing may go on the legacy default stream, which it does not order against.  An entry point
// that hands host memory to an async copy waits for ctx->stream before it returns.
template <class T> struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    void alloc_uninit(size_t count) {
        release();
        n = count;
        if (count) CK(cudaMalloc(&p, count * sizeof(T)));
    }
    void alloc(size_t count, cudaStream_t stream) { // zero-filled
        alloc_uninit(count);
        if (count) CK(cudaMemsetAsync(p, 0, count * sizeof(T), stream));
    }
    // the contents of `host`; the storage is kept when the size matches
    void upload(const std::vector<T> &host, cudaStream_t stream) {
        if (n != host.size()) alloc_uninit(host.size());
        if (n) CK(cudaMemcpyAsync(p, host.data(), n * sizeof(T), cudaMemcpyHostToDevice, stream));
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
    ~DevBuf() { release(); }
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
};

struct Layout {
    bool set = false;
    int nb = 0;
    std::vector<int> i0, i1;
    std::vector<uint8_t> last;
    DevBuf<int> d_i0, d_i1;
    DevBuf<uint8_t> d_last, d_ok, d_last_acc, d_acc_hist;
    DevBuf<double> d_rho, d_ll, d_ll_hist; // d_rho: [nb][M]
    LayoutDev dev{};
    // pCN memory adaptation (dmt_set_rho_adaptation): per (block, chain) the logit s of ρ in (rho_min, rho_max) and the accepts of the
    // current window; the call counter is the same on every rank, so it stays on the host
    bool adapt = false;
    double ad_target = 0, ad_gamma0 = 0, ad_decay = 0, ad_rho_min = 0, ad_rho_max = 0;
    int ad_window = 0;
    uint64_t ad_calls = 0;
    DevBuf<double> d_ad_s;
    DevBuf<int32_t> d_ad_nacc;
    // guiding cache (dmt_enable_guiding_cache): layout-private accepted-law guiding term + its affine decomposition in v
    bool cache_enabled = false, cache_valid = false;
    bool F_stale = false; // cache valid but F/c of the private store not materialised for the current artificial observations
    DevBuf<double> d_Gl[2], d_c0l[2], d_FP[2], d_cq, d_vlast;
    DevBuf<int> d_blk_of_k;
    // the persistent schedule of the pipelined sweep (PipeSched, sweep_kernel.cuh): its task entries, tickets and hand-over state
    DevBuf<int> d_task;
    DevBuf<unsigned> d_ticket;
    DevBuf<double> d_hand;
};

// ---- NCCL, resolved at run time so that libdmt.so has no link-time dependency on it
struct NcclApi {
    void *h = nullptr;
    int (*GetUniqueId)(void *) = nullptr;
    int (*CommInitRank)(void **, int, struct UidByValue, int) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
struct UidByValue { char internal[128]; };
NcclApi g_nccl;
void load_nccl() {
    if (g_nccl.h) return;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *nm : names) {
        g_nccl.h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.h) break;
    }
    REQUIRE(g_nccl.h, DMT_ERR_NCCL, std::string("dlopen(libnccl.so.2) failed: ") + dlerror());
    g_nccl.GetUniqueId = (int (*)(void *))dlsym(g_nccl.h, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(void **, int, UidByValue, int))dlsym(g_nccl.h, "ncclCommInitRank");
    g_nccl.AllReduce = (int (*)(const void *, void *, size_t, int, int, void *, cudaStream_t))dlsym(g_nccl.h, "ncclAllReduce");
    g_nccl.CommDestroy = (int (*)(void *))dlsym(g_nccl.h, "ncclCommDestroy");
    g_nccl.GetErrorString = (const char *(*)(int))dlsym(g_nccl.h, "ncclGetErrorString");
    REQUIRE(g_nccl.GetUniqueId && g_nccl.CommInitRank && g_nccl.AllReduce && g_nccl.CommDestroy, DMT_ERR_NCCL, "NCCL symbols missing");
}
#define NCK(call)                                                                                                  \
    do {                                                                                                           \
        int r_ = (call);                                                                                           \
        if (r_ != 0)                                                                                               \
            throw DmtError(DMT_ERR_NCCL, std::string(#call) + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "nccl error")); \
    } while (0)

} // namespace

struct dmt_ctx {
    dmt_config cfg{};
    ModelDims md{};
    int D = 0, DW = 0, NPAR = 0, NH = 0, NG = 0, NAUX = 0, NOBS = 0;
    int K = 0, M = 0, P = 0, m = 0, NT = 0, NTb = 0, S = 0, NP = 0;
    std::vector<int> nsteps, tile0, step0, pt0, ppb_tile0, pset; // host copies of the d_ maps below
    cudaStream_t stream = nullptr;
    DevCtx dev{};
    std::vector<Layout> layouts;
    std::string err;
    // device storage
    DevBuf<int> d_tile0, d_step0, d_pt0, d_nsteps, d_ppb_tile0, d_pset, d_k_of_tile, d_k_of_ppbtile;
    DevBuf<double> d_dt, d_sqdt, d_X, d_W, d_X0;
    DevBuf<uint8_t> d_parX, d_parW, d_parP[2];
    DevBuf<double> d_G[2][2], d_c0[2][2], d_theta[2][2], d_aux[2][2], d_obs[2], d_vart[2];
    DevBuf<double> d_scratch, d_partial, d_stats;
    DevBuf<uint8_t> d_mask;
    DevBuf<int> d_flag;
    void *nccl_comm = nullptr;
    // peer-memory all-reduce (dmt_p2p_export / dmt_p2p_init)
    P2PBuf *p2p_local = nullptr;
    P2PArgs p2p{};
    bool p2p_ready = false;
    int n_ranks = 1;
    int fwd_lanes = 0;       // dmt_set_fwd_lanes: 0 = automatic
    int bwd_solver = 0;      // dmt_set_bwd_solver: 0 = classical RK4 on the path grid, 1 = adaptive Tsit5 (upstream's solver)
    double bwd_reltol = 1e-3, bwd_abstol = 1e-6;
    DevBuf<int> d_steps;     // accepted / rejected steps of the last Tsit5 launch
    int bwd_mode = 0;        // dmt_set_bwd_mode: 0 = automatic, 1 = one thread per (pset, block), 2 = lanes cooperate on one pset
    DevBuf<double> d_xbar[2]; // linearisation points [K][D][P] per store, kept so that a parameter update re-linearises on the device
    std::vector<char> xbar_set[2];
    // thinned path saving (dmt_snapshot_paths_async): staging buffer + copy stream
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_gathered = nullptr, ev_copied = nullptr, ev_hist = nullptr;
    DevBuf<double> d_snap;
    DevBuf<int> d_snap_sel;
    bool pipe_ok = false;    // P == M with the identity pset map: a warp's guiding-term sectors are contiguous (sweep_pipe_kernel)
    int sweep_mode = 0;      // dmt_set_sweep_mode: 0 = automatic (pick_sweep), 1 = register-tile kernel, 2 / 3 / 5 = pipelined /
                             // warp-specialised / step-parallel kernel or error
    std::unordered_map<const void *, size_t> resident; // kernel -> CTAs resident at once on this context's device (resident_ctas)
    int n_sm = 0;            // SMs of this context's device (resident_ctas)
    bool lazy_W = false;     // dmt_set_lazy_noise: blocking sweeps do not materialise W_acc / W°
    char last_fwd_kernel[96] = ""; // name and mapping of the forward kernel launched last (dmt_get_last_forward_kernel)
    int W_stale_layout = -1; // >= 0: W_acc is not materialised; K5 over this layout rebuilds it (ensure_W)
    int G_owner = -1;        // layout whose K1 wrote the shared accepted-law store last (-1: unknown / laws changed)
    bool parP_mixed = false; // a masked swap_PP! made the law parity chain-dependent
    bool aux_all_linearised = true; // every auxiliary law so far came from dmt_set_aux_linearised: B has the Jacobian's sparsity (JacMask)
    // posterior path moments (dmt_path_moments_add): per-chain Welford accumulators in the X layout, tiles then interval starts,
    // [NT*D*M*4 + K*D*M] each; allocated on the first update.  Per-pset chain lists (CSR) built on the first pooled read.
    DevBuf<double> d_pm_mean, d_pm_m2;
    uint64_t pm_count = 0;
    DevBuf<int> d_pm_cs, d_pm_chains;

    double *scratch(size_t n) {
        if (d_scratch.n < n) d_scratch.alloc_uninit(n);
        return d_scratch.p;
    }
};

namespace {

Layout &layout_of(dmt_ctx *c, int id) {
    REQUIRE(id >= 0 && id < (int)c->layouts.size(), DMT_ERR_ARG, "layout index out of range");
    REQUIRE(c->layouts[id].set, DMT_ERR_STATE, "layout not registered (dmt_set_blocks)");
    return c->layouts[id];
}

void check_side(dmt_ctx *c, int side) {
    REQUIRE(side == 0 || side == 1, DMT_ERR_ARG, "side must be 0 (accepted) or 1 (proposal)");
}
void check_law_side(dmt_ctx *c, int side) {
    check_side(c, side);
    REQUIRE(side == 0 || c->cfg.two_sided_laws, DMT_ERR_STATE, "proposal laws not allocated (dmt_config.two_sided_laws = 0)");
}
void check_range(dmt_ctx *c, int k0, int k1) { REQUIRE(0 <= k0 && k0 <= k1 && k1 < c->K, DMT_ERR_ARG, "interval range out of bounds"); }

dim3 chain_grid(dmt_ctx *c, int ny, int tpb) { return dim3((c->M + tpb - 1) / tpb, ny, 1); }
dim3 pset_grid(dmt_ctx *c, int ny, int tpb, int nz = 1) { return dim3((c->P + tpb - 1) / tpb, ny, nz); }

// CTAs of `kernel` resident at once on the context's device with `threads` threads and `smem` bytes of dynamic shared memory each.
// Raises the kernel's dynamic-shared-memory limit to `smem` first, so every launch of the kernels below goes through here once
// before its first launch.  Cached per context: the answer depends on the device, and a context owns one device.
template <class Kernel> size_t resident_ctas(dmt_ctx *c, Kernel *kernel, int threads, size_t smem) {
    const auto it = c->resident.find((const void *)kernel);
    if (it != c->resident.end()) return it->second;
    int per_sm = 0;
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    if (!c->n_sm) CK(cudaDeviceGetAttribute(&c->n_sm, cudaDevAttrMultiProcessorCount, c->cfg.device));
    return c->resident[(const void *)kernel] = (size_t)per_sm * c->n_sm;
}

// ---- the register-tile kernel (fwd_kernel.cuh): G lanes per (chain, block), G > 1 for the ops that draw normals
template <int OP> constexpr bool fwd_coop() { return OP == OP_DRAW || OP == OP_INIT || OP == OP_SWEEP; }
template <class MD> constexpr int fwd_tpb() { return MD::D >= 6 ? 32 : FWD_TPB; } // wide guiding terms: smaller CTAs
template <class MD, int OP, int G> size_t fwd_wave_threads(dmt_ctx *c) {
    return resident_ctas(c, fwd_kernel<MD, OP, fwd_tpb<MD>(), G>, fwd_tpb<MD>(), 0) * fwd_tpb<MD>();
}
template <class MD, int OP, int G> void launch_fwd_g(dmt_ctx *c, Layout &L, const FwdArgs &fa) {
    constexpr int TPB = fwd_tpb<MD>();
    fwd_wave_threads<MD, OP, G>(c);
    const dim3 grid((unsigned)(((size_t)c->M * G + TPB - 1) / TPB), L.nb, 1);
    snprintf(c->last_fwd_kernel, sizeof(c->last_fwd_kernel), "fwd_kernel<op=%d, lanes=%d%s>", OP, G, (OP == OP_SWEEP && fa.lazy_w) ? ", lazy" : "");
    ++g_launches, fwd_kernel<MD, OP, TPB, G><<<grid, TPB, 0, c->stream>>>(c->dev, L.dev, fa);
}
template <class MD, int OP> void launch_fwd_tile(dmt_ctx *c, Layout &L, const FwdArgs &fa, int lanes) {
    if constexpr (fwd_coop<OP>()) {
        if (lanes == 8) return launch_fwd_g<MD, OP, 8>(c, L, fa);
        if (lanes == 4) return launch_fwd_g<MD, OP, 4>(c, L, fa);
        if (lanes == 2) return launch_fwd_g<MD, OP, 2>(c, L, fa);
    }
    launch_fwd_g<MD, OP, 1>(c, L, fa);
}
// Lanes per (chain, block): dmt_set_fwd_lanes if set; else 1 when the ensemble fills the GPU by itself, and 2, 4 or 8 when
// chains x blocks x lanes still fits one wave (the generator is split over the lanes, fwd_kernel.cuh).
template <class MD, int OP> int tile_lanes(dmt_ctx *c, const Layout &L) {
    if constexpr (fwd_coop<OP>()) {
        if (c->fwd_lanes) return c->fwd_lanes;
        // with one Wiener coordinate the generator is a small part of the tile: redundant lanes only cost issue slots
        // (Jansen-Rit draw, 8192 chains: 87 ms with 1 lane, 121 ms with 4)
        if (MD::DW < 2) return 1;
        const size_t units = (size_t)c->M * L.nb;
        if (OP != OP_SWEEP) {
            if (units * 8 <= fwd_wave_threads<MD, OP, 8>(c)) return 8;
            if (units * 4 <= fwd_wave_threads<MD, OP, 4>(c)) return 4;
        }
        // the fused sweep: two lanes whenever the doubled grid still fits one wave — measured best at every ensemble size where
        // it applies (Lorenz, lazy noise, fused pass in ms for 512 / 768 / 1024 / 1536 chains: 1 lane 2.12 / 2.14 / 2.15 / 2.17,
        // 2 lanes 1.03 / 1.05 / 1.35 / 1.39, 4 lanes 1.14 / 1.17 / 1.81 / 2.29; profiles/r02_tuning.md)
        if (units * 2 <= fwd_wave_threads<MD, OP, 2>(c)) return 2;
    }
    return 1;
}

void ensure_guiding(dmt_ctx *c, Layout &L);
void ensure_W(dmt_ctx *c);
bool covers_all_intervals(dmt_ctx *c, const Layout &L) {
    std::vector<char> seen(c->K, 0);
    for (int b = 0; b < L.nb; b++)
        for (int k = L.i0[b]; k <= L.i1[b]; k++) seen[k] = 1;
    return std::all_of(seen.begin(), seen.end(), [](char s) { return s != 0; });
}

// ---- the other kernels of the fused sweep pass.  All three need one parameter set per chain in chain order, uniform law parity
// and device RNG; each is compiled with and without lazy noise.
// the software-pipelined sweep (sweep_kernel.cuh): one lane per (chain, block), guiding term through a TMA shared-memory ring.
// Schedule, with S = 4 schedulers x SMs and U = (32-chain group, block) units: one unit per warp leaves up to three warps on some
// schedulers, and the pass lasts as long as those do (Lorenz, C3: 1.40 / 1.72 / 2.32 ms for at most 1 / 2 / 3 warps per scheduler,
// profiles/r02_tuning.md §4d).  So where U allows an even spread the grid is persistent (PipeSched) and warps take the units'
// intervals by ticket: 2S warps, two on every scheduler, when U >= 2S; S warps when S <= U < 1.23 S (1.23 = 1.72 / 1.40: one warp per
// scheduler at the one-warp rate beats U / S warps at the two-warp rate); else one unit per warp.  For d <= 3 the warps come four to a
// CTA, two CTAs per SM; wider models keep one-warp CTAs (four warps' rings do not fit twice).  profiles/r03_tuning.md.
template <class MD, bool LAZY> void launch_sweep_pipe(dmt_ctx *c, Layout &L, const FwdArgs &fa) {
    constexpr size_t smem = sweep_pipe_smem<MD>();
    constexpr int WPC = MD::D <= 3 ? 4 : 1;
    const size_t groups = (c->M + 31) / 32, units = groups * L.nb;
    const size_t warps = resident_ctas(c, sweep_pipe_kernel<MD, LAZY, WPC>, 32 * WPC, WPC * smem) * WPC;
    const size_t S = (size_t)c->n_sm * 4;
    const size_t n = std::min(warps, units >= 2 * S ? 2 * S : (units >= S && units * 100 < S * 123) ? S : 0);
    snprintf(c->last_fwd_kernel, sizeof(c->last_fwd_kernel), "sweep_pipe_kernel<lanes=1%s>", LAZY ? ", lazy" : "");
    if (n < S) {
        resident_ctas(c, sweep_pipe_kernel<MD, LAZY, 1>, 32, smem);
        ++g_launches, sweep_pipe_kernel<MD, LAZY, 1><<<dim3((unsigned)groups, L.nb, 1), 32, smem, c->stream>>>(c->dev, L.dev, fa, PipeSched{});
        return;
    }
    if (L.d_ticket.n != 1 + units) L.d_ticket.alloc_uninit(1 + units);
    if (L.d_hand.n != (size_t)(MD::D + 3) * units * 32) L.d_hand.alloc_uninit((size_t)(MD::D + 3) * units * 32);
    CK(cudaMemsetAsync(L.d_ticket.p, 0, sizeof(unsigned) * (1 + units), c->stream));
    const PipeSched sc{L.d_task.p, (int)(L.d_task.n * groups), L.d_ticket.p, L.d_hand.p};
    ++g_launches, sweep_pipe_kernel<MD, LAZY, WPC><<<(unsigned)(n / WPC), 32 * WPC, WPC * smem, c->stream>>>(c->dev, L.dev, fa, sc);
}
// the warp-specialised sweep (sweep_ws_kernel.cuh): a pipeline of 16 warps per group of 32 chains and block, one CTA per SM.  Six
// generator warps; ring depths by state dimension (a stage of the G ring is (d(d+1)/2 + d) KiB, the D ring holds the same again per
// slot): G ring 8 / 6 / 3 stages and Z, D, X rings 4 / 3 / 2 slots for d <= 3 / d = 4 / d >= 5
template <class MD> using WsWide = WsShape<6, (MD::D <= 3 ? 8 : MD::D == 4 ? 6 : 3), (MD::D <= 3 ? 4 : MD::D == 4 ? 3 : 2)>;
template <class MD, bool LAZY> size_t ws_resident_ctas(dmt_ctx *c) {
    constexpr size_t smem = sweep_ws_smem<MD, WsWide<MD>>();
    static_assert(smem <= 227 * 1024, "the rings of the warp-specialised sweep must fit one SM's shared memory");
    return resident_ctas(c, sweep_ws_kernel<MD, LAZY, WsWide<MD>>, WsWide<MD>::THREADS, smem);
}
template <class MD, bool LAZY> void launch_sweep_ws(dmt_ctx *c, Layout &L, const FwdArgs &fa) {
    using SH = WsWide<MD>;
    ws_resident_ctas<MD, LAZY>(c);
    const dim3 grid((unsigned)((c->M + 31) / 32), L.nb, 1);
    snprintf(c->last_fwd_kernel, sizeof(c->last_fwd_kernel), "sweep_ws_kernel<wide, %s>", LAZY ? "lazy" : "eager");
    ++g_launches, sweep_ws_kernel<MD, LAZY, SH><<<grid, SH::THREADS, sweep_ws_smem<MD, SH>(), c->stream>>>(c->dev, L.dev, fa);
}
// the step-parallel sweep (sweep_sp_kernel.cuh): four lanes per (chain, block), lane = step of the tile
template <class MD, bool LAZY> void launch_sweep_sp(dmt_ctx *c, Layout &L, const FwdArgs &fa) {
    const dim3 grid((unsigned)((c->M + 7) / 8), L.nb, 1);
    snprintf(c->last_fwd_kernel, sizeof(c->last_fwd_kernel), "sweep_sp_kernel<step lanes=4%s>", LAZY ? ", lazy" : "");
    ++g_launches, sweep_sp_kernel<MD, LAZY><<<grid, 32, 0, c->stream>>>(c->dev, L.dev, fa);
}

// What the fused sweep pass (K5 + K4 + K3 + K2 + K4, OP_SWEEP) launches: the kernel, the register-tile kernel's lanes per
// (chain, block), and whether the pass skips the W_acc / W° stores (dmt_set_lazy_noise; then W is rebuilt on demand, ensure_W)
struct SweepChoice {
    enum Kernel { TILE, PIPE, WS, SP } kernel;
    int lanes;
    bool lazy;
};
template <class MD> SweepChoice pick_sweep(dmt_ctx *c, const Layout &L, const FwdArgs &fa) {
    const bool lazy = c->lazy_W && !fa.Z && covers_all_intervals(c, L);
    const bool eligible = c->pipe_ok && !c->parP_mixed && !fa.Z && fa.skip == 0;
    const int mode = c->sweep_mode;
    if (mode >= 2) { // forced: 2 pipelined, 3 warp-specialised, 5 step-parallel
        REQUIRE(eligible, DMT_ERR_UNSUPPORTED, "pipelined sweep needs one parameter set per chain in chain order, uniform law parity and device RNG");
        if (mode == 3) return {SweepChoice::WS, 1, lazy};
        if (mode == 5) return {SweepChoice::SP, 1, lazy};
        REQUIRE(c->fwd_lanes <= 1, DMT_ERR_UNSUPPORTED, "the pipelined sweep maps one lane to a (chain, block)");
        return {SweepChoice::PIPE, 1, lazy};
    }
    const SweepChoice tile{SweepChoice::TILE, tile_lanes<MD, OP_SWEEP>(c, L), lazy};
    if (mode == 1 || !eligible || c->fwd_lanes) return tile;
    // automatic.  Warp-specialised while its grid fits ONE round of CTAs: a round costs ~0.5 ms on C3 whatever the ensemble size, so a
    // second round loses to the one-thread-per-(chain, block) kernels (profiles/r02_tuning.md).
    const size_t ws_units = (size_t)((c->M + 31) / 32) * L.nb;
    if (ws_units <= (lazy ? ws_resident_ctas<MD, true>(c) : ws_resident_ctas<MD, false>(c))) return {SweepChoice::WS, 1, lazy};
    // Then step-parallel up to 14,080 (chain, block) units: 1280 chains x 11 blocks (12 resident warps per SM at 168 registers).
    // Measured (Lorenz, lazy noise, fused pass in ms at 512 / 1024 / 1280 chains x 10 blocks; profiles/r02_tuning.md §4e):
    // step-parallel 0.83 / 1.10 / 1.18, two lanes per (chain, block) in the register-tile kernel 1.03 / 1.35 / 1.37.
    if (MD::DW >= 2 && (size_t)c->M * L.nb <= 14080) return {SweepChoice::SP, 1, lazy};
    // Then the register-tile kernel with two lanes while that grid fits one wave (1.35 against 1.40 ms for the pipelined kernel at
    // 1024 chains, 1.03 against 1.38 ms at 512).  With the noise stored every sweep the pipelined kernel's live set (two more tile
    // buffers) spills and it loses to the register-tile kernel (3.9 against 3.5 ms on C3); it wins where the noise is lazy (2.44 ms).
    if (tile.lanes == 2 || !lazy) return tile;
    return {SweepChoice::PIPE, 1, lazy};
}

template <class MD, int OP> void launch_fwd_model(dmt_ctx *c, Layout &L, FwdArgs fa) {
    if constexpr (OP == OP_SWEEP) {
        const SweepChoice s = pick_sweep<MD>(c, L, fa);
        fa.lazy_w = s.lazy;
        switch (s.kernel) {
        case SweepChoice::TILE: launch_fwd_tile<MD, OP>(c, L, fa, s.lanes); break;
        case SweepChoice::PIPE: s.lazy ? launch_sweep_pipe<MD, true>(c, L, fa) : launch_sweep_pipe<MD, false>(c, L, fa); break;
        case SweepChoice::WS: s.lazy ? launch_sweep_ws<MD, true>(c, L, fa) : launch_sweep_ws<MD, false>(c, L, fa); break;
        case SweepChoice::SP: s.lazy ? launch_sweep_sp<MD, true>(c, L, fa) : launch_sweep_sp<MD, false>(c, L, fa); break;
        }
        if (s.lazy) c->W_stale_layout = L.dev.id;
    } else {
        launch_fwd_tile<MD, OP>(c, L, fa, tile_lanes<MD, OP>(c, L));
    }
}

template <int OP> void launch_fwd(dmt_ctx *c, Layout &L, const FwdArgs &fa) {
    // lazy noise (dmt_set_lazy_noise): an op that reads W, or rewrites only part of it, first rebuilds it from X; an op that
    // rewrites all of it just clears the flag
    if (c->W_stale_layout >= 0 && OP != OP_LOGLIK) {
        const bool rewrites_all = (OP == OP_INIT) || ((OP == OP_INVSOLVE || OP == OP_INVSOLVE_LL || OP == OP_SWEEP) && covers_all_intervals(c, L));
        if (rewrites_all) c->W_stale_layout = -1;
        else ensure_W(c);
    }
    ensure_guiding(c, L);
#define DMT_CASE(MID)                                                                                              \
    case MID: launch_fwd_model<Model<MID>, OP>(c, L, fa); break;
    switch (c->cfg.model) {
        DMT_FOR_MODELS(DMT_CASE)
        default: throw DmtError(DMT_ERR_UNSUPPORTED, "model not compiled into this build of libdmt");
    }
#undef DMT_CASE
    CK(cudaGetLastError());
}

template <class MD> void launch_bwd_model(dmt_ctx *c, Layout &L, const BwdArgs &ba) {
    const int nz = c->cfg.two_sided_laws ? 2 : 1;
    if (c->bwd_solver == 1) { // upstream's solver (tsit5_kernel.cuh); the guiding cache's probes need the fixed-grid discretisation
        REQUIRE(!ba.use_override, DMT_ERR_UNSUPPORTED, "the guiding cache needs the RK4 backward filter (its F is affine in v only there)");
        if (c->d_steps.n < 2) c->d_steps.alloc(2, c->stream);
        CK(cudaMemsetAsync(c->d_steps.p, 0, 2 * sizeof(int), c->stream));
        Tsit5Args ta{ba.side_mask, c->bwd_reltol, c->bwd_abstol, c->d_steps.p};
        ++g_launches, bwd_tsit5_kernel<MD><<<pset_grid(c, L.nb, 32, nz), 32, 0, c->stream>>>(c->dev, L.dev, ta);
        return;
    }
    bool all_terminal = true;
    for (int b = 0; b < L.nb; b++) all_terminal = all_terminal && L.last[b];
    const bool coop_ok = MD::ATIL_DIAG && MD::D >= 5 && all_terminal;
    REQUIRE(c->bwd_mode != 2 || coop_ok, DMT_ERR_UNSUPPORTED, "cooperative backward filter not available for this model / layout");
    if (coop_ok && c->bwd_mode != 1) {
        // wide state, no exact-observation interval: D lanes per parameter set (kernels.cuh, bwd_coop_kernel)
        constexpr int per_cta = 4 * (32 / MD::D);
        const dim3 grid((c->P + per_cta - 1) / per_cta, L.nb, nz);
        if (JacMask<MD>::SPARSE && c->aux_all_linearised && !getenv("DMT_K1_DENSE"))
            ++g_launches, bwd_coop_kernel<MD, JacMask<MD>::SPARSE><<<grid, 128, 0, c->stream>>>(c->dev, L.dev, ba);
        else
            ++g_launches, bwd_coop_kernel<MD, false><<<grid, 128, 0, c->stream>>>(c->dev, L.dev, ba);
    } else {
        ++g_launches, bwd_kernel<MD><<<pset_grid(c, L.nb, BWD_TPB, nz), BWD_TPB, 0, c->stream>>>(c->dev, L.dev, ba);
    }
}

void launch_bwd(dmt_ctx *c, Layout &L, int side_mask, const double *v_override = nullptr) {
    if ((side_mask & 1) && !(L.cache_enabled && L.dev.Gl[0])) c->G_owner = v_override ? -1 : L.dev.id; // accepted laws, shared store
    BwdArgs ba{};
    ba.side_mask = side_mask;
    if (v_override) {
        ba.use_override = 1;
        for (int i = 0; i < c->D; i++) ba.v[i] = v_override[i];
    }
#define DMT_CASE(MID)                                                                                              \
    case MID: launch_bwd_model<Model<MID>>(c, L, ba); break;
    switch (c->cfg.model) {
        DMT_FOR_MODELS(DMT_CASE)
        default: throw DmtError(DMT_ERR_UNSUPPORTED, "model not compiled into this build of libdmt");
    }
#undef DMT_CASE
    CK(cudaGetLastError());
}

// ---- guiding cache (see kernels.cuh "guiding cache"): build by probing bwd_kernel, apply per sweep
#define DMT_D_SWITCH(Dval, ...)                                                                                    \
    switch (Dval) {                                                                                                \
    case 2: { constexpr int DD = 2; __VA_ARGS__; } break;                                                          \
    case 3: { constexpr int DD = 3; __VA_ARGS__; } break;                                                          \
    case 4: { constexpr int DD = 4; __VA_ARGS__; } break;                                                          \
    case 6: { constexpr int DD = 6; __VA_ARGS__; } break;                                                          \
    default: throw DmtError(DMT_ERR_UNSUPPORTED, "state dimension not supported by the guiding cache");          \
    }

void cache_set_private(Layout &L, bool on) {
    for (int st = 0; st < 2; st++) {
        L.dev.Gl[st] = on ? L.d_Gl[st].p : nullptr;
        L.dev.c0l[st] = on ? L.d_c0l[st].p : nullptr;
    }
}
void invalidate_caches(dmt_ctx *c) { // every caller is about to change the accepted laws (or just did, for parity flips)
    c->G_owner = -1;
    for (auto &L : c->layouts) {
        L.cache_valid = false;
        L.F_stale = false;
        cache_set_private(L, false);
    }
}
void cache_apply(dmt_ctx *c, Layout &L) { // the per-sweep K1: F = F0 + Psi v ; c = c0 + q.v + v'Qv/2
    L.F_stale = false;
    int tiles_max = 1; // longest block, in tiles: ~24 tile groups per thread
    for (int b = 0; b < L.nb; b++) tiles_max = std::max(tiles_max, c->tile0[L.i1[b] + 1] - c->tile0[L.i0[b]]);
    const int Z = std::min(16, std::max(1, tiles_max / (FPG * 24)));
    const dim3 g(((size_t)c->P * FPG + 127) / 128, L.nb, Z);
    DMT_D_SWITCH(c->D,
                 ++g_launches, cache_apply_kernel<DD><<<g, 128, 0, c->stream>>>(c->dev, L.dev);
                 ++g_launches, cache_apply_c_kernel<DD><<<pset_grid(c, L.nb, 128), 128, 0, c->stream>>>(c->dev, L.dev));
    CK(cudaGetLastError());
}
void cache_build(dmt_ctx *c, Layout &L) {
    const size_t P = c->P, NF = c->D + c->D * c->D, NC = 1 + c->D + c->NH;
    const size_t nt[2] = {(size_t)c->NT, (size_t)std::max(c->NTb, 1)};
    for (int st = 0; st < 2; st++) {
        if (L.d_Gl[st].n != nt[st] * c->NG * P * 4) L.d_Gl[st].alloc(nt[st] * c->NG * P * 4, c->stream);
        if (L.d_FP[st].n != fp_tiles_padded(nt[st]) * NF * P * 4) L.d_FP[st].alloc(fp_tiles_padded(nt[st]) * NF * P * 4, c->stream);
        if (L.d_c0l[st].n != (size_t)c->K * P) L.d_c0l[st].alloc((size_t)c->K * P, c->stream);
        L.dev.FP[st] = L.d_FP[st].p;
    }
    if (L.d_cq.n != (size_t)L.nb * NC * P) L.d_cq.alloc((size_t)L.nb * NC * P, c->stream);
    L.dev.cq = L.d_cq.p;
    // "no end point seen yet": NaN compares unequal to everything, so the first apply after a (re)build materialises every block
    L.d_vlast.upload(std::vector<double>((size_t)L.nb * c->D * P, NAN), c->stream);
    CK(cudaStreamSynchronize(c->stream));
    L.dev.v_last = L.d_vlast.p;
    {
        std::vector<int> bk(c->K, 0);
        for (int b = 0; b < L.nb; b++)
            for (int k = L.i0[b]; k <= L.i1[b]; k++) bk[k] = b;
        L.d_blk_of_k.upload(bk, c->stream);
        CK(cudaStreamSynchronize(c->stream));
        L.dev.blk_of_k = L.d_blk_of_k.p;
    }
    cache_set_private(L, true); // the probe runs below write the private store through these pointers
    try {
    const int D = c->D, nruns = 1 + 2 * D + D * (D - 1) / 2;
    const double s = 8.0; // probe scale (a power of two: exact scaling)
    DevBuf<double> Crun;
    Crun.alloc((size_t)nruns * L.nb * P, c->stream);
    const dim3 g0((c->P + 127) / 128, c->NT), g1((c->P + 127) / 128, std::max(c->NTb, 1));
    std::vector<std::vector<double>> probes;
    probes.push_back(std::vector<double>(6, 0.0));
    for (int sign = 1; sign >= -1; sign -= 2)
        for (int m = 0; m < D; m++) { std::vector<double> v(6, 0.0); v[m] = sign * s; probes.push_back(v); }
    for (int m = 0; m < D; m++)
        for (int n = m + 1; n < D; n++) { std::vector<double> v(6, 0.0); v[m] = s; v[n] = s; probes.push_back(v); }
    for (int r = 0; r < nruns; r++) {
        launch_bwd(c, L, DMT_P_ONLY, probes[r].data());
        ++g_launches, cache_collect_c_kernel<<<pset_grid(c, L.nb, 128), 128, 0, c->stream>>>(c->dev, L.dev, r, Crun.p);
        if (r <= D) {
            const int mode = r == 0 ? 0 : 1, m = r - 1;
            DMT_D_SWITCH(c->D,
                         ++g_launches, cache_extract_kernel<DD><<<g0, 128, 0, c->stream>>>(c->dev, L.dev, 0, c->d_k_of_tile.p, mode, m, 1.0 / s);
                         if (c->NTb > 0) ++g_launches, cache_extract_kernel<DD><<<g1, 128, 0, c->stream>>>(c->dev, L.dev, 1, c->d_k_of_ppbtile.p, mode, m, 1.0 / s));
        }
        CK(cudaGetLastError());
    }
    DMT_D_SWITCH(c->D, ++g_launches, cache_solve_cq_kernel<DD><<<pset_grid(c, L.nb, 128), 128, 0, c->stream>>>(c->dev, L.dev, Crun.p, s));
    CK(cudaGetLastError());
    cache_apply(c, L); // the actual artificial observations
    CK(cudaStreamSynchronize(c->stream));
    } catch (...) { // a half-built private store must never be read by the forward kernels
        cache_set_private(L, false);
        L.cache_valid = false;
        throw;
    }
    L.cache_valid = true;
}
// dmt_set_lazy_noise: W_acc := the noise that reproduces X_acc under the law of the layout swept last (find_W_for_X!, K5)
void ensure_W(dmt_ctx *c) {
    if (c->W_stale_layout < 0) return;
    Layout &L = c->layouts[c->W_stale_layout];
    c->W_stale_layout = -1; // (first: launch_fwd below would recurse otherwise)
    const bool priv = L.cache_enabled && L.cache_valid;
    const int prev = c->G_owner;
    const bool borrow = !priv && prev != L.dev.id; // another layout's K1 has overwritten the shared store since the sweep
    if (borrow) launch_bwd(c, L, DMT_P_ONLY);
    launch_fwd<OP_INVSOLVE>(c, L, FwdArgs{0, 0, 0, 0, nullptr});
    if (borrow && prev >= 0) launch_bwd(c, c->layouts[prev], DMT_P_ONLY); // give the store back to the layout the caller prepared it for
}
// F_stale: the private store's F belongs to older block end points than the current artificial observations (set by paths that
// defer cache_apply); every forward launch materialises it first.  dmt_blocking_sweep itself applies the cache eagerly.
void ensure_guiding(dmt_ctx *c, Layout &L) {
    if (L.cache_enabled && L.cache_valid && L.F_stale) cache_apply(c, L);
}

// dst record arrays [K][NREC][P] (per slot, resolved by the law parity of `store`): write ncomp components at offset
// `off` for k = k0..k1 from src [nk or 1][ncomp][P]
__global__ void put_record_kernel(const DevCtx cx, int side, int store, double *rec0, double *rec1, int NREC, int off, int ncomp,
                                  int k0, int k1, const double *src, int bcast_k) {
    const int ps = blockIdx.x * blockDim.x + threadIdx.x, k = k0 + blockIdx.y;
    if (ps >= cx.P || k > k1) return;
    const size_t P = cx.P;
    const int slot = side ^ cx.parP[store][(size_t)k * P + ps];
    double *dst = slot ? rec1 : rec0;
    for (int q = 0; q < ncomp; q++)
        dst[((size_t)k * NREC + off + q) * P + ps] = src[((size_t)(bcast_k ? 0 : (k - k0)) * ncomp + q) * P + ps];
}
// accepted -> proposal copy of a whole record (equalize_*); *changed |= 1 when the proposal record differed (the reference's
// equalize_obs_params! / equalize_law_params! return exactly that, src/biblock.jl:362-363)
__global__ void copy_record_kernel(const DevCtx cx, int store, double *rec0, double *rec1, int NREC, int k0, int k1, int *changed) {
    const int ps = blockIdx.x * blockDim.x + threadIdx.x, k = k0 + blockIdx.y;
    if (ps >= cx.P || k > k1) return;
    const size_t P = cx.P;
    const int sa = cx.parP[store][(size_t)k * P + ps];
    const double *src = sa ? rec1 : rec0;
    double *dst = sa ? rec0 : rec1;
    bool diff = false;
    for (int q = 0; q < NREC; q++) {
        const double v = src[((size_t)k * NREC + q) * P + ps];
        double *d = &dst[((size_t)k * NREC + q) * P + ps];
        diff = diff || !(*d == v);
        *d = v;
    }
    if (diff) atomicOr(changed, 1);
}

void put_record(dmt_ctx *c, int side, int store, double *rec0, double *rec1, int NREC, int off, int ncomp, int k0, int k1,
                const double *host, bool bcast_k) {
    const size_t nk = bcast_k ? 1 : (size_t)(k1 - k0 + 1);
    const size_t n = nk * ncomp * c->P;
    double *tmp = c->scratch(n);
    CK(cudaMemcpyAsync(tmp, host, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    ++g_launches, put_record_kernel<<<pset_grid(c, k1 - k0 + 1, 128), 128, 0, c->stream>>>(c->dev, side, store, rec0, rec1, NREC, off, ncomp, k0,
                                                                             k1, tmp, bcast_k ? 1 : 0);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(c->stream)); // the host buffer is the caller's; scratch is reused
}

void rebuild_ppb_store(dmt_ctx *c) {
    // intervals that end a non-terminal block in ANY layout need a blocking-law guiding term (P_last, src/block.jl:68)
    std::vector<int> t0(c->K, -1);
    int nt = 0;
    std::vector<char> need(c->K, 0);
    for (auto &L : c->layouts)
        if (L.set)
            for (int b = 0; b < L.nb; b++)
                if (!L.last[b]) need[L.i1[b]] = 1;
    for (int k = 0; k < c->K; k++)
        if (need[k]) { t0[k] = nt; nt += (c->nsteps[k] + 3) / 4; }
    if (t0 == c->ppb_tile0 && nt == c->NTb) return;
    c->ppb_tile0 = t0;
    c->NTb = nt;
    CK(cudaStreamSynchronize(c->stream)); // kernels in flight still read the old map / the old store
    c->d_ppb_tile0.upload(t0, c->stream);
    for (int s = 0; s < (c->cfg.two_sided_laws ? 2 : 1); s++) {
        c->d_G[s][1].alloc((size_t)std::max(nt, 1) * c->NG * c->P * 4, c->stream);
        c->dev.G[s][1] = c->d_G[s][1].p;
    }
    c->dev.NTb = nt;
    {   // tile -> interval map of the PPb store (guiding cache kernels); a changed PPb store invalidates every cache
        std::vector<int> kt(std::max(nt, 1), 0);
        for (int k = 0; k < c->K; k++)
            if (t0[k] >= 0)
                for (int q = 0; q < (c->nsteps[k] + 3) / 4; q++) kt[t0[k] + q] = k;
        c->d_k_of_ppbtile.upload(kt, c->stream);
        invalidate_caches(c);
    }
}

void fill_stats(dmt_ctx *c, Layout &L, double *host_out /* [2+3nb] */) {
    const int ncta = (c->M + 255) / 256;
    if (c->d_partial.n < (size_t)3 * L.nb * ncta) c->d_partial.alloc((size_t)3 * L.nb * ncta, c->stream);
    if (c->d_stats.n < (size_t)(2 + 3 * L.nb)) c->d_stats.alloc(2 + 3 * L.nb, c->stream);
    ++g_launches, reduce_stats_kernel<<<dim3(ncta, L.nb), 256, 0, c->stream>>>(L.d_ll.p, L.d_last_acc.p, c->M, L.nb, c->d_partial.p);
    CK(cudaGetLastError());
    ++g_launches, finish_stats_kernel<<<1, 64, 0, c->stream>>>(c->d_partial.p, ncta, L.nb, c->d_stats.p);
    CK(cudaGetLastError());
    if (host_out) {
        CK(cudaMemcpyAsync(host_out, c->d_stats.p, sizeof(double) * (2 + 3 * L.nb), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
}

// ---- ρ per (block, chain): rho[b] of every chain, [nb][M]
std::vector<double> rho_per_chain(dmt_ctx *c, int nb, const double *rho) {
    std::vector<double> r((size_t)nb * c->M);
    for (int b = 0; b < nb; b++) std::fill(r.begin() + (size_t)b * c->M, r.begin() + (size_t)(b + 1) * c->M, rho[b]);
    return r;
}
// adaptation (re)starts from ρ: s = logit of ρ's position in (rho_min, rho_max), kept 1e-6 away from either end; nacc = 0
void restart_adaptation(dmt_ctx *c, Layout &L, const std::vector<double> &rho) {
    std::vector<double> s(rho.size());
    for (size_t i = 0; i < rho.size(); i++) {
        const double u = std::min(std::max((rho[i] - L.ad_rho_min) / (L.ad_rho_max - L.ad_rho_min), 1e-6), 1.0 - 1e-6);
        s[i] = std::log(u / (1.0 - u));
    }
    CK(cudaMemcpyAsync(L.d_ad_s.p, s.data(), sizeof(double) * s.size(), cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(L.d_ad_nacc.p, 0, sizeof(int32_t) * L.d_ad_nacc.n, c->stream));
    CK(cudaStreamSynchronize(c->stream));
}
void upload_rho(dmt_ctx *c, Layout &L, const std::vector<double> &rho) {
    CK(cudaMemcpyAsync(L.d_rho.p, rho.data(), sizeof(double) * rho.size(), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (L.adapt) restart_adaptation(c, L, rho);
}

// NVTX range around a C-ABI operation (nsys / ncu --nvtx): off unless DMT_NVTX=1, so the hot loop pays one predictable branch
struct NvtxRange {
    bool on;
    explicit NvtxRange(const char *name) {
        static int enabled = -1;
        if (enabled < 0) { const char *e = getenv("DMT_NVTX"); enabled = (e && e[0] == '1') ? 1 : 0; }
        on = enabled == 1;
        if (on) nvtxRangePushA(name);
    }
    ~NvtxRange() { if (on) nvtxRangePop(); }
};
#define DMT_RANGE(name) NvtxRange nvtx_range_(name)

template <class F> int32_t guarded(dmt_ctx *ctx, F &&f) {
    if (!ctx) return DMT_ERR_ARG;
    try {
        CK(cudaSetDevice(ctx->cfg.device));
        f();
        return DMT_OK;
    } catch (const DmtError &e) {
        ctx->err = e.what();
        return e.code;
    } catch (const std::exception &e) {
        ctx->err = e.what();
        return DMT_ERR_STATE;
    }
}

} // namespace

// =============================================================================================================== API
extern "C" {

int32_t dmt_version(void) { return 200; }

int32_t dmt_launch_count(uint64_t *n) {
    if (!n) return DMT_ERR_ARG;
    *n = g_launches;
    return DMT_OK;
}

int32_t dmt_model_dims(int32_t model, int32_t *d, int32_t *dw, int32_t *npar, int32_t *constdiff) {
    ModelDims md;
    if (!model_dims(model, md)) return DMT_ERR_ARG;
    if (d) *d = md.D;
    if (dw) *dw = md.DW;
    if (npar) *npar = md.NPAR;
    if (constdiff) *constdiff = md.constdiff ? 1 : 0;
    return DMT_OK;
}

const char *dmt_last_error(const dmt_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int32_t dmt_create(const dmt_config *cfg, const int32_t *n_pts, const double *tt, const int32_t *pset_of_chain, dmt_ctx **out) {
    if (!cfg || !n_pts || !tt || !out) { g_create_error = "null argument"; return DMT_ERR_ARG; }
    dmt_ctx *c = nullptr;
    try {
        c = new dmt_ctx();
        c->cfg = *cfg;
        REQUIRE(model_dims(cfg->model, c->md), DMT_ERR_ARG, "unknown model id");
        c->D = c->md.D; c->DW = c->md.DW; c->NPAR = c->md.NPAR;
        c->NH = c->D * (c->D + 1) / 2; c->NG = c->NH + c->D; c->NAUX = c->D * c->D + c->D + c->NH;
        c->K = cfg->n_intervals; c->M = cfg->n_chains; c->P = cfg->n_psets; c->m = cfg->obs_dim;
        REQUIRE(c->K >= 1 && c->M >= 1, DMT_ERR_ARG, "need n_intervals >= 1 and n_chains >= 1");
        REQUIRE(c->P >= 1 && c->P <= c->M, DMT_ERR_ARG, "need 1 <= n_psets <= n_chains");
        REQUIRE(c->m >= 1 && c->m <= c->D, DMT_ERR_ARG, "need 1 <= obs_dim <= d");
        REQUIRE(cfg->n_layouts >= 1 && cfg->n_layouts <= 64, DMT_ERR_ARG, "need 1 <= n_layouts <= 64");
        REQUIRE(cfg->artificial_noise > 0.0, DMT_ERR_ARG, "artificial_noise must be > 0");
        c->NOBS = c->m * c->D + c->m * c->m + c->m;
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        REQUIRE(e == cudaSuccess && ndev > 0, DMT_ERR_CUDA, "no CUDA device: libdmt has no CPU fallback");
        REQUIRE(cfg->device >= 0 && cfg->device < ndev, DMT_ERR_ARG, "device ordinal out of range");
        CK(cudaSetDevice(cfg->device));
        CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        // every lane streams whole 32-byte sectors that it alone owns (kernels.cuh): ask L2 not to promote DRAM fetches to
        // 64/128 B, which only drags in sectors of the other accepted/proposal buffer
        cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, 32);

        // ---- time grid -> tiles
        const int K = c->K;
        c->nsteps.resize(K); c->tile0.resize(K + 1); c->step0.resize(K + 1); c->pt0.resize(K + 1);
        c->tile0[0] = c->step0[0] = c->pt0[0] = 0;
        for (int k = 0; k < K; k++) {
            REQUIRE(n_pts[k] >= 2, DMT_ERR_ARG, "every interval needs >= 2 grid points");
            c->nsteps[k] = n_pts[k] - 1;
            c->tile0[k + 1] = c->tile0[k] + (c->nsteps[k] + 3) / 4;
            c->step0[k + 1] = c->step0[k] + c->nsteps[k];
            c->pt0[k + 1] = c->pt0[k] + n_pts[k];
        }
        c->NT = c->tile0[K]; c->S = c->step0[K]; c->NP = c->pt0[K];
        std::vector<double> dt((size_t)c->NT * 4, 0.0), sq((size_t)c->NT * 4, 0.0);
        for (int k = 0; k < K; k++)
            for (int j = 0; j < c->nsteps[k]; j++) {
                const double h = tt[c->pt0[k] + j + 1] - tt[c->pt0[k] + j];
                REQUIRE(h > 0.0, DMT_ERR_ARG, "time grid must be strictly increasing inside an interval");
                dt[(size_t)c->tile0[k] * 4 + j] = h;
                sq[(size_t)c->tile0[k] * 4 + j] = std::sqrt(h);
            }
        c->ppb_tile0.assign(K, -1);
        c->pset.resize(c->M);
        for (int i = 0; i < c->M; i++) {
            c->pset[i] = pset_of_chain ? pset_of_chain[i] : (c->P == c->M ? i : 0);
            REQUIRE(c->pset[i] >= 0 && c->pset[i] < c->P, DMT_ERR_ARG, "pset_of_chain entry out of range");
            REQUIRE(pset_of_chain || c->P == c->M || c->P == 1, DMT_ERR_ARG, "pset_of_chain required when 1 < P < M");
        }
        {
            bool ident = (c->P == c->M);
            for (int i = 0; i < c->M && ident; i++) ident = (c->pset[i] == i);
            c->pipe_ok = ident;
        }
        c->d_tile0.upload(c->tile0, c->stream); c->d_step0.upload(c->step0, c->stream); c->d_pt0.upload(c->pt0, c->stream);
        c->d_nsteps.upload(c->nsteps, c->stream); c->d_ppb_tile0.upload(c->ppb_tile0, c->stream); c->d_pset.upload(c->pset, c->stream);
        c->d_dt.upload(dt, c->stream); c->d_sqdt.upload(sq, c->stream);

        // ---- SoA containers (SamplingPair: accepted + proposal buffers)
        const size_t M = c->M, P = c->P, NT = c->NT;
        const size_t xb = NT * c->D * M * 4, wb = NT * c->DW * M * 4, x0b = (size_t)K * c->D * M;
        c->d_X.alloc(2 * xb, c->stream); c->d_W.alloc(2 * wb, c->stream); c->d_X0.alloc(2 * x0b, c->stream);
        c->d_parX.alloc((size_t)K * M, c->stream); c->d_parW.alloc((size_t)K * M, c->stream);
        const int nslot = cfg->two_sided_laws ? 2 : 1;
        for (int st = 0; st < 2; st++) c->d_parP[st].alloc((size_t)K * P, c->stream);
        for (int s = 0; s < nslot; s++) {
            c->d_G[s][0].alloc(NT * c->NG * P * 4, c->stream);
            c->d_G[s][1].alloc((size_t)c->NG * P * 4, c->stream);
            for (int st = 0; st < 2; st++) {
                c->d_c0[s][st].alloc((size_t)K * P, c->stream);
                c->d_theta[s][st].alloc((size_t)K * c->NPAR * P, c->stream);
                c->d_aux[s][st].alloc((size_t)K * c->NAUX * P, c->stream);
            }
            c->d_obs[s].alloc((size_t)K * c->NOBS * P, c->stream);
            c->d_vart[s].alloc((size_t)K * c->D * P, c->stream);
        }
        DevCtx &d = c->dev;
        d.M = c->M; d.P = c->P; d.K = K; d.NT = c->NT; d.NTb = 0; d.m = c->m; d.two_sided = cfg->two_sided_laws ? 1 : 0;
        d.tile0 = c->d_tile0.p; d.step0 = c->d_step0.p; d.pt0 = c->d_pt0.p; d.nsteps = c->d_nsteps.p; d.ppb_tile0 = c->d_ppb_tile0.p;
        d.dt = c->d_dt.p; d.sqdt = c->d_sqdt.p; d.pset = c->d_pset.p;
        {
            std::vector<int> kt(c->NT, 0);
            for (int k = 0; k < K; k++)
                for (int t = c->tile0[k]; t < c->tile0[k + 1]; t++) kt[t] = k;
            c->d_k_of_tile.upload(kt, c->stream);
            d.k_of_tile = c->d_k_of_tile.p;
        }
        d.X = c->d_X.p; d.W = c->d_W.p; d.X0 = c->d_X0.p; d.Xbuf = xb; d.Wbuf = wb; d.X0buf = x0b;
        d.parX = c->d_parX.p; d.parW = c->d_parW.p;
        for (int st = 0; st < 2; st++) d.parP[st] = c->d_parP[st].p;
        for (int s = 0; s < 2; s++) {
            for (int st = 0; st < 2; st++) {
                d.G[s][st] = c->d_G[s][st].p; d.c0[s][st] = c->d_c0[s][st].p;
                d.theta[s][st] = c->d_theta[s][st].p; d.aux[s][st] = c->d_aux[s][st].p;
            }
            d.obs[s] = c->d_obs[s].p; d.vart[s] = c->d_vart[s].p;
        }
        d.eps = cfg->artificial_noise; d.seed = cfg->seed; d.chain_offset = (uint32_t)cfg->chain_offset;
        c->layouts.resize(cfg->n_layouts);
        CK(cudaStreamSynchronize(c->stream));
        *out = c;
        return DMT_OK;
    } catch (const DmtError &e) {
        g_create_error = e.what();
        delete c;
        return e.code;
    } catch (const std::exception &e) {
        g_create_error = e.what();
        delete c;
        return DMT_ERR_STATE;
    }
}

int32_t dmt_destroy(dmt_ctx *ctx) {
    if (!ctx) return DMT_OK;
    cudaSetDevice(ctx->cfg.device);
    if (ctx->nccl_comm && g_nccl.CommDestroy) g_nccl.CommDestroy(ctx->nccl_comm);
    if (ctx->p2p_ready)
        for (int r = 0; r < ctx->p2p.world; r++)
            if (r != ctx->p2p.rank && ctx->p2p.peer[r]) cudaIpcCloseMemHandle(ctx->p2p.peer[r]);
    if (ctx->p2p_local) cudaFree(ctx->p2p_local);
    if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
    if (ctx->ev_gathered) cudaEventDestroy(ctx->ev_gathered);
    if (ctx->ev_copied) cudaEventDestroy(ctx->ev_copied);
    if (ctx->ev_hist) cudaEventDestroy(ctx->ev_hist);
    if (ctx->stream) { cudaStreamSynchronize(ctx->stream); cudaStreamDestroy(ctx->stream); }
    delete ctx;
    return DMT_OK;
}

int32_t dmt_sync(dmt_ctx *ctx) {
    return guarded(ctx, [&] { CK(cudaStreamSynchronize(ctx->stream)); });
}
int32_t dmt_get_stream(dmt_ctx *ctx, void **s) {
    return guarded(ctx, [&] { REQUIRE(s, DMT_ERR_ARG, "null"); *s = (void *)ctx->stream; });
}


// ---------------------------------------------------------------------------------------------------------------- laws
int32_t dmt_set_params(dmt_ctx *ctx, int32_t side, int32_t store_mask, int32_t k0, int32_t k1, const double *theta) {
    return guarded(ctx, [&] {
        check_law_side(ctx, side); check_range(ctx, k0, k1);
        if (side == 0) { ensure_W(ctx); invalidate_caches(ctx); } // the accepted laws change: cached guiding terms are stale
        REQUIRE(theta && (store_mask & 3), DMT_ERR_ARG, "null theta or empty store mask");
        for (int st = 0; st < 2; st++)
            if ((store_mask >> st) & 1)
                put_record(ctx, side, st, ctx->d_theta[0][st].p, ctx->d_theta[1][st].p, ctx->NPAR, 0, ctx->NPAR, k0, k1, theta, true);
    });
}

int32_t dmt_set_aux(dmt_ctx *ctx, int32_t side, int32_t store, int32_t k0, int32_t k1, const double *B, const double *beta, const double *atil) {
    return guarded(ctx, [&] {
        check_law_side(ctx, side); check_range(ctx, k0, k1);
        if (side == 0) { ensure_W(ctx); invalidate_caches(ctx); } // the accepted laws change: cached guiding terms are stale
        REQUIRE(store == 0 || store == 1, DMT_ERR_ARG, "store must be 0 (PP) or 1 (PPb)");
        REQUIRE(B && beta && atil, DMT_ERR_ARG, "null aux array");
        ctx->aux_all_linearised = false; // a host-evaluated B may be dense: the backward filter stops skipping the Jacobian's structural zeros
        const int D = ctx->D, NH = ctx->NH, nk = k1 - k0 + 1;
        const size_t P = ctx->P;
        double *r0 = ctx->d_aux[0][store].p, *r1 = ctx->d_aux[1][store].p;
        put_record(ctx, side, store, r0, r1, ctx->NAUX, 0, D * D, k0, k1, B, false);
        put_record(ctx, side, store, r0, r1, ctx->NAUX, D * D, D, k0, k1, beta, false);
        std::vector<double> packed((size_t)nk * NH * P); // symmetric part of atilde, packed upper
        for (int k = 0; k < nk; k++)
            for (int i = 0; i < D; i++)
                for (int j = i; j < D; j++) {
                    const int si = i * D - i * (i - 1) / 2 + (j - i);
                    for (size_t p = 0; p < P; p++)
                        packed[((size_t)k * NH + si) * P + p] =
                            0.5 * (atil[((size_t)k * D * D + i * D + j) * P + p] + atil[((size_t)k * D * D + j * D + i) * P + p]);
                }
        put_record(ctx, side, store, r0, r1, ctx->NAUX, D * D + D, NH, k0, k1, packed.data(), false);
    });
}

int32_t dmt_set_aux_linearised(dmt_ctx *ctx, int32_t side, int32_t store, int32_t k0, int32_t k1, const double *xbar) {
    return guarded(ctx, [&] {
        check_law_side(ctx, side); check_range(ctx, k0, k1);
        if (side == 0) { ensure_W(ctx); invalidate_caches(ctx); } // the accepted laws change: cached guiding terms are stale
        REQUIRE(store == 0 || store == 1, DMT_ERR_ARG, "store must be 0 (PP) or 1 (PPb)");
        const size_t per_k = (size_t)ctx->D * ctx->P, n = (size_t)(k1 - k0 + 1) * per_k;
        if (ctx->d_xbar[store].n < (size_t)ctx->K * per_k) { ctx->d_xbar[store].alloc((size_t)ctx->K * per_k, ctx->stream); ctx->xbar_set[store].assign(ctx->K, 0); }
        double *tmp = ctx->d_xbar[store].p + (size_t)k0 * per_k;
        if (xbar) { // new linearisation points: keep them on the device
            CK(cudaMemcpyAsync(tmp, xbar, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            for (int k = k0; k <= k1; k++) ctx->xbar_set[store][k] = 1;
        } else {    // NULL: re-linearise at the points of the last call (only theta changed)
            for (int k = k0; k <= k1; k++) REQUIRE(ctx->xbar_set[store][k], DMT_ERR_STATE, "no linearisation points stored for this interval yet");
        }
        dim3 grid = pset_grid(ctx, k1 - k0 + 1, 128);
#define DMT_CASE(MID)                                                                                              \
    case MID: ++g_launches, aux_linearise_kernel<Model<MID>><<<grid, 128, 0, ctx->stream>>>(ctx->dev, side, store, k0, k1, tmp); break;
        switch (ctx->cfg.model) {
            DMT_FOR_MODELS(DMT_CASE)
        default: throw DmtError(DMT_ERR_UNSUPPORTED, "model not compiled into this build of libdmt");
        }
#undef DMT_CASE
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(ctx->stream));
    });
}

int32_t dmt_set_obs(dmt_ctx *ctx, int32_t side, int32_t k0, int32_t k1, const double *L, const double *Sigma, const double *v) {
    return guarded(ctx, [&] {
        check_law_side(ctx, side); check_range(ctx, k0, k1);
        if (side == 0) { ensure_W(ctx); invalidate_caches(ctx); } // the accepted laws change: cached guiding terms are stale
        REQUIRE(L && Sigma && v, DMT_ERR_ARG, "null observation array");
        const int m = ctx->m, D = ctx->D;
        double *r0 = ctx->d_obs[0].p, *r1 = ctx->d_obs[1].p;
        put_record(ctx, side, 0, r0, r1, ctx->NOBS, 0, m * D, k0, k1, L, false);
        put_record(ctx, side, 0, r0, r1, ctx->NOBS, m * D, m * m, k0, k1, Sigma, false);
        put_record(ctx, side, 0, r0, r1, ctx->NOBS, m * D + m * m, m, k0, k1, v, false);
    });
}

int32_t dmt_equalize_laws(dmt_ctx *ctx, int32_t store_mask, int32_t k0, int32_t k1, int32_t *changed) {
    return guarded(ctx, [&] {
        check_law_side(ctx, 1); check_range(ctx, k0, k1);
        dim3 grid = pset_grid(ctx, k1 - k0 + 1, 128);
        if (ctx->d_flag.n < 1) ctx->d_flag.alloc(1, ctx->stream);
        CK(cudaMemsetAsync(ctx->d_flag.p, 0, sizeof(int), ctx->stream));
        for (int st = 0; st < 2; st++) {
            if (!((store_mask >> st) & 1)) continue;
            ++g_launches, copy_record_kernel<<<grid, 128, 0, ctx->stream>>>(ctx->dev, st, ctx->d_theta[0][st].p, ctx->d_theta[1][st].p, ctx->NPAR, k0, k1, ctx->d_flag.p);
            ++g_launches, copy_record_kernel<<<grid, 128, 0, ctx->stream>>>(ctx->dev, st, ctx->d_aux[0][st].p, ctx->d_aux[1][st].p, ctx->NAUX, k0, k1, ctx->d_flag.p);
            if (st == 0) ++g_launches, copy_record_kernel<<<grid, 128, 0, ctx->stream>>>(ctx->dev, 0, ctx->d_obs[0].p, ctx->d_obs[1].p, ctx->NOBS, k0, k1, ctx->d_flag.p);
        }
        CK(cudaGetLastError());
        if (changed) { // b° had to be changed: its guiding term belongs to other parameters => the caller escalates critical_change
            int h = 0;
            CK(cudaMemcpyAsync(&h, ctx->d_flag.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            *changed = h;
        }
    });
}

// ---------------------------------------------------------------------------------------------------------------- layouts
int32_t dmt_set_blocks(dmt_ctx *ctx, int32_t layout, int32_t n_blocks, const int32_t *i0, const int32_t *i1, const double *rho,
                       const uint8_t *last, int32_t ll_hist_len) {
    return guarded(ctx, [&] {
        REQUIRE(layout >= 0 && layout < (int)ctx->layouts.size(), DMT_ERR_ARG, "layout index out of range");
        REQUIRE(n_blocks >= 1 && n_blocks <= 64 && i0 && i1 && rho, DMT_ERR_ARG, "need 1 <= n_blocks <= 64 and non-null ranges/rho");
        Layout &L = ctx->layouts[layout];
        std::vector<uint8_t> lst(n_blocks);
        for (int b = 0; b < n_blocks; b++) {
            lst[b] = last ? (last[b] ? 1 : 0) : (b == n_blocks - 1 ? 1 : 0); // BlockCollection: i == N (src/block_collection.jl:29)
            REQUIRE(0 <= i0[b] && i0[b] <= i1[b] && i1[b] < ctx->K, DMT_ERR_ARG, "block range out of bounds");
            // a non-terminal block needs >= 2 intervals: the reference indexes b.PP[1] and XX[end-1] (src/block.jl:164,177)
            REQUIRE(lst[b] || i1[b] > i0[b], DMT_ERR_ARG, "a non-terminal block must span at least 2 intervals");
            REQUIRE(lst[b] || ctx->P == ctx->M, DMT_ERR_UNSUPPORTED,
                    "blocking freezes a per-recording artificial observation: needs n_psets == n_chains");
            REQUIRE(std::abs(rho[b]) <= 1.0, DMT_ERR_ARG, "rho must be in [-1, 1]");
        }
        const size_t M = ctx->M;
        L.nb = n_blocks;
        L.i0.assign(i0, i0 + n_blocks); L.i1.assign(i1, i1 + n_blocks); L.last = lst;
        L.d_i0.upload(L.i0, ctx->stream); L.d_i1.upload(L.i1, ctx->stream); L.d_last.upload(L.last, ctx->stream);
        L.d_rho.upload(rho_per_chain(ctx, n_blocks, rho), ctx->stream);
        L.d_ll.upload(std::vector<double>(2 * n_blocks * M, -INFINITY), ctx->stream); // Block ctor: ll = -Inf (src/block.jl:74)
        L.d_ok.alloc(n_blocks * M, ctx->stream); L.d_last_acc.alloc(n_blocks * M, ctx->stream);
        L.adapt = false;
        L.d_ad_s.release(); L.d_ad_nacc.release();
        const int hl_req = ll_hist_len >= 0 ? ll_hist_len : ctx->cfg.ll_hist_len;
        const size_t hl = hl_req > 0 ? hl_req : 0;
        if (hl) { L.d_acc_hist.alloc(hl * n_blocks * M, ctx->stream); L.d_ll_hist.alloc(hl * 2 * n_blocks * M, ctx->stream); }
        L.dev.nb = n_blocks; L.dev.id = layout;
        L.dev.i0 = L.d_i0.p; L.dev.i1 = L.d_i1.p; L.dev.last = L.d_last.p; L.dev.rho = L.d_rho.p;
        L.dev.ll = L.d_ll.p; L.dev.ok = L.d_ok.p; L.dev.last_acc = L.d_last_acc.p;
        L.dev.acc_hist = hl ? L.d_acc_hist.p : nullptr; L.dev.ll_hist = hl ? L.d_ll_hist.p : nullptr; L.dev.hist_len = (int)hl;
        {   // the pipelined sweep's task entries (PipeSched): (block b, its interval j) as b + 64 j, every block's first interval first
            std::vector<int> task;
            for (int j = 0;; j++) {
                const size_t n0 = task.size();
                for (int b = 0; b < n_blocks; b++)
                    if (i0[b] + j <= i1[b]) task.push_back(b + 64 * j);
                if (task.size() == n0) break;
            }
            L.d_task.upload(task, ctx->stream);
        }
        L.set = true;
        L.cache_enabled = false; L.cache_valid = false;
        cache_set_private(L, false);
        rebuild_ppb_store(ctx);
        CK(cudaStreamSynchronize(ctx->stream));
    });
}

int32_t dmt_set_rho(dmt_ctx *ctx, int32_t layout, const double *rho) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(rho, DMT_ERR_ARG, "null rho");
        for (int b = 0; b < L.nb; b++) REQUIRE(std::abs(rho[b]) <= 1.0, DMT_ERR_ARG, "rho must be in [-1, 1]");
        upload_rho(ctx, L, rho_per_chain(ctx, L.nb, rho));
    });
}
int32_t dmt_set_rho_chains(dmt_ctx *ctx, int32_t layout, const double *rho) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(rho, DMT_ERR_ARG, "null rho");
        const size_t n = (size_t)L.nb * ctx->M;
        for (size_t i = 0; i < n; i++) REQUIRE(std::abs(rho[i]) <= 1.0, DMT_ERR_ARG, "rho must be in [-1, 1]");
        upload_rho(ctx, L, std::vector<double>(rho, rho + n));
    });
}
int32_t dmt_get_rho_chains(dmt_ctx *ctx, int32_t layout, double *out) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(out, DMT_ERR_ARG, "null");
        CK(cudaMemcpyAsync(out, L.d_rho.p, sizeof(double) * L.d_rho.n, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}
int32_t dmt_set_rho_adaptation(dmt_ctx *ctx, int32_t layout, double target, double gamma0, double decay, int32_t window, double rho_min,
                               double rho_max) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        if (!(target > 0.0)) { // (NaN included: nothing to adapt toward)
            REQUIRE(!std::isnan(target), DMT_ERR_ARG, "target is NaN");
            L.adapt = false;
            L.d_ad_s.release(); L.d_ad_nacc.release();
            return;
        }
        REQUIRE(target < 1.0 && gamma0 > 0.0 && std::isfinite(gamma0) && decay > 0.5 && decay <= 1.0 && window >= 1, DMT_ERR_ARG,
                "need 0 < target < 1, gamma0 > 0, 0.5 < decay <= 1 and window >= 1");
        REQUIRE(rho_min >= 0.0 && rho_min < rho_max && rho_max <= 1.0, DMT_ERR_ARG, "need 0 <= rho_min < rho_max <= 1");
        L.ad_target = target; L.ad_gamma0 = gamma0; L.ad_decay = decay; L.ad_window = window;
        L.ad_rho_min = rho_min; L.ad_rho_max = rho_max;
        const size_t n = (size_t)L.nb * ctx->M;
        if (L.d_ad_s.n != n) { L.d_ad_s.alloc_uninit(n); L.d_ad_nacc.alloc_uninit(n); }
        std::vector<double> rho(n);
        CK(cudaMemcpyAsync(rho.data(), L.d_rho.p, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        L.adapt = true;
        L.ad_calls = 0;
        restart_adaptation(ctx, L, rho);
    });
}
int32_t dmt_adapt_rho(dmt_ctx *ctx, int32_t layout) {
    DMT_RANGE("dmt_adapt_rho");
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(L.adapt, DMT_ERR_ARG, "rho adaptation is off for this layout (dmt_set_rho_adaptation)");
        const uint64_t calls = L.ad_calls + 1;
        const bool update = calls % (uint64_t)L.ad_window == 0;
        const double gamma = update ? L.ad_gamma0 * std::pow((double)(calls / (uint64_t)L.ad_window), -L.ad_decay) : 0.0;
        const int n = L.nb * ctx->M;
        ++g_launches, adapt_rho_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(L.d_rho.p, L.d_ad_s.p, L.d_ad_nacc.p, L.d_last_acc.p, n,
                                                                              L.ad_window, update ? 1 : 0, gamma, L.ad_target,
                                                                              L.ad_rho_min, L.ad_rho_max);
        CK(cudaGetLastError());
        L.ad_calls = calls;
    });
}
int32_t dmt_get_rho_adaptation_state(dmt_ctx *ctx, int32_t layout, double *s, int32_t *nacc, uint64_t *calls) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(L.adapt, DMT_ERR_STATE, "rho adaptation is off for this layout (dmt_set_rho_adaptation)");
        REQUIRE(s && nacc && calls, DMT_ERR_ARG, "null output");
        CK(cudaMemcpyAsync(s, L.d_ad_s.p, sizeof(double) * L.d_ad_s.n, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(nacc, L.d_ad_nacc.p, sizeof(int32_t) * L.d_ad_nacc.n, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        *calls = L.ad_calls;
    });
}
int32_t dmt_set_rho_adaptation_state(dmt_ctx *ctx, int32_t layout, const double *s, const int32_t *nacc, uint64_t calls) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(L.adapt, DMT_ERR_STATE, "rho adaptation is off for this layout (dmt_set_rho_adaptation)");
        REQUIRE(s && nacc, DMT_ERR_ARG, "null input");
        const size_t n = (size_t)L.nb * ctx->M;
        for (size_t i = 0; i < n; i++) {
            REQUIRE(std::isfinite(s[i]), DMT_ERR_ARG, "s must be finite");
            REQUIRE(nacc[i] >= 0 && nacc[i] < L.ad_window, DMT_ERR_ARG, "need 0 <= nacc < window");
        }
        CK(cudaMemcpyAsync(L.d_ad_s.p, s, sizeof(double) * n, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(L.d_ad_nacc.p, nacc, sizeof(int32_t) * n, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        L.ad_calls = calls;
    });
}

// ---------------------------------------------------------------------------------------------------------------- paths
int32_t dmt_set_start(dmt_ctx *ctx, const double *x0) {
    return guarded(ctx, [&] {
        REQUIRE(x0, DMT_ERR_ARG, "null x0");
        const size_t n = (size_t)ctx->D * ctx->M;
        for (int s = 0; s < 2; s++) // interval 0 is the head of both X0 buffers
            CK(cudaMemcpyAsync(ctx->d_X0.p + s * ctx->dev.X0buf, x0, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}

static void xfer_paths(dmt_ctx *ctx, int side, double *host, bool is_x, bool upload) {
    check_side(ctx, side);
    REQUIRE(host, DMT_ERR_ARG, "null host array");
    if (!is_x) { // lazy noise: reading W materialises it first; overwriting the accepted noise makes it current
        if (upload && side == 0) ctx->W_stale_layout = -1;
        else ensure_W(ctx);
    }
    const size_t n = is_x ? (size_t)ctx->NP * ctx->D * ctx->M : (size_t)ctx->S * ctx->DW * ctx->M;
    DevBuf<double> nat;
    nat.alloc_uninit(n);
    if (upload) CK(cudaMemcpyAsync(nat.p, host, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    dim3 grid = chain_grid(ctx, ctx->K, 128);
    if (is_x) ++g_launches, xfer_X_kernel<<<grid, 128, 0, ctx->stream>>>(ctx->dev, side, ctx->D, nat.p, upload ? 1 : 0);
    else ++g_launches, xfer_W_kernel<<<grid, 128, 0, ctx->stream>>>(ctx->dev, side, ctx->DW, nat.p, upload ? 1 : 0);
    CK(cudaGetLastError());
    if (!upload) CK(cudaMemcpyAsync(host, nat.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
}
int32_t dmt_set_X(dmt_ctx *ctx, int32_t side, const double *X) { return guarded(ctx, [&] { xfer_paths(ctx, side, (double *)X, true, true); }); }
int32_t dmt_get_X(dmt_ctx *ctx, int32_t side, double *X) { return guarded(ctx, [&] { xfer_paths(ctx, side, X, true, false); }); }
int32_t dmt_set_W(dmt_ctx *ctx, int32_t side, const double *W) { return guarded(ctx, [&] { xfer_paths(ctx, side, (double *)W, false, true); }); }
int32_t dmt_get_W(dmt_ctx *ctx, int32_t side, double *W) { return guarded(ctx, [&] { xfer_paths(ctx, side, W, false, false); }); }

// the stream of the asynchronous read-backs and its events, created on first use
static void ensure_copy_stream(dmt_ctx *ctx) {
    if (ctx->copy_stream) return;
    CK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ctx->ev_gathered, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->ev_copied, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->ev_hist, cudaEventDisableTiming));
    CK(cudaEventRecord(ctx->ev_copied, ctx->copy_stream));
}

int32_t dmt_snapshot_paths_async(dmt_ctx *ctx, int32_t side, int32_t n_sel, const int32_t *chains, double *host_out) {
    return guarded(ctx, [&] {
        check_side(ctx, side);
        REQUIRE(n_sel >= 1 && chains && host_out, DMT_ERR_ARG, "bad snapshot arguments");
        for (int i = 0; i < n_sel; i++) REQUIRE(chains[i] >= 0 && chains[i] < ctx->M, DMT_ERR_ARG, "chain index out of range");
        ensure_copy_stream(ctx);
        const size_t n = (size_t)ctx->NP * ctx->D * n_sel;
        // the staging buffer is reused: the gather may not start before the previous snapshot has left the device
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_copied, 0));
        if (ctx->d_snap.n < n) { CK(cudaStreamSynchronize(ctx->copy_stream)); ctx->d_snap.alloc_uninit(n); }
        if (ctx->d_snap_sel.n < (size_t)n_sel) { CK(cudaStreamSynchronize(ctx->copy_stream)); ctx->d_snap_sel.alloc_uninit(n_sel); }
        CK(cudaMemcpyAsync(ctx->d_snap_sel.p, chains, sizeof(int) * n_sel, cudaMemcpyHostToDevice, ctx->stream));
        ++g_launches, gather_X_kernel<<<dim3((n_sel + 63) / 64, ctx->K), 64, 0, ctx->stream>>>(ctx->dev, side, ctx->D, ctx->d_snap_sel.p, n_sel, ctx->d_snap.p);
        CK(cudaGetLastError());
        CK(cudaEventRecord(ctx->ev_gathered, ctx->stream));
        // the copy runs on its own stream: the compute stream goes on with the next sweep while the paths travel
        CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_gathered, 0));
        CK(cudaMemcpyAsync(host_out, ctx->d_snap.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->copy_stream));
        CK(cudaEventRecord(ctx->ev_copied, ctx->copy_stream));
    });
}
// bb.b.XX / bb.b.WW of a few recordings (the reference reads them per recording: be.recordings[i].blocks[j].b.XX)
static void get_paths_of(dmt_ctx *ctx, int side, int n_sel, const int32_t *chains, double *out, bool is_x) {
    check_side(ctx, side);
    if (!is_x) ensure_W(ctx);
    REQUIRE(n_sel >= 1 && chains && out, DMT_ERR_ARG, "bad chain selection");
    for (int i = 0; i < n_sel; i++) REQUIRE(chains[i] >= 0 && chains[i] < ctx->M, DMT_ERR_ARG, "chain index out of range");
    const size_t n = (is_x ? (size_t)ctx->NP * ctx->D : (size_t)ctx->S * ctx->DW) * n_sel;
    DevBuf<double> d;
    DevBuf<int> sel;
    d.alloc_uninit(n);
    sel.alloc_uninit(n_sel);
    CK(cudaMemcpyAsync(sel.p, chains, sizeof(int) * n_sel, cudaMemcpyHostToDevice, ctx->stream));
    const dim3 grid((n_sel + 63) / 64, ctx->K);
    if (is_x) ++g_launches, gather_X_kernel<<<grid, 64, 0, ctx->stream>>>(ctx->dev, side, ctx->D, sel.p, n_sel, d.p);
    else ++g_launches, gather_W_kernel<<<grid, 64, 0, ctx->stream>>>(ctx->dev, side, ctx->DW, sel.p, n_sel, d.p);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
}
int32_t dmt_get_X_chains(dmt_ctx *ctx, int32_t side, int32_t n_sel, const int32_t *chains, double *X) {
    return guarded(ctx, [&] { get_paths_of(ctx, side, n_sel, chains, X, true); });
}
int32_t dmt_get_W_chains(dmt_ctx *ctx, int32_t side, int32_t n_sel, const int32_t *chains, double *W) {
    return guarded(ctx, [&] { get_paths_of(ctx, side, n_sel, chains, W, false); });
}
// ll_history / accpt_history (src/block.jl:57-58, src/biblock.jl:47) rows it0..it1 to the host without stalling the sampler: the copy
// waits (on the copy stream) for everything queued so far on the compute stream, which goes on with the next sweeps
int32_t dmt_histories_async(dmt_ctx *ctx, int32_t layout, uint32_t it0, uint32_t it1, double *host_ll, uint8_t *host_acc) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE((host_ll || host_acc) && it0 <= it1 && it1 < (uint32_t)L.dev.hist_len, DMT_ERR_ARG, "bad history range");
        ensure_copy_stream(ctx);
        const size_t per = (size_t)L.nb * ctx->M, n = (size_t)(it1 - it0 + 1);
        CK(cudaEventRecord(ctx->ev_hist, ctx->stream));
        CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_hist, 0));
        if (host_ll) // rows are [2][n_blocks][M] (accepted, proposal), contiguous over iterations
            CK(cudaMemcpyAsync(host_ll, L.d_ll_hist.p + (size_t)it0 * 2 * per, n * 2 * per * sizeof(double), cudaMemcpyDeviceToHost, ctx->copy_stream));
        if (host_acc)
            CK(cudaMemcpyAsync(host_acc, L.d_acc_hist.p + (size_t)it0 * per, n * per, cudaMemcpyDeviceToHost, ctx->copy_stream));
    });
}
int32_t dmt_snapshot_wait(dmt_ctx *ctx) {
    return guarded(ctx, [&] {
        if (ctx->copy_stream) CK(cudaStreamSynchronize(ctx->copy_stream));
    });
}

int32_t dmt_init_paths(dmt_ctx *ctx, int32_t layout, uint32_t iter0, int32_t max_tries, int32_t *n_failed) {
    DMT_RANGE("dmt_init_paths");
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(L.nb == 1 && L.last[0] && L.i0[0] == 0 && L.i1[0] == ctx->K - 1, DMT_ERR_ARG,
                "init_paths needs a layout made of one terminal block over all intervals");
        REQUIRE(max_tries >= 1, DMT_ERR_ARG, "max_tries must be >= 1");
        CK(cudaMemsetAsync(L.d_ok.p, 0, L.d_ok.n, ctx->stream));
        std::vector<uint8_t> ok(L.d_ok.n);
        int bad = 0;
        for (int t = 0; t < max_tries; t++) { // while true: forward_guide!(...) && return   (src/sampling_unit.jl:84-86)
            FwdArgs fa{iter0 + (uint32_t)t, 0, 0, 0, nullptr};
            launch_fwd<OP_INIT>(ctx, L, fa);
            CK(cudaMemcpyAsync(ok.data(), L.d_ok.p, ok.size(), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            bad = 0;
            for (uint8_t o : ok) bad += !o;
            if (!bad) break;
        }
        ++g_launches, copy_acc_to_prop_kernel<<<chain_grid(ctx, ctx->K, 128), 128, 0, ctx->stream>>>(ctx->dev, ctx->D, ctx->DW);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(ctx->stream));
        if (n_failed) *n_failed = bad;
    });
}

// ---------------------------------------------------------------------------------------------------------------- hot path
int32_t dmt_set_artificial_obs(dmt_ctx *ctx, int32_t layout) {
    DMT_RANGE("dmt_set_artificial_obs");
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        ++g_launches, set_artificial_obs_kernel<<<chain_grid(ctx, L.nb, 128), 128, 0, ctx->stream>>>(ctx->dev, L.dev, ctx->D);
        CK(cudaGetLastError());
    });
}

int32_t dmt_recompute_guiding_term(dmt_ctx *ctx, int32_t layout, int32_t which) {
    DMT_RANGE("dmt_recompute_guiding_term");
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(which >= 1 && which <= 3, DMT_ERR_ARG, "which must be DMT_P_ONLY, DMT_PO_ONLY or DMT_P_BOTH");
        if (which & 2) check_law_side(ctx, 1);
        if (L.cache_enabled && (which & 1)) { // accepted laws through the guiding cache: build once, then F = F0 + Psi v
            if (!L.cache_valid) cache_build(ctx, L);
            else cache_apply(ctx, L);
            if (which & 2) launch_bwd(ctx, L, DMT_PO_ONLY);
        } else {
            launch_bwd(ctx, L, which);
        }
    });
}

int32_t dmt_find_W_for_X(dmt_ctx *ctx, int32_t layout) {
    return guarded(ctx, [&] { launch_fwd<OP_INVSOLVE>(ctx, layout_of(ctx, layout), FwdArgs{0, 0, 0, 0, nullptr}); });
}
int32_t dmt_loglikhd(dmt_ctx *ctx, int32_t layout, int32_t side, int32_t skip) {
    DMT_RANGE("dmt_loglikhd");
    return guarded(ctx, [&] {
        check_law_side(ctx, side);
        REQUIRE(skip >= 0, DMT_ERR_ARG, "skip must be >= 0");
        launch_fwd<OP_LOGLIK>(ctx, layout_of(ctx, layout), FwdArgs{0, side, 0, skip, nullptr});
    });
}
int32_t dmt_find_W_and_loglikhd(dmt_ctx *ctx, int32_t layout) {
    return guarded(ctx, [&] { launch_fwd<OP_INVSOLVE_LL>(ctx, layout_of(ctx, layout), FwdArgs{0, 0, 0, 0, nullptr}); });
}

int32_t dmt_draw_proposal_path(dmt_ctx *ctx, int32_t layout, uint32_t iter, const double *Z) {
    DMT_RANGE("dmt_draw_proposal_path");
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        FwdArgs fa{iter, 0, 0, 0, nullptr};
        if (Z) {
            const size_t n = (size_t)ctx->S * ctx->DW * ctx->M;
            double *tmp = ctx->scratch(n);
            CK(cudaMemcpyAsync(tmp, Z, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            fa.Z = tmp;
        }
        launch_fwd<OP_DRAW>(ctx, L, fa);
        if (Z) CK(cudaStreamSynchronize(ctx->stream));
    });
}

int32_t dmt_find_W_loglikhd_draw(dmt_ctx *ctx, int32_t layout, uint32_t iter, const double *Z) {
    DMT_RANGE("dmt_find_W_loglikhd_draw");
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        FwdArgs fa{iter, 0, 0, 0, nullptr};
        if (Z) {
            const size_t n = (size_t)ctx->S * ctx->DW * ctx->M;
            double *tmp = ctx->scratch(n);
            CK(cudaMemcpyAsync(tmp, Z, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            fa.Z = tmp;
        }
        launch_fwd<OP_SWEEP>(ctx, L, fa);
        if (Z) CK(cudaStreamSynchronize(ctx->stream));
    });
}

int32_t dmt_blocking_sweep(dmt_ctx *ctx, int32_t layout, uint32_t iter) {
    DMT_RANGE("dmt_blocking_sweep");
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        ++g_launches, set_artificial_obs_kernel<<<chain_grid(ctx, L.nb, 128), 128, 0, ctx->stream>>>(ctx->dev, L.dev, ctx->D); // GP.set_obs!(be)
        CK(cudaGetLastError());
        if (L.cache_enabled) {                       // recompute_guiding_term!(be, Val(:P_only)) through the guiding cache
            if (!L.cache_valid) cache_build(ctx, L);
            else cache_apply(ctx, L);
        } else {
            launch_bwd(ctx, L, DMT_P_ONLY);
        }
        launch_fwd<OP_SWEEP>(ctx, L, FwdArgs{iter, 0, 0, 0, nullptr}); // find_W_for_X!; loglikhd!; draw_proposal_path!
    });
}

int32_t dmt_recompute_path(dmt_ctx *ctx, int32_t layout, int32_t law_side, int32_t noise_side, int32_t skip) {
    DMT_RANGE("dmt_recompute_path");
    return guarded(ctx, [&] {
        check_law_side(ctx, law_side); check_side(ctx, noise_side);
        REQUIRE(skip >= 0, DMT_ERR_ARG, "skip must be >= 0");
        launch_fwd<OP_RECOMPUTE>(ctx, layout_of(ctx, layout), FwdArgs{0, law_side, noise_side, skip, nullptr});
    });
}

int32_t dmt_set_proposal_law(dmt_ctx *ctx, int32_t layout, int32_t critical_change, int32_t skip) {
    DMT_RANGE("dmt_set_proposal_law");
    return guarded(ctx, [&] {
        check_law_side(ctx, 1);
        Layout &L = layout_of(ctx, layout);
        if (critical_change) launch_bwd(ctx, L, DMT_PO_ONLY);                           // src/biblock.jl:342
        launch_fwd<OP_RECOMPUTE>(ctx, L, FwdArgs{0, 1, 0, skip, nullptr});              // src/biblock.jl:343
    });
}

int32_t dmt_accept_reject_path(dmt_ctx *ctx, int32_t layout, uint32_t iter, const double *E) {
    DMT_RANGE("dmt_accept_reject_path");
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        const double *dE = nullptr;
        if (E) {
            const size_t n = (size_t)L.nb * ctx->M;
            double *tmp = ctx->scratch(n);
            CK(cudaMemcpyAsync(tmp, E, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            dE = tmp;
        }
        ++g_launches, accept_kernel<<<chain_grid(ctx, L.nb, 128), 128, 0, ctx->stream>>>(ctx->dev, L.dev, iter, dE);
        CK(cudaGetLastError());
        if (E) CK(cudaStreamSynchronize(ctx->stream));
    });
}

static void swap_impl(dmt_ctx *ctx, int32_t layout, int32_t what, const uint8_t *mask, bool per_block) {
    Layout &L = layout_of(ctx, layout);
    REQUIRE(what > 0 && what < 16, DMT_ERR_ARG, "empty or unknown swap mask");
    if (what & (DMT_SWAP_WW | DMT_SWAP_PP)) ensure_W(ctx); // (lazy noise) the noise about to change sides / laws must exist
    const uint8_t *dm = nullptr;
    if (mask) {
        REQUIRE(!(what & DMT_SWAP_PP) || ctx->P == ctx->M, DMT_ERR_UNSUPPORTED, "masked swap_PP! needs n_psets == n_chains");
        const size_t n = (size_t)ctx->M * (per_block ? L.nb : 1);
        if (ctx->d_mask.n < n) ctx->d_mask.alloc(n, ctx->stream);
        CK(cudaMemcpyAsync(ctx->d_mask.p, mask, n, cudaMemcpyHostToDevice, ctx->stream));
        dm = ctx->d_mask.p;
    }
    if (what & (DMT_SWAP_XX | DMT_SWAP_WW | DMT_SWAP_LL))
        ++g_launches, swap_paths_kernel<<<chain_grid(ctx, L.nb, 128), 128, 0, ctx->stream>>>(ctx->dev, L.dev, what, dm, per_block ? 1 : 0);
    if (what & DMT_SWAP_PP) {
        check_law_side(ctx, 1);
        invalidate_caches(ctx); // the accepted laws are now the former proposals (their guiding term is in the shared store)
        if (mask) ctx->parP_mixed = true;
        ++g_launches, swap_laws_kernel<<<pset_grid(ctx, L.nb, 128), 128, 0, ctx->stream>>>(ctx->dev, L.dev, dm, per_block ? 1 : 0);
    }
    CK(cudaGetLastError());
    if (mask) CK(cudaStreamSynchronize(ctx->stream));
}
int32_t dmt_swap(dmt_ctx *ctx, int32_t layout, int32_t what, const uint8_t *chain_mask) {
    return guarded(ctx, [&] { swap_impl(ctx, layout, what, chain_mask, false); });
}
int32_t dmt_swap_blocks(dmt_ctx *ctx, int32_t layout, int32_t what, const uint8_t *block_chain_mask) {
    return guarded(ctx, [&] {
        if (!block_chain_mask) throw DmtError(DMT_ERR_ARG, "dmt_swap_blocks needs a [n_blocks][n_chains] mask (dmt_swap swaps everything)");
        swap_impl(ctx, layout, what, block_chain_mask, true);
    });
}

int32_t dmt_save_ll(dmt_ctx *ctx, int32_t layout, uint32_t iter) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(L.dev.hist_len > 0 && iter < (uint32_t)L.dev.hist_len, DMT_ERR_ARG, "iteration beyond ll_hist_len");
        ++g_launches, save_ll_kernel<<<chain_grid(ctx, L.nb, 128), 128, 0, ctx->stream>>>(ctx->dev, L.dev, iter);
        CK(cudaGetLastError());
    });
}

// ---------------------------------------------------------------------------------------------------------------- read-back
int32_t dmt_fetch_ll(dmt_ctx *ctx, int32_t layout, int32_t side, double *total, double *per_block) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        check_side(ctx, side);
        std::vector<double> out(2 + 3 * L.nb);
        fill_stats(ctx, L, out.data());
        if (total) *total = out[side];
        if (per_block)
            for (int b = 0; b < L.nb; b++) per_block[b] = out[2 + (1 + side) * L.nb + b];
    });
}

int32_t dmt_get_ll(dmt_ctx *ctx, int32_t layout, int32_t side, double *ll) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        check_side(ctx, side); REQUIRE(ll, DMT_ERR_ARG, "null");
        const size_t n = (size_t)L.nb * ctx->M;
        CK(cudaMemcpyAsync(ll, L.d_ll.p + side * n, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}
int32_t dmt_set_ll(dmt_ctx *ctx, int32_t layout, int32_t side, const double *ll) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        check_side(ctx, side); REQUIRE(ll, DMT_ERR_ARG, "null");
        const size_t n = (size_t)L.nb * ctx->M;
        CK(cudaMemcpyAsync(L.d_ll.p + side * n, ll, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}
int32_t dmt_get_success(dmt_ctx *ctx, int32_t layout, uint8_t *ok) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(ok, DMT_ERR_ARG, "null");
        CK(cudaMemcpyAsync(ok, L.d_ok.p, (size_t)L.nb * ctx->M, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}
int32_t dmt_get_last_accept(dmt_ctx *ctx, int32_t layout, uint8_t *acc) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(acc, DMT_ERR_ARG, "null");
        CK(cudaMemcpyAsync(acc, L.d_last_acc.p, (size_t)L.nb * ctx->M, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}
int32_t dmt_get_accept_history(dmt_ctx *ctx, int32_t layout, uint32_t it0, uint32_t it1, uint8_t *acc) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(acc && it0 <= it1 && it1 < (uint32_t)L.dev.hist_len, DMT_ERR_ARG, "bad history range");
        const size_t per = (size_t)L.nb * ctx->M;
        CK(cudaMemcpyAsync(acc, L.d_acc_hist.p + it0 * per, (size_t)(it1 - it0 + 1) * per, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}
int32_t dmt_get_ll_history(dmt_ctx *ctx, int32_t layout, int32_t side, uint32_t it0, uint32_t it1, double *ll) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        check_side(ctx, side);
        REQUIRE(ll && it0 <= it1 && it1 < (uint32_t)L.dev.hist_len, DMT_ERR_ARG, "bad history range");
        const size_t per = (size_t)L.nb * ctx->M;
        for (uint32_t it = it0; it <= it1; ++it)
            CK(cudaMemcpyAsync(ll + (size_t)(it - it0) * per, L.d_ll_hist.p + ((size_t)it * 2 + side) * per, per * sizeof(double),
                               cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}
int32_t dmt_set_accepted(dmt_ctx *ctx, int32_t layout, uint32_t iter, const uint8_t *acc) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(acc && iter < (uint32_t)L.dev.hist_len, DMT_ERR_ARG, "bad history index");
        const size_t per = (size_t)L.nb * ctx->M;
        CK(cudaMemcpyAsync(L.d_acc_hist.p + iter * per, acc, per, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}
int32_t dmt_set_ll_history(dmt_ctx *ctx, int32_t layout, int32_t side, uint32_t iter, const double *ll) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        check_side(ctx, side);
        REQUIRE(ll && iter < (uint32_t)L.dev.hist_len, DMT_ERR_ARG, "bad history index");
        const size_t per = (size_t)L.nb * ctx->M;
        CK(cudaMemcpyAsync(L.d_ll_hist.p + ((size_t)iter * 2 + side) * per, ll, per * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}
int32_t dmt_accept_counts(dmt_ctx *ctx, int32_t layout, uint32_t it0, uint32_t it1, int64_t *counts) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(counts && it0 <= it1 && it1 < (uint32_t)L.dev.hist_len, DMT_ERR_ARG, "bad history range");
        DevBuf<unsigned long long> d;
        d.alloc(L.nb, ctx->stream);
        ++g_launches, accept_counts_kernel<<<chain_grid(ctx, L.nb, 128), 128, 0, ctx->stream>>>(L.d_acc_hist.p, L.nb, ctx->M, it0, it1, d.p);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(counts, d.p, sizeof(int64_t) * L.nb, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}

// ---------------------------------------------------------------------------------------------------------------- guiding term
static void xfer_guiding(dmt_ctx *ctx, int side, int store, int k, double *H, double *F, double *c, bool upload, Layout *priv = nullptr) {
    check_law_side(ctx, side); check_range(ctx, k, k);
    if (upload && side == 0) { ensure_W(ctx); invalidate_caches(ctx); }
    REQUIRE(store == 0 || store == 1, DMT_ERR_ARG, "store must be 0 (PP) or 1 (PPb)");
    REQUIRE(store == 0 || ctx->ppb_tile0[k] >= 0, DMT_ERR_STATE, "interval has no blocking law in any registered layout");
    REQUIRE(H && F && c, DMT_ERR_ARG, "null");
    const size_t n = ctx->nsteps[k] + 1, P = ctx->P, D = ctx->D;
    DevBuf<double> dH, dF, dc;
    dH.alloc_uninit(n * D * D * P); dF.alloc_uninit(n * D * P); dc.alloc_uninit(n * P);
    if (upload) {
        CK(cudaMemcpyAsync(dH.p, H, dH.n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(dF.p, F, dF.n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(dc.p, c, dc.n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (priv) ensure_guiding(ctx, *priv);
    double *Gpriv = (priv && priv->cache_valid && side == 0) ? priv->d_Gl[store].p : nullptr;
    double *cpriv = Gpriv ? priv->d_c0l[store].p : nullptr;
    ++g_launches, xfer_guiding_kernel<<<pset_grid(ctx, 1, 128), 128, 0, ctx->stream>>>(ctx->dev, side, store, k, ctx->D, dH.p, dF.p, dc.p, upload ? 1 : 0, Gpriv, cpriv);
    CK(cudaGetLastError());
    if (!upload) {
        CK(cudaMemcpyAsync(H, dH.p, dH.n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(F, dF.p, dF.n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(c, dc.p, dc.n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    if (!upload && Gpriv) { // the cache refreshes c only where it is read: at the first interval of each block, accepted PP store
        bool block_start = false;
        for (int b = 0; b < priv->nb; b++) block_start = block_start || (priv->i0[b] == k && store == 0);
        if (!block_start)
            for (size_t p = 0; p < P; p++) c[p] = NAN;
    }
}
int32_t dmt_get_guiding_term(dmt_ctx *ctx, int32_t side, int32_t store, int32_t k, double *H, double *F, double *c) {
    return guarded(ctx, [&] { xfer_guiding(ctx, side, store, k, H, F, c, false); });
}
int32_t dmt_upload_guiding_term(dmt_ctx *ctx, int32_t side, int32_t store, int32_t k, const double *H, const double *F, const double *c) {
    return guarded(ctx, [&] { xfer_guiding(ctx, side, store, k, (double *)H, (double *)F, (double *)c, true); });
}
int32_t dmt_get_layout_guiding_term(dmt_ctx *ctx, int32_t layout, int32_t store, int32_t k, double *H, double *F, double *c) {
    return guarded(ctx, [&] { xfer_guiding(ctx, 0, store, k, H, F, c, false, &layout_of(ctx, layout)); });
}
int32_t dmt_set_fwd_lanes(dmt_ctx *ctx, int32_t lanes) {
    return guarded(ctx, [&] {
        if (lanes != 0 && lanes != 1 && lanes != 2 && lanes != 4 && lanes != 8) throw DmtError(DMT_ERR_ARG, "lanes must be 0 (auto), 1, 2, 4 or 8");
        ctx->fwd_lanes = lanes;
    });
}
int32_t dmt_get_last_forward_kernel(dmt_ctx *ctx, char *buf, int32_t len) {
    return guarded(ctx, [&] {
        if (!buf || len <= 0) throw DmtError(DMT_ERR_ARG, "need a buffer");
        snprintf(buf, (size_t)len, "%s", ctx->last_fwd_kernel);
    });
}
int32_t dmt_set_sweep_mode(dmt_ctx *ctx, int32_t mode) {
    return guarded(ctx, [&] {
        if (mode < 0 || mode > 5 || mode == 4) throw DmtError(DMT_ERR_ARG, "mode must be 0 (auto), 1 (register-tile kernel), 2 (software-pipelined kernel), 3 (warp-specialised kernel) or 5 (step-parallel kernel)");
        ctx->sweep_mode = mode;
    });
}
int32_t dmt_set_lazy_noise(dmt_ctx *ctx, int32_t enable) {
    return guarded(ctx, [&] {
        if (!enable) ensure_W(ctx);
        ctx->lazy_W = enable != 0;
    });
}
int32_t dmt_set_bwd_solver(dmt_ctx *ctx, int32_t solver, double reltol, double abstol) {
    return guarded(ctx, [&] {
        if (solver != DMT_K1_RK4 && solver != DMT_K1_TSIT5) throw DmtError(DMT_ERR_ARG, "solver must be DMT_K1_RK4 or DMT_K1_TSIT5");
        if (solver == DMT_K1_TSIT5) {
            if (!(reltol > 0.0) || !(abstol >= 0.0)) throw DmtError(DMT_ERR_ARG, "need reltol > 0 and abstol >= 0");
            for (auto &L : ctx->layouts)
                if (L.set && L.cache_enabled) throw DmtError(DMT_ERR_STATE, "switch the guiding cache off first: it needs the RK4 backward filter");
            ctx->bwd_reltol = reltol; ctx->bwd_abstol = abstol;
        }
        ensure_W(ctx);
        invalidate_caches(ctx);
        ctx->bwd_solver = solver;
    });
}
int32_t dmt_get_bwd_steps(dmt_ctx *ctx, int32_t *accepted, int32_t *rejected) {
    return guarded(ctx, [&] {
        int h[2] = {0, 0};
        if (ctx->d_steps.n >= 2) {
            CK(cudaMemcpyAsync(h, ctx->d_steps.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
        }
        if (accepted) *accepted = h[0];
        if (rejected) *rejected = h[1];
    });
}
int32_t dmt_set_bwd_mode(dmt_ctx *ctx, int32_t mode) {
    return guarded(ctx, [&] {
        if (mode < 0 || mode > 2) throw DmtError(DMT_ERR_ARG, "mode must be 0 (auto), 1 (thread per parameter set) or 2 (cooperative)");
        ctx->bwd_mode = mode;
    });
}
int32_t dmt_enable_guiding_cache(dmt_ctx *ctx, int32_t layout, int32_t enable) {
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(!enable || ctx->bwd_solver == 0, DMT_ERR_STATE, "the guiding cache needs the RK4 backward filter (dmt_set_bwd_solver)");
        L.cache_enabled = enable != 0;
        L.cache_valid = false;
        cache_set_private(L, false);
        if (!enable) {
            for (int st = 0; st < 2; st++) { L.d_Gl[st].release(); L.d_FP[st].release(); L.d_c0l[st].release(); }
            L.d_cq.release(); L.d_vlast.release();
        }
    });
}

// ---------------------------------------------------------------------------------------------------------------- test hooks
int32_t dmt_debug_normals(dmt_ctx *ctx, uint32_t chain0, uint32_t tile0, uint32_t iter, uint32_t layout, int32_t n_chains, int32_t n_tiles, double *out) {
    return guarded(ctx, [&] {
        REQUIRE(out && n_chains > 0 && n_tiles > 0, DMT_ERR_ARG, "bad arguments");
        const size_t n = (size_t)n_chains * n_tiles * 4 * ctx->DW;
        DevBuf<double> d;
        d.alloc_uninit(n);
        const int tot = n_chains * n_tiles;
        dim3 grid((tot + 127) / 128);
        switch (ctx->DW) {
        case 1: ++g_launches, debug_normals_kernel<1><<<grid, 128, 0, ctx->stream>>>(ctx->cfg.seed, chain0, tile0, iter, layout, n_chains, n_tiles, d.p); break;
        case 2: ++g_launches, debug_normals_kernel<2><<<grid, 128, 0, ctx->stream>>>(ctx->cfg.seed, chain0, tile0, iter, layout, n_chains, n_tiles, d.p); break;
        case 3: ++g_launches, debug_normals_kernel<3><<<grid, 128, 0, ctx->stream>>>(ctx->cfg.seed, chain0, tile0, iter, layout, n_chains, n_tiles, d.p); break;
        default: ++g_launches, debug_normals_kernel<4><<<grid, 128, 0, ctx->stream>>>(ctx->cfg.seed, chain0, tile0, iter, layout, n_chains, n_tiles, d.p); break;
        }
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(out, d.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}
int32_t dmt_debug_exponentials(dmt_ctx *ctx, uint32_t chain0, uint32_t iter, uint32_t layout, int32_t n_chains, int32_t n_blocks, double *out) {
    return guarded(ctx, [&] {
        REQUIRE(out && n_chains > 0 && n_blocks > 0, DMT_ERR_ARG, "bad arguments");
        const int tot = n_chains * n_blocks;
        DevBuf<double> d;
        d.alloc_uninit(tot);
        ++g_launches, debug_exponentials_kernel<<<(tot + 127) / 128, 128, 0, ctx->stream>>>(ctx->cfg.seed, chain0, iter, layout, n_chains, n_blocks, d.p);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(out, d.p, tot * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}

// ---------------------------------------------------------------------------------------------------------------- multi-GPU
int32_t dmt_nccl_unique_id(uint8_t *id128) {
    try {
        REQUIRE(id128, DMT_ERR_ARG, "null");
        load_nccl();
        NCK(g_nccl.GetUniqueId(id128));
        return DMT_OK;
    } catch (const DmtError &e) {
        g_create_error = e.what();
        return e.code;
    }
}
int32_t dmt_comm_init(dmt_ctx *ctx, int32_t n_ranks, int32_t rank, const uint8_t *id128) {
    return guarded(ctx, [&] {
        REQUIRE(id128 && n_ranks >= 1 && rank >= 0 && rank < n_ranks, DMT_ERR_ARG, "bad communicator arguments");
        load_nccl();
        UidByValue uid;
        memcpy(uid.internal, id128, 128);
        NCK(g_nccl.CommInitRank(&ctx->nccl_comm, n_ranks, uid, rank));
        ctx->n_ranks = n_ranks;
    });
}
int32_t dmt_p2p_export(dmt_ctx *ctx, uint8_t *handle64) {
    return guarded(ctx, [&] {
        REQUIRE(handle64, DMT_ERR_ARG, "null");
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
        if (!ctx->p2p_local) {
            CK(cudaMalloc(&ctx->p2p_local, sizeof(P2PBuf)));
            CK(cudaMemsetAsync(ctx->p2p_local, 0, sizeof(P2PBuf), ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
        }
        cudaIpcMemHandle_t h;
        CK(cudaIpcGetMemHandle(&h, ctx->p2p_local));
        memcpy(handle64, &h, 64);
    });
}
int32_t dmt_p2p_init(dmt_ctx *ctx, int32_t n_ranks, int32_t rank, const uint8_t *handles) {
    return guarded(ctx, [&] {
        REQUIRE(handles && n_ranks >= 1 && n_ranks <= P2P_MAX_RANKS && rank >= 0 && rank < n_ranks, DMT_ERR_ARG, "bad peer arguments");
        REQUIRE(ctx->p2p_local, DMT_ERR_STATE, "dmt_p2p_export first");
        ctx->p2p = P2PArgs{};
        for (int r = 0; r < n_ranks; r++) {
            if (r == rank) { ctx->p2p.peer[r] = ctx->p2p_local; continue; }
            cudaIpcMemHandle_t h;
            memcpy(&h, handles + (size_t)r * 64, 64);
            void *p = nullptr;
            CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
            ctx->p2p.peer[r] = (P2PBuf *)p;
        }
        ctx->p2p.rank = rank;
        ctx->p2p.world = n_ranks;
        ctx->p2p.seq = 0;
        ctx->n_ranks = n_ranks;
        ctx->p2p_ready = true;
    });
}
int32_t dmt_p2p_disable(dmt_ctx *ctx) {
    return guarded(ctx, [&] { ctx->p2p_ready = false; });
}
int32_t dmt_allreduce_stats(dmt_ctx *ctx, int32_t layout, double *out) {
    DMT_RANGE("dmt_allreduce_stats");
    return guarded(ctx, [&] {
        Layout &L = layout_of(ctx, layout);
        REQUIRE(out, DMT_ERR_ARG, "null");
        fill_stats(ctx, L, nullptr);
        if (ctx->p2p_ready && 2 + L.nb <= P2P_MAX_VALS) { // own one-shot all-reduce over NVLink peer memory (kernels.cuh)
            ctx->p2p.seq++;
            ctx->p2p.nval = 2 + L.nb;
            ++g_launches, p2p_allreduce_kernel<<<1, P2P_MAX_VALS, 0, ctx->stream>>>(ctx->p2p, ctx->d_stats.p);
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(out, ctx->d_stats.p, sizeof(double) * (2 + L.nb), cudaMemcpyDeviceToHost, ctx->stream));
            int err = 0;
            CK(cudaMemcpyAsync(&err, &ctx->p2p_local->error, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            if (err) throw DmtError(DMT_ERR_NCCL, "peer all-reduce timed out: a rank did not arrive within 20 s");
            return;
        }
        if (ctx->nccl_comm) // ONE small allreduce: [sum ll, sum ll°, accept counts per block]  (SURVEY §8e, C1)
            NCK(g_nccl.AllReduce(ctx->d_stats.p, ctx->d_stats.p, (size_t)(2 + L.nb), 8 /* ncclDouble */, 0 /* ncclSum */, ctx->nccl_comm, ctx->stream));
        CK(cudaMemcpyAsync(out, ctx->d_stats.p, sizeof(double) * (2 + L.nb), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}

} // extern "C"

// ------------------------------------------------------------------------------------------------ posterior path moments
namespace {
size_t pm_tile_len(dmt_ctx *c) { return (size_t)c->NT * c->D * c->M * 4; }
size_t pm_len(dmt_ctx *c) { return pm_tile_len(c) + (size_t)c->K * c->D * c->M; }
void pm_alloc(dmt_ctx *c) {
    if (c->d_pm_mean.p) return;
    const size_t n = pm_len(c);
    for (DevBuf<double> *b : {&c->d_pm_mean, &c->d_pm_m2}) {
        if (cudaMalloc(&b->p, n * sizeof(double)) != cudaSuccess) {
            cudaGetLastError();
            c->d_pm_mean.release(); c->d_pm_m2.release();
            throw DmtError(DMT_ERR_CUDA, "path moments: cannot allocate 2 x " + std::to_string(n * sizeof(double)) + " bytes of device memory");
        }
        b->n = n;
    }
}
// accumulators <-> natural [NP][d][n] (sel == null: chains 0..n-1)
void pm_xfer(dmt_ctx *c, double *A, int n, const int32_t *chains, double *host, bool upload) {
    const size_t len = (size_t)c->NP * c->D * n;
    DevBuf<double> nat;
    DevBuf<int> sel;
    nat.alloc_uninit(len);
    if (chains) {
        sel.alloc_uninit(n);
        CK(cudaMemcpyAsync(sel.p, chains, sizeof(int) * n, cudaMemcpyHostToDevice, c->stream));
    }
    if (upload) CK(cudaMemcpyAsync(nat.p, host, len * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    ++g_launches, moments_xfer_kernel<<<dim3((n + 63) / 64, c->K), 64, 0, c->stream>>>(c->dev, c->D, A, A + pm_tile_len(c), sel.p, n, nat.p,
                                                                                       upload ? 1 : 0);
    CK(cudaGetLastError());
    if (!upload) CK(cudaMemcpyAsync(host, nat.p, len * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
}
template <int D> void launch_path_moments(dmt_ctx *c, double w, int first) {
    const dim3 grid((unsigned)((c->M + 127) / 128), (unsigned)std::min(c->NT + c->K, 65535), 1);
    double *mu = c->d_pm_mean.p, *m2 = c->d_pm_m2.p;
    const size_t t = pm_tile_len(c);
    ++g_launches, path_moments_kernel<D><<<grid, 128, 0, c->stream>>>(c->dev, mu, m2, mu + t, m2 + t, w, first);
}
} // namespace

extern "C" {

int32_t dmt_path_moments_add(dmt_ctx *ctx) {
    DMT_RANGE("dmt_path_moments_add");
    return guarded(ctx, [&] {
        pm_alloc(ctx);
        const uint64_t n = ctx->pm_count + 1;
        const double w = 1.0 / (double)n;
        const int first = n == 1 ? 1 : 0;
        switch (ctx->D) { // reads X only: under lazy noise W stays as it is
        case 2: launch_path_moments<2>(ctx, w, first); break;
        case 3: launch_path_moments<3>(ctx, w, first); break;
        case 4: launch_path_moments<4>(ctx, w, first); break;
        case 6: launch_path_moments<6>(ctx, w, first); break;
        default: throw DmtError(DMT_ERR_UNSUPPORTED, "path moments: no kernel for this state dimension");
        }
        CK(cudaGetLastError());
        ctx->pm_count = n;
    });
}
int32_t dmt_path_moments_reset(dmt_ctx *ctx) {
    return guarded(ctx, [&] { ctx->pm_count = 0; });
}
int32_t dmt_get_path_moments(dmt_ctx *ctx, int32_t n_sel, const int32_t *chains, double *mean, double *m2, uint64_t *count) {
    return guarded(ctx, [&] {
        REQUIRE(mean && m2 && count, DMT_ERR_ARG, "null output array");
        REQUIRE(ctx->pm_count > 0, DMT_ERR_STATE, "no path moments accumulated (dmt_path_moments_add)");
        if (chains) {
            REQUIRE(n_sel >= 1, DMT_ERR_ARG, "bad chain selection");
            for (int i = 0; i < n_sel; i++) REQUIRE(chains[i] >= 0 && chains[i] < ctx->M, DMT_ERR_ARG, "chain index out of range");
        } else {
            n_sel = ctx->M;
        }
        pm_xfer(ctx, ctx->d_pm_mean.p, n_sel, chains, mean, false);
        pm_xfer(ctx, ctx->d_pm_m2.p, n_sel, chains, m2, false);
        *count = ctx->pm_count;
    });
}
int32_t dmt_set_path_moments(dmt_ctx *ctx, const double *mean, const double *m2, uint64_t count) {
    return guarded(ctx, [&] {
        REQUIRE(mean && m2, DMT_ERR_ARG, "null input array");
        REQUIRE(count > 0, DMT_ERR_ARG, "count must be >= 1 (dmt_path_moments_reset clears the moments)");
        pm_alloc(ctx);
        pm_xfer(ctx, ctx->d_pm_mean.p, ctx->M, nullptr, (double *)mean, true);
        pm_xfer(ctx, ctx->d_pm_m2.p, ctx->M, nullptr, (double *)m2, true);
        ctx->pm_count = count;
    });
}
int32_t dmt_get_pset_path_moments(dmt_ctx *ctx, double *mean, double *var, double *rhat) {
    return guarded(ctx, [&] {
        REQUIRE(mean && var && rhat, DMT_ERR_ARG, "null output array");
        REQUIRE(ctx->pm_count > 0, DMT_ERR_STATE, "no path moments accumulated (dmt_path_moments_add)");
        const int M = ctx->M, P = ctx->P;
        if (!ctx->d_pm_cs.p) { // chains of every pset in ascending order
            std::vector<int> cs(P + 1, 0), list(M);
            for (int c = 0; c < M; c++) cs[ctx->pset[c] + 1]++;
            for (int q = 0; q < P; q++) cs[q + 1] += cs[q];
            std::vector<int> fill(cs.begin(), cs.end() - 1);
            for (int c = 0; c < M; c++) list[fill[ctx->pset[c]]++] = c;
            ctx->d_pm_cs.upload(cs, ctx->stream);
            ctx->d_pm_chains.upload(list, ctx->stream);
        }
        const size_t len = (size_t)ctx->NP * ctx->D * P, t = pm_tile_len(ctx);
        DevBuf<double> out;
        out.alloc_uninit(3 * len);
        int nk_max = 0;
        for (int k = 0; k < ctx->K; k++) nk_max = std::max(nk_max, ctx->nsteps[k] + 1);
        const size_t per_k = (size_t)nk_max * ctx->D * P;
        const double *mu = ctx->d_pm_mean.p, *m2 = ctx->d_pm_m2.p;
        ++g_launches, pset_moments_kernel<<<dim3((unsigned)((per_k + 127) / 128), ctx->K), 128, 0, ctx->stream>>>(
            ctx->dev, ctx->D, mu, m2, mu + t, m2 + t, ctx->d_pm_cs.p, ctx->d_pm_chains.p, (double)ctx->pm_count, out.p, out.p + len, out.p + 2 * len);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(mean, out.p, len * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(var, out.p + len, len * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(rhat, out.p + 2 * len, len * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    });
}

} // extern "C"
