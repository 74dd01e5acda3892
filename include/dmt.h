/*
 * dmt.h — C ABI of libdmt.so: the B200-native guided-proposal path update behind the
 * SamplingUnit / SamplingPair / SamplingEnsemble / Block / BiBlock / BlockCollection / BlockEnsemble API of
 * DiffusionMCMCTools.jl.  File:line citations are into /root/reference/.
 *
 * One dmt_ctx == one SamplingEnsemble (src/sampling_ensemble.jl:17-41) resident on ONE GPU: M chains
 * ("recordings"), each a SamplingPair (accepted u / proposal u°, src/sampling_pair.jl:36-38) over K observation
 * intervals, plus any number of block layouts (each layout == what a BlockEnsemble holds: one BlockCollection per
 * recording with identical ranges, src/block_ensemble.jl:20-33, src/block_collection.jl:20-30).
 * A Block is an index range (i0,i1,last) instead of six Julia views (src/block.jl:66-72).
 *
 * Conventions
 *   - every function returns int32 status (DMT_OK == 0); no C++ exception crosses the boundary; dmt_last_error()
 *     gives the message.  A numerical path failure is NOT an error: the chain's success flag is 0 and its ll is -Inf
 *     (mirrors src/block.jl:163,181 and src/biblock.jl:81-82).
 *   - all pointers are caller-owned HOST pointers, copied during the call, never retained (Julia-GC safe).  The one
 *     exception are the output buffers of dmt_snapshot_paths_async / dmt_histories_async, which the library writes until dmt_snapshot_wait returns
 *     (keep it alive and unmoved until then: GC.@preserve / page-locked memory).
 *   - bulk host arrays are structure-of-arrays with the chain (or parameter-set) index FASTEST:
 *       X[point][dim][chain], W[step][dw][chain], theta[par][pset], B[k][row*d+col][pset], ...
 *     "point" runs over the concatenated per-interval grids (interval k has n_k points; boundary points are stored
 *     twice, like XX[k].x[end] and XX[k+1].x[1] in the reference); "step" over the concatenated n_k-1 steps.
 *     W holds Wiener INCREMENTS.
 *   - side: 0 = accepted (u, b), 1 = proposal (u°, b°).  store: 0 = PP, 1 = PPb (blocking laws,
 *     src/sampling_unit.jl:49-50,61-66).  Intervals are 0-based, ranges inclusive.
 *   - there is no CPU fallback: without a CUDA device every entry point fails with DMT_ERR_CUDA.
 *   - a ctx is single-owner, not thread-safe (the reference is single-threaded); ops enqueue on the ctx stream and
 *     calls returning host data synchronise.
 */
#ifndef DMT_H
#define DMT_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

enum { DMT_OK = 0, DMT_ERR_ARG = 1, DMT_ERR_CUDA = 2, DMT_ERR_STATE = 3, DMT_ERR_UNSUPPORTED = 4, DMT_ERR_NCCL = 5 };

/* models (SURVEY.md Appendix B); parameter order in the comments */
enum {
    DMT_FITZHUGH_NAGUMO = 0, /* d=2 dw=1 (eps, s, gamma, beta, sigma)                     docs/src/tutorials/preamble.md:27-28,77 */
    DMT_LOTKA_VOLTERRA = 1,  /* d=2 dw=2 (alpha, beta, gamma, delta, sigma1, sigma2)      */
    DMT_LORENZ = 2,          /* d=3 dw=3 (theta1, theta2, theta3, sigma)                  */
    DMT_PROKARYOTE = 3,      /* d=4 dw=4 (c1..c8, K)  state-dependent diffusion           */
    DMT_JANSEN_RIT = 4,      /* d=6 dw=1 (A, a, B, b, C, nu_max, v0, r, mu, sigma_y)      */
    DMT_OU2 = 5              /* d=2 dw=2 (B11,B12,B21,B22, beta1,beta2, sigma1,sigma2) linear test model */
};

enum { DMT_ACCEPTED = 0, DMT_PROPOSAL = 1 };
enum { DMT_STORE_PP = 0, DMT_STORE_PPB = 1 };
/* which laws recompute_guiding_term! touches: Val(:P_only) / Val(:P°_only) / both (src/block_collection.jl:208-221) */
enum { DMT_P_ONLY = 1, DMT_PO_ONLY = 2, DMT_P_BOTH = 3 };
/* dmt_swap masks (src/biblock.jl:148-209) */
enum { DMT_SWAP_XX = 1, DMT_SWAP_WW = 2, DMT_SWAP_PP = 4, DMT_SWAP_LL = 8 };

typedef struct dmt_ctx dmt_ctx;

typedef struct {
    int32_t model;           /* DMT_* model id */
    int32_t n_chains;        /* M: recordings held by THIS ctx / GPU */
    int32_t n_psets;         /* P: parameter/data sets, 1 <= P <= M (P == M: every recording owns its laws, as in the reference) */
    int32_t n_intervals;     /* K */
    int32_t obs_dim;         /* m: rows of L */
    int32_t device;          /* CUDA device ordinal */
    int32_t two_sided_laws;  /* 1: also allocate the proposal laws u°.PP/u°.PPb (parameter updates, src/biblock.jl:334-344) */
    int32_t ll_hist_len;     /* length of ll_history / accpt_history (src/block.jl:58, src/biblock.jl:47); 0 = none */
    int32_t n_layouts;       /* number of block layouts that will be registered with dmt_set_blocks */
    int32_t chain_offset;    /* global index of local chain 0 (Philox counters => results independent of sharding) */
    uint64_t seed;           /* Philox4x32-10 key */
    double artificial_noise; /* src/sampling_unit.jl:57 (1e-11) */
} dmt_config;

/* ---- lifetime ------------------------------------------------------------------------------------------------- */
/* SamplingEnsemble(...) containers (src/sampling_ensemble.jl:20-40; src/sampling_unit.jl:55-74 minus init_paths!).
 * n_pts[K]: points per interval; tt[sum n_pts]: imputation grid (OBS.setup_time_grids output);
 * pset_of_chain[M] or NULL (NULL: identity if P == M, all-zero if P == 1). */
int32_t dmt_create(const dmt_config *cfg, const int32_t *n_pts, const double *tt, const int32_t *pset_of_chain, dmt_ctx **out);
int32_t dmt_destroy(dmt_ctx *ctx);
const char *dmt_last_error(const dmt_ctx *ctx); /* ctx may be NULL: message of the last failed dmt_create */
int32_t dmt_sync(dmt_ctx *ctx);
int32_t dmt_get_stream(dmt_ctx *ctx, void **cuda_stream); /* for CUDA-event timing by the caller */
int32_t dmt_model_dims(int32_t model, int32_t *d, int32_t *dw, int32_t *npar, int32_t *constdiff);
int32_t dmt_version(void);
/* number of CUDA kernels this library has launched so far in this process (bench.py's gpu_launches is a difference of two reads) */
int32_t dmt_launch_count(uint64_t *n);

/* ---- laws: parameters, auxiliary laws, observations --------------------------------------------------------- */
/* DD.set_parameters!(PP, θ°, ...) result (src/biblock.jl:366-369): theta[npar][P] written into the laws of
 * intervals k0..k1 of `store_mask` (bit0 PP, bit1 PPb) on `side`. */
int32_t dmt_set_params(dmt_ctx *ctx, int32_t side, int32_t store_mask, int32_t k0, int32_t k1, const double *theta);
/* auxiliary law coefficients, host-evaluated: B[k][d*d][P], beta[k][d][P], atil[k][d*d][P] for k = k0..k1 */
int32_t dmt_set_aux(dmt_ctx *ctx, int32_t side, int32_t store, int32_t k0, int32_t k1, const double *B, const double *beta, const double *atil);
/* auxiliary law = Jacobian linearisation of the target at xbar[k][d][P] using the law's current theta (device-evaluated).
 * The points are kept on the device per store: xbar = NULL re-linearises at the points of the last call, so a parameter
 * update (dmt_set_params, then this) uploads npar x P doubles instead of K x d x P. */
int32_t dmt_set_aux_linearised(dmt_ctx *ctx, int32_t side, int32_t store, int32_t k0, int32_t k1, const double *xbar);
/* observation at the END of interval k (LinearGsnObs): L[k][m*d][P], Sigma[k][m*m][P], v[k][m][P] */
int32_t dmt_set_obs(dmt_ctx *ctx, int32_t side, int32_t k0, int32_t k1, const double *L, const double *Sigma, const double *v);
/* GP.equalize_*: copy the law records (theta, aux, obs; NOT the guiding term) of intervals k0..k1 accepted -> proposal
 * (src/biblock.jl:384-443 expressed as "copy slots").  *changed (may be NULL) := 1 when a proposal record had to be changed,
 * the value GP.equalize_obs_params! / equalize_law_params! return: the caller then escalates critical_change
 * (src/biblock.jl:362-363), because the proposal slot's guiding term belongs to other parameters. */
int32_t dmt_equalize_laws(dmt_ctx *ctx, int32_t store_mask, int32_t k0, int32_t k1, int32_t *changed);

/* ---- block layouts (src/block_collection.jl:20-30; src/biblock.jl:49-62) ------------------------------------ */
/* last[] NULL => only block n_blocks-1 is terminal (BlockCollection rule i==N).  rho[n_blocks] in [-1, 1]: the pCN memory of
 * block b for every chain (each BiBlock owns its ρ, src/biblock.jl:46; the layout stores one per (block, chain)).
 * ll_hist_len: length of this layout's ll_history / accpt_history (src/biblock.jl:49-55); < 0 => dmt_config.ll_hist_len.
 * Re-registering a layout turns its ρ adaptation off. */
int32_t dmt_set_blocks(dmt_ctx *ctx, int32_t layout, int32_t n_blocks, const int32_t *i0, const int32_t *i1, const double *rho,
                       const uint8_t *last, int32_t ll_hist_len);
/* rho[n_blocks] for every chain: ρρ of BlockEnsemble (src/block_collection.jl:27) */
int32_t dmt_set_rho(dmt_ctx *ctx, int32_t layout, const double *rho);
/* bb.ρ of every BiBlock, one per (block, local chain): rho[n_blocks][M], every entry in [-1, 1] (src/biblock.jl:46).  On a layout
 * that adapts ρ, dmt_set_rho and dmt_set_rho_chains restart the adaptation state from the new values (s from ρ, nacc = 0). */
int32_t dmt_set_rho_chains(dmt_ctx *ctx, int32_t layout, const double *rho);
int32_t dmt_get_rho_chains(dmt_ctx *ctx, int32_t layout, double *out /* [n_blocks][M] */);
/* Adaptation of ρ toward a target acceptance rate: the tutorials tune bb.ρ by hand and watch accpt_rate (src/biblock.jl:46,232).
 * Per (block, chain), from that chain's own decisions only, so a sharded run adapts exactly like the unsharded one.
 * target <= 0: freeze ρ at its current values (adaptation off).  Otherwise 0 < target < 1, gamma0 > 0, 0.5 < decay <= 1, window >= 1,
 * 0 <= rho_min < rho_max <= 1 (else DMT_ERR_ARG), and for every (b, c): u = clamp((ρ - rho_min) / (rho_max - rho_min), 1e-6, 1 - 1e-6),
 * s = log(u / (1 - u)), nacc = 0; the layout's call counter restarts at 0. */
int32_t dmt_set_rho_adaptation(dmt_ctx *ctx, int32_t layout, double target, double gamma0, double decay, int32_t window, double rho_min,
                               double rho_max);
/* One adaptation step after accept_reject_proposal_path!(be, i) (src/biblock.jl:121-127), ONE kernel launch: calls += 1;
 * nacc += the layout's last accept decisions; when calls % window == 0, with n = calls / window and gamma = gamma0 n^-decay:
 * s += gamma (target - nacc / window), ρ = rho_min + (rho_max - rho_min) / (1 + exp(-s)), nacc = 0.  Low acceptance raises ρ
 * (smaller moves).  DMT_ERR_ARG when the layout does not adapt.  Draws made while ρ adapts are not from a fixed Markov kernel:
 * keep samples from after the adaptation is frozen. */
int32_t dmt_adapt_rho(dmt_ctx *ctx, int32_t layout);
/* checkpoint / resume of the adaptation of bb.ρ (src/biblock.jl:46): s[n_blocks][M], nacc[n_blocks][M] (0 <= nacc < window), calls.  DMT_ERR_STATE when the
 * layout does not adapt (set ρ with dmt_set_rho_chains and enable the adaptation first, then restore the state) */
int32_t dmt_get_rho_adaptation_state(dmt_ctx *ctx, int32_t layout, double *s, int32_t *nacc, uint64_t *calls);
int32_t dmt_set_rho_adaptation_state(dmt_ctx *ctx, int32_t layout, const double *s, const int32_t *nacc, uint64_t calls);

/* ---- paths ---------------------------------------------------------------------------------------------------- */
int32_t dmt_set_start(dmt_ctx *ctx, const double *x0 /* [d][M] */); /* XX[1].x[1] of u and u° */
/* Thinned path saving (the tutorials keep one path every few hundred iterations, docs/src/tutorials/biblock/smoothing.md:55):
 * the paths of the n_sel listed chains, host_out[point][dim][n_sel], as they are at this point of the call sequence.  The call
 * returns at once: a gather kernel runs in order on the context's stream, the device-to-host copy on a second stream, so the
 * next sweeps overlap the transfer (pass page-locked memory for a truly asynchronous copy).  host_out may be read after
 * dmt_snapshot_wait; a further snapshot may be queued before that (it waits for the staging buffer on the device). */
int32_t dmt_snapshot_paths_async(dmt_ctx *ctx, int32_t side, int32_t n_sel, const int32_t *chains, double *host_out);
int32_t dmt_snapshot_wait(dmt_ctx *ctx);
/* History streaming: rows it0..it1 of a layout's ll_history (host_ll[it][2][n_blocks][M]: accepted, proposal — b.ll_history and
 * b°.ll_history, src/block.jl:57-58) and accpt_history (host_acc[it][n_blocks][M], src/biblock.jl:47), either may be NULL.  Like the
 * path snapshots the call returns at once: the copies run on the second stream once everything queued before the call has finished,
 * and the sampler goes on; read the buffers after dmt_snapshot_wait (page-locked memory keeps the copy asynchronous).  Rows must not be
 * rewritten (same iteration index) before the wait.  A long run streams its histories in chunks instead of reading them at the end. */
int32_t dmt_histories_async(dmt_ctx *ctx, int32_t layout, uint32_t it0, uint32_t it1, double *host_ll, uint8_t *host_acc);
/* init_paths! (src/sampling_unit.jl:83-87): fresh-noise forward_guide! of the whole path into u, retried per chain
 * until success (at most max_tries), then u° = deepcopy(u) (src/sampling_pair.jl:51). Needs the guiding term of a
 * single-terminal-block layout `layout`.  n_failed: chains still failing. */
int32_t dmt_init_paths(dmt_ctx *ctx, int32_t layout, uint32_t iter0, int32_t max_tries, int32_t *n_failed);
int32_t dmt_set_X(dmt_ctx *ctx, int32_t side, const double *X /* [NP][d][M] */);
int32_t dmt_get_X(dmt_ctx *ctx, int32_t side, double *X);
int32_t dmt_set_W(dmt_ctx *ctx, int32_t side, const double *W /* [S][dw][M] increments */);
int32_t dmt_get_W(dmt_ctx *ctx, int32_t side, double *W);
/* the same for a few recordings only — what reading be.recordings[i].blocks[j].b.XX / .WW does in the reference
 * (src/block_ensemble.jl:17-19, src/block.jl:49-58): X[NP][d][n_sel], W[S][dw][n_sel] of the listed chains */
int32_t dmt_get_X_chains(dmt_ctx *ctx, int32_t side, int32_t n_sel, const int32_t *chains, double *X);
int32_t dmt_get_W_chains(dmt_ctx *ctx, int32_t side, int32_t n_sel, const int32_t *chains, double *W);

/* ---- posterior summaries of the paths ------------------------------------------------------------------------- */
/* The smoothing tutorials keep a copy of the accepted path every few hundred iterations (docs/src/tutorials/biblock/smoothing.md:55)
 * and summarise the copies by their mean and spread.  Here every chain carries running moments of its ACCEPTED path on the device
 * instead: Welford updates, one streaming launch over X per call, no copy of the paths.  Point axis as in dmt_get_X (concatenated
 * per-interval grids, boundary points twice).  Memory: 16 d (S + K) M bytes (mean and m2), allocated by the first update (or set),
 * freed by dmt_destroy; failing allocation is DMT_ERR_CUDA.  The update reads X only (under lazy noise W is not rebuilt).
 * The moments describe the chains THIS context holds: per-chain moments are keyed by the chain, so a sharded run has exactly the
 * unsharded per-chain moments; the pooled moments below cover this rank's chains only. */
/* accumulate the current accepted paths of all chains (the `deepcopy(bb.b.XX)` step of docs/src/tutorials/biblock/smoothing.md:55);
 * count := count + 1.  n = count: mean += (x - mean) / n, m2 += (x - mean_old)(x - mean_new), each operation rounded on its own */
int32_t dmt_path_moments_add(dmt_ctx *ctx);
/* count := 0; the buffers are kept (the next update starts afresh) — e.g. at the end of burn-in */
int32_t dmt_path_moments_reset(dmt_ctx *ctx);
/* mean[NP][d][n_sel], m2[NP][d][n_sel] (sum of squared deviations: var = m2 / count) of the listed chains (chains == NULL: all M,
 * n_sel ignored); *count = number of updates.  DMT_ERR_STATE when count == 0, DMT_ERR_ARG for a chain index out of range.
 * The posterior mean and band of every recording of docs/src/tutorials/biblock/smoothing.md:55 without copying paths. */
int32_t dmt_get_path_moments(dmt_ctx *ctx, int32_t n_sel, const int32_t *chains, double *mean, double *m2, uint64_t *count);
/* restore all M chains' moments as dmt_get_path_moments(chains = NULL) returned them (checkpoint / resume of the saving loop of
 * docs/src/tutorials/biblock/smoothing.md:55); count == 0 is DMT_ERR_ARG (use dmt_path_moments_reset) */
int32_t dmt_set_path_moments(dmt_ctx *ctx, const double *mean, const double *m2, uint64_t count);
/* pooled over the chains that share a parameter / data set (chains c with pset_of_chain[c] == q, m of them), [NP][d][P]:
 *   mean = (1/m) sum mu_c;  var = (sum m2_c / n + sum (mu_c - mean)^2) / m, the variance of all n m draws;
 *   rhat = sqrt(var+ / W), the Gelman-Rubin statistic with W = sum m2_c / (m (n-1)), B = n sum (mu_c - mean)^2 / (m-1),
 *   var+ = (n-1)/n W + B/n; NaN when m < 2, n < 2 or W == 0 (e.g. at the known start point).
 * Sums in a fixed order: bitwise reproducible for a given (M, pset map).  LOCAL to this context (rank): pooling across GPUs is
 * not done here.  The ensemble-wide summary of many chains on one recording (docs/src/tutorials/biblock/smoothing.md:55). */
int32_t dmt_get_pset_path_moments(dmt_ctx *ctx, double *mean, double *var, double *rhat);

/* ---- the hot path --------------------------------------------------------------------------------------------- */
/* GP.set_obs!(be)                          src/block_ensemble.jl:192 -> src/biblock.jl:275-280            (K7) */
int32_t dmt_set_artificial_obs(dmt_ctx *ctx, int32_t layout);
/* recompute_guiding_term!(be[, Val])       src/block_ensemble.jl:202-212 -> src/block.jl:104-110          (K1) */
int32_t dmt_recompute_guiding_term(dmt_ctx *ctx, int32_t layout, int32_t which);
/* find_W_for_X!(be)                        src/block_ensemble.jl:221 -> src/block.jl:120-131              (K5) */
int32_t dmt_find_W_for_X(dmt_ctx *ctx, int32_t layout);
/* loglikhd!(be) / loglikhd°!(be)           src/block_ensemble.jl:121,128 -> src/block.jl:140-152          (K4) */
int32_t dmt_loglikhd(dmt_ctx *ctx, int32_t layout, int32_t side, int32_t skip);
/* find_W_for_X!(be); loglikhd!(be) in one pass over X (same results as the two calls)                  (K5+K4) */
int32_t dmt_find_W_and_loglikhd(dmt_ctx *ctx, int32_t layout);
/* draw_proposal_path!(be)                  src/block_ensemble.jl:50 -> src/biblock.jl:80-106        (K3+K2+K4)
 * Z == NULL: N(0,1) from Philox4x32-10, counter (chain, tile, iter, stream).  Z != NULL: host normals [S][dw][M]
 * (the parity hook: "feed the reference's own Wiener increments into both implementations"). */
int32_t dmt_draw_proposal_path(dmt_ctx *ctx, int32_t layout, uint32_t iter, const double *Z);
/* find_W_for_X!(be); loglikhd!(be); draw_proposal_path!(be) — the three consecutive calls of the blocking sweep
 * (docs/src/tutorials/block_collection/inference_with_blocking.md:55-57) — in ONE pass over the path: the accepted noise
 * recovered by K5 feeds the pCN refresh in registers.  Same results as the three calls up to FP64 rounding. (K5+K4+K3+K2+K4) */
int32_t dmt_find_W_loglikhd_draw(dmt_ctx *ctx, int32_t layout, uint32_t iter, const double *Z);
/* The whole body of the blocking sweep before the accept step, in the tutorial's order
 * (docs/src/tutorials/block_collection/inference_with_blocking.md:52-57):
 *   GP.set_obs!(be); recompute_guiding_term!(be, Val(:P_only)); find_W_for_X!(be); loglikhd!(be); draw_proposal_path!(be)
 * as three launches: the end-point gather, K1 (through the guiding cache when enabled) and ONE fused forward pass over the
 * path.  Same results as the five calls up to FP64 rounding. */
int32_t dmt_blocking_sweep(dmt_ctx *ctx, int32_t layout, uint32_t iter);
/* recompute_path!(b°, b.WW; skip) as used by set_proposal_law! (src/biblock.jl:343 -> src/block.jl:161-187):
 * law and X of `law_side`, noise of `noise_side`; sets ll[law_side].                                    (K2+K4) */
int32_t dmt_recompute_path(dmt_ctx *ctx, int32_t layout, int32_t law_side, int32_t noise_side, int32_t skip);
/* set_proposal_law! minus the host-side name translation (src/biblock.jl:334-344): if critical, K1 on the proposal
 * laws; then recompute_path!(b°, b.WW; skip). Parameters must have been uploaded with dmt_set_params/_aux first. */
int32_t dmt_set_proposal_law(dmt_ctx *ctx, int32_t layout, int32_t critical_change, int32_t skip);
/* accept_reject_proposal_path!(be, i)      src/block_ensemble.jl:63-67 -> src/biblock.jl:121-127          (K6)
 * E == NULL: Exp(1) = -log(u) from Philox; else host E[n_blocks][M].  iter indexes the histories (0-based). */
int32_t dmt_accept_reject_path(dmt_ctx *ctx, int32_t layout, uint32_t iter, const double *E);
/* swap_XX!/swap_WW!/swap_PP!/swap_ll!/swap_paths! (src/biblock.jl:148-209); chain_mask[M] or NULL (= all) */
int32_t dmt_swap(dmt_ctx *ctx, int32_t layout, int32_t what, const uint8_t *chain_mask);
/* The same swaps for SOME blocks of SOME recordings: mask[n_blocks][M], 1 = swap — the BiBlock-level methods swap_XX!(bb) ...
 * swap_ll!(bb) of one block of one recording (src/biblock.jl:148-209) and the BlockCollection-level ones (src/block_collection.jl:84-118). */
int32_t dmt_swap_blocks(dmt_ctx *ctx, int32_t layout, int32_t what, const uint8_t *block_chain_mask);
/* save_ll!(be, i)                          src/biblock.jl:256-259 */
int32_t dmt_save_ll(dmt_ctx *ctx, int32_t layout, uint32_t iter);

/* ---- reductions / read-back ----------------------------------------------------------------------------------- */
/* fetch_ll(be)/fetch_ll°(be)  (src/block_ensemble.jl:140,152; src/block_collection.jl:144,156): LOCAL (this GPU)
 * sum over chains and blocks in a fixed tree order; per_block[n_blocks] optional.  Cross-GPU: dmt_allreduce or host. */
int32_t dmt_fetch_ll(dmt_ctx *ctx, int32_t layout, int32_t side, double *total, double *per_block);
int32_t dmt_get_ll(dmt_ctx *ctx, int32_t layout, int32_t side, double *ll /* [n_blocks][M] */);
int32_t dmt_set_ll(dmt_ctx *ctx, int32_t layout, int32_t side, const double *ll);
int32_t dmt_get_success(dmt_ctx *ctx, int32_t layout, uint8_t *ok /* [n_blocks][M], last forward op */);
/* accpt_history / ll_history (src/biblock.jl:47, src/block.jl:58) for iterations it0..it1 inclusive */
int32_t dmt_get_accept_history(dmt_ctx *ctx, int32_t layout, uint32_t it0, uint32_t it1, uint8_t *acc /* [it][n_blocks][M] */);
/* set_accepted!(bb, i, v)  src/biblock.jl:130-135 and set_ll!(b, i, v)  src/block.jl:82-86: overwrite one history entry */
int32_t dmt_set_accepted(dmt_ctx *ctx, int32_t layout, uint32_t iter, const uint8_t *acc /* [n_blocks][M] */);
int32_t dmt_set_ll_history(dmt_ctx *ctx, int32_t layout, int32_t side, uint32_t iter, const double *ll /* [n_blocks][M] */);
int32_t dmt_get_ll_history(dmt_ctx *ctx, int32_t layout, int32_t side, uint32_t it0, uint32_t it1, double *ll /* [it][n_blocks][M] */);
/* accpt_rate numerators (src/biblock.jl:232): LOCAL accept counts per block over it0..it1 */
int32_t dmt_accept_counts(dmt_ctx *ctx, int32_t layout, uint32_t it0, uint32_t it1, int64_t *counts /* [n_blocks] */);
/* the last accept decisions of dmt_accept_reject_path, [n_blocks][M] */
int32_t dmt_get_last_accept(dmt_ctx *ctx, int32_t layout, uint8_t *acc);

/* ---- guiding term access (parity hook, SURVEY §7.1: inject the real reference's H,F,c) ---------------------- */
/* H[n_k][d*d][P], F[n_k][d][P], c[n_k][P] of interval k; on upload only grid points 0..n_k-2 and c[0] are kept
 * (left-point rule: nothing on the path reads the right end point). */
int32_t dmt_get_guiding_term(dmt_ctx *ctx, int32_t side, int32_t store, int32_t k, double *H, double *F, double *c);
int32_t dmt_upload_guiding_term(dmt_ctx *ctx, int32_t side, int32_t store, int32_t k, const double *H, const double *F, const double *c);

/* ---- guiding cache: the fast path of recompute_guiding_term!(be, Val(:P_only)) in smoothing-with-blocking sweeps ----- */
/* Between two sweeps of the tutorial loop (docs/src/tutorials/block_collection/inference_with_blocking.md:52-58) only the
 * artificial end-point observation of each non-terminal block changes (GP.set_obs!, src/biblock.jl:275-278).  With the cache
 * enabled for a layout, dmt_recompute_guiding_term keeps a layout-private copy of the accepted laws' guiding term together
 * with its exact affine (F) / quadratic (c) dependence on that observation; the first call after any change of the accepted
 * laws rebuilds it (1 + 2d + d(d-1)/2 backward-filter passes), every later call is a single streaming pass F = F0 + Psi v.
 * Results equal the uncached ones up to FP64 rounding.  Worth it only when the laws stay fixed for many sweeps (smoothing);
 * leave it off when parameters change every iteration.  Costs (d + d^2) extra doubles per grid point and pset per layout.
 * While enabled, the layout's guiding term is private to the layout (read it with dmt_get_layout_guiding_term). */
int32_t dmt_enable_guiding_cache(dmt_ctx *ctx, int32_t layout, int32_t enable);
/* accepted-side guiding term as ops on `layout` see it (the layout-private store when the cache is valid, else the shared one) */
int32_t dmt_get_layout_guiding_term(dmt_ctx *ctx, int32_t layout, int32_t store, int32_t k, double *H, double *F, double *c);

/* ---- tuning: lanes per (chain, block) in the register-tile forward kernel (K2-K5) ------------------------------------
 * 0 (default) = automatic: 1 lane when chains x blocks fill the GPU, else the largest of 2/4/8 for which all threads are still
 * resident at once — the lanes split the tile's Philox/Box-Muller calls and compute everything else redundantly, so results
 * and random streams are bit-identical for every setting.  1, 2, 4, 8 force a value; under dmt_set_sweep_mode(0) a forced value
 * also makes the fused sweep pass run the register-tile kernel.  No counterpart in the reference (its per-recording loop,
 * src/block_ensemble.jl:50, is serial). */
int32_t dmt_set_fwd_lanes(dmt_ctx *ctx, int32_t lanes);

/* ---- tuning: memory schedule of the fused blocking-sweep pass (dmt_blocking_sweep / dmt_find_W_loglikhd_draw) ----------
 * 1 = always the register-tile kernel (fwd_kernel.cuh), with dmt_set_fwd_lanes lanes per (chain, block).  The other kernels need every
 * chain to own its parameter set in chain order, a uniform law parity and Z == NULL; modes 2, 3 and 5 force one of them and return
 * DMT_ERR_UNSUPPORTED where these do not hold:
 *   2 = software-pipelined kernel (sweep_kernel.cuh: guiding term through a TMA shared-memory ring, X double-buffered in registers),
 *       one lane per (chain, block): DMT_ERR_UNSUPPORTED unless dmt_set_fwd_lanes is 0 or 1;
 *   3 = warp-specialised kernel (sweep_ws_kernel.cuh: per group of 32 chains and block a CTA of 16 warps that form a pipeline — TMA
 *       producer, generator warps, inverse solve + accepted likelihood, the proposal's recursion, the proposal's likelihood — over
 *       shared-memory rings, one CTA per SM);
 *   5 = step-parallel kernel (sweep_sp_kernel.cuh: four lanes per (chain, block), lane s owns step s of every 4-step tile; only the
 *       proposal's recursion runs as four rounds with a shuffle broadcast).
 * 0 (default) = automatic: the register-tile kernel where the conditions above do not hold or dmt_set_fwd_lanes forces lanes; else
 * warp-specialised while the grid of (32 chains, block) units fits one round of CTAs, then (models with >= 2 Wiener coordinates)
 * step-parallel up to 14,080 (chain, block) units, then two lanes per (chain, block) in the register-tile kernel while that grid fits
 * one wave, then the pipelined kernel with lazy noise or the register-tile kernel with eager noise.  Other modes (4 included) are
 * DMT_ERR_ARG.  Same arithmetic, results equal up to FP64 rounding (different FMA contraction). */
int32_t dmt_set_sweep_mode(dmt_ctx *ctx, int32_t mode);
/* Diagnostics: name and thread mapping of the forward kernel (K2-K5) this context launched last, e.g. "sweep_ws_kernel<wide, lazy>",
 * "sweep_pipe_kernel<lanes=1, lazy>", "fwd_kernel<op=6, lanes=4>" — what a benchmark should print instead of guessing the automatic
 * choice.  No counterpart in the reference. */
int32_t dmt_get_last_forward_kernel(dmt_ctx *ctx, char *buf, int32_t len);
/* Lazy noise.  In the blocking loop find_W_for_X!(be) overwrites b.WW at the start of EVERY sweep
 * (docs/src/tutorials/block_collection/inference_with_blocking.md:52-58, src/block.jl:120-131), so the accepted noise W and the
 * proposal noise W° the sweep produces are never read.  With enable = 1 the pipelined sweep over a layout that covers all intervals
 * does not store them (120 instead of 168 B per step for Lorenz); X, X°, ll, ll° and the accept decisions are unchanged.  The accepted
 * noise is rebuilt on demand — by K5 over the layout swept last, i.e. exactly what find_W_for_X! would return — before anything
 * reads it (dmt_get_W, dmt_get_W_chains, a draw or recompute_path! without a preceding find_W_for_X!, swap_WW!) or changes the
 * accepted laws.  W° is unspecified while the mode is on.  Rebuilding after ANOTHER layout's GP.set_obs! has moved a shared block
 * end point uses the current artificial observation (a difference of the order of sqrt(artificial_noise) in that block). */
int32_t dmt_set_lazy_noise(dmt_ctx *ctx, int32_t enable);

/* ---- the ODE solver of the backward filter (K1) --------------------------------------------------------------------------
 * DMT_K1_RK4 (default): classical RK4 on the path grid, covariance form on exact-observation intervals (DESIGN.md §4).
 * DMT_K1_TSIT5: upstream's solver — GuidedProposals integrates (H,F,c) with OrdinaryDiffEq's Tsit5() (OrdinaryDiffEq 5.41.0,
 * Manifest.toml:352-356; call sites src/sampling_unit.jl:60-66, src/block.jl:104-110): Tsitouras' adaptive 5(4) pair with
 * OrdinaryDiffEq's default controller and its free interpolant on the path grid; reltol / abstol as passed (OrdinaryDiffEq's defaults:
 * 1e-3, 1e-6).  Restated from the published method, not bit-equal to upstream (no Julia here) — it carries upstream's O(tolerance)
 * error, which the RK4 mode does not.  Incompatible with the guiding cache (F is exactly affine in the block end point only under a
 * fixed-grid discretisation).  dmt_get_bwd_steps: accepted / rejected steps of the last Tsit5 launch, summed over all threads. */
enum { DMT_K1_RK4 = 0, DMT_K1_TSIT5 = 1 };
int32_t dmt_set_bwd_solver(dmt_ctx *ctx, int32_t solver, double reltol, double abstol);
int32_t dmt_get_bwd_steps(dmt_ctx *ctx, int32_t *accepted, int32_t *rejected);

/* ---- tuning: thread mapping of the backward filter (K1) -------------------------------------------------------------
 * 0 (default) = automatic; 1 = one thread per (parameter set, block, side); 2 = d lanes share one parameter set, lane r owning
 * row r of H (wide states; DMT_ERR_UNSUPPORTED where it is not implemented).  Results agree to FP64 rounding. */
int32_t dmt_set_bwd_mode(dmt_ctx *ctx, int32_t mode);

/* ---- test hooks: the device's counter-based random streams for given counters ------------------------------- */
/* out[n_chains][n_tiles][4*dw]: the N(0,1) draws the pCN refresh (K3) uses for chains chain0.., tiles tile0.., iteration iter.
 * Replaces nothing in the reference (its Wnr/randn draws are not reproducible elsewhere); lets tests pin the generator. */
int32_t dmt_debug_normals(dmt_ctx *ctx, uint32_t chain0, uint32_t tile0, uint32_t iter, uint32_t layout, int32_t n_chains, int32_t n_tiles, double *out);
/* out[n_chains][n_blocks]: the Exp(1) draws of accept_reject_proposal_path! (src/biblock.jl:122) */
int32_t dmt_debug_exponentials(dmt_ctx *ctx, uint32_t chain0, uint32_t iter, uint32_t layout, int32_t n_chains, int32_t n_blocks, double *out);

/* ---- multi-GPU: the small allreduce of ll sums / accept counts (SURVEY §8e, C1) ----------------------------- */
/* NCCL is dlopen'ed at first use.  unique_id: the 128-byte ncclUniqueId from dmt_nccl_unique_id on rank 0. */
int32_t dmt_nccl_unique_id(uint8_t *id128);
int32_t dmt_comm_init(dmt_ctx *ctx, int32_t n_ranks, int32_t rank, const uint8_t *id128);
/* Peer-memory variant of the same exchange (preferred on one NVLink/NVSwitch node): every rank exports a 64-byte CUDA IPC
 * handle of its exchange buffer, the host all-gathers the handles by any means, dmt_p2p_init maps the peers.  After that
 * dmt_allreduce_stats is ONE single-CTA kernel that stores this rank's values into every peer's buffer, publishes / awaits a
 * sequence number with system-scope release / acquire, and sums the slots in rank order (bitwise reproducible, identical on
 * all ranks) — no NCCL call on the path.  One process per GPU (IPC handles cannot be opened by the exporting process). */
int32_t dmt_p2p_export(dmt_ctx *ctx, uint8_t *handle64);
int32_t dmt_p2p_init(dmt_ctx *ctx, int32_t n_ranks, int32_t rank, const uint8_t *handles /* [n_ranks][64] */);
int32_t dmt_p2p_disable(dmt_ctx *ctx); /* back to dmt_comm_init's communicator (e.g. another rank could not map its peers) */
/* out[0]=sum ll, out[1]=sum ll°, out[2..2+n_blocks)=accept counts of the last accept step, summed over ranks */
int32_t dmt_allreduce_stats(dmt_ctx *ctx, int32_t layout, double *out /* [2+n_blocks] */);

#ifdef __cplusplus
}
#endif
#endif
