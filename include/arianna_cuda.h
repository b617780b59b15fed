/*
 * arianna_cuda.h -- C ABI of libarianna_cuda.so, the B200 (sm_100a) multi-chain Metropolis engine that
 * drops in behind Arianna.jl's `Metropolis` / `StoreCallbacks` / `StoreTrajectories` /
 * `PolicyGradientEstimator` for `particle_1d`-type systems.
 *
 * Arianna has no FFI of its own (it is pure Julia); the "reference interface" each entry point replaces is
 * the Julia method it stands in for, cited as path:line under the reference tree.  INTEGRATION.md shows the
 * `ccall` bindings of the Julia shim.
 *
 * Conventions
 *   - every function returns an int32 status (ARIANNA_OK == 0); nothing throws or aborts across the ABI;
 *   - arianna_last_error(h) returns a NUL-terminated message owned by the handle (h may be NULL for errors
 *     raised by arianna_create itself: thread-local storage);
 *   - host pointers are borrowed for the duration of the call only;  all calls on one handle must come from
 *     one host thread at a time;
 *   - kernels are enqueued asynchronously on the handle's stream; every function that returns numbers to the
 *     host synchronises that stream first;
 *   - one handle == one GPU == one contiguous shard [chain_offset, chain_offset + n_chains) of the global
 *     ensemble.  Multi-GPU = one process (or handle) per GPU; per-chain results do not depend on the sharding
 *     because the RNG stream of a chain is keyed by its GLOBAL index.
 */
#ifndef ARIANNA_CUDA_H
#define ARIANNA_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ARIANNA_ABI_VERSION 2
#if defined(__GNUC__)
#define ARIANNA_API __attribute__((visibility("default")))
#else
#define ARIANNA_API
#endif
#define ARIANNA_MAX_MOVES 16

typedef struct arianna_handle arianna_handle;

enum arianna_status {
    ARIANNA_OK = 0,
    ARIANNA_ERR_INVALID = 1,     /* bad argument (the Julia shim throws ArgumentError)                   */
    ARIANNA_ERR_CUDA = 2,        /* a CUDA runtime call failed; message holds cudaGetErrorString          */
    ARIANNA_ERR_NOMEM = 3,       /* device or host allocation failed                                      */
    ARIANNA_ERR_UNSUPPORTED = 4, /* valid request this build cannot serve (e.g. replay with XOSHIRO rng)  */
    ARIANNA_ERR_NO_DEVICE = 5,   /* no CUDA device: there is NO CPU fallback                              */
    ARIANNA_ERR_NCCL = 6         /* libnccl could not be loaded or an NCCL call failed                    */
};

/* potential(x): the script-level global of the examples (MC_harmonic_oscillator.jl:4, test/runtests). */
enum arianna_potential {
    ARIANNA_POT_HARMONIC = 0,    /* x^2                                                                   */
    ARIANNA_POT_QUARTIC = 1,     /* x^4                                                                   */
    ARIANNA_POT_DOUBLE_WELL = 2  /* (x^2 - 1)^2                                                           */
};

enum arianna_rng_mode {
    ARIANNA_RNG_PHILOX = 0,      /* in-register counter-based Philox4x32-10 + Box-Muller (native mode)     */
    ARIANNA_RNG_XOSHIRO = 1      /* per-chain xoshiro256++ state + ziggurat randn, the reference's generator
                                    family (Random.Xoshiro [EXT]); states uploaded with arianna_set_rng_state */
};

enum arianna_arith_mode {
    ARIANNA_ARITH_EXACT = 0,     /* the reference's exact binary64 operation order, no FMA contraction
                                    (SURVEY.md Appendix A.1)                                               */
    ARIANNA_ARITH_FAST = 1       /* algebraically equal, symmetric-proposal cancellation, exact restore on
                                    reject                                                                 */
};

/* Element type of the ensemble: `Particle{T<:AbstractFloat}` (particle_1d.jl:9-16) with matching action and parameter
 * types.  F32 = Particle{Float32}, Displacement{Float32}, ComponentArray(σ = 0.1f0): state and proposal arithmetic in
 * Float32, log-proposal constants and the accept test in Float64 exactly as Julia's promotion rules make the
 * reference's generic code run (csrc/kernels_f32.cuh).  F32 handles: single-move pools, native Philox stream or replay,
 * arianna_sweep / arianna_sweep_replay / the callbacks; series, host jobs, PGMC and XOSHIRO return UNSUPPORTED. */
enum arianna_dtype {
    ARIANNA_F64 = 0,
    ARIANNA_F32 = 1
};

/* Flags of arianna_sweep */
#define ARIANNA_SWEEP_REDUCE 1u  /* fuse the callback reductions (energy / acceptance sums) into the sweep  */

typedef struct arianna_config {
    uint32_t struct_size;        /* = sizeof(arianna_config); ABI guard                                    */
    int32_t device;              /* CUDA device ordinal; -1 = the calling thread's current device          */
    int64_t n_chains;            /* chains held by THIS handle (local shard), >= 1                         */
    int64_t chain_offset;        /* global 0-based index of the first local chain                          */
    int64_t n_chains_total;      /* global ensemble size (denominator of the callback means); 0 = n_chains */
    int64_t seed;                /* `seed` of Metropolis(chains; seed=...) (metropolis.jl:288): chain c
                                    (1-based, global) owns stream  seed + c - 1  (metropolis.jl:262)        */
    double beta;                 /* Particle.β (particle_1d.jl:11), shared by all chains unless
                                    arianna_set_betas is called                                            */
    int32_t potential;           /* enum arianna_potential                                                 */
    int32_t n_moves;             /* pool size, 1 .. ARIANNA_MAX_MOVES                                      */
    double sigma[ARIANNA_MAX_MOVES];  /* Move.parameters.σ per move (ComponentArray(σ=...))                */
    double weight[ARIANNA_MAX_MOVES]; /* Move.weight per move; must sum to 1 (Categorical validates [EXT]) */
    int32_t rng_mode;            /* enum arianna_rng_mode                                                  */
    int32_t arith_mode;          /* enum arianna_arith_mode                                                */
    void *stream;                /* optional cudaStream_t to run on; NULL = the handle creates its own     */
    int32_t dtype;               /* enum arianna_dtype                                                     */
    int32_t reserved;            /* must be 0                                                              */
} arianna_config;

/* Summed GradientData record of one learnable move (gradients.jl:41-47), P = 1 parameter (σ). */
typedef struct arianna_gradient_data {
    double j;                    /* Σ objective r·α                                                        */
    double dj;                   /* Σ ∇j                                                                   */
    double dlogq_forward;        /* Σ ∇logq_forward                                                        */
    double g;                    /* Σ ∇logq_f · ∇logq_fᵀ                                                   */
    double n;                    /* sample count (exact integer in binary64)                               */
} arianna_gradient_data;

ARIANNA_API uint32_t arianna_abi_version(void);
ARIANNA_API const char *arianna_last_error(const arianna_handle *h);

/* Lifecycle.  Replaces Metropolis(chains; pool, seed, ...) (metropolis.jl:240-291) + the per-chain heap
 * objects of `chains::Vector{Particle}` (particle_1d.jl:9-16): chains live only in HBM. */
ARIANNA_API int32_t arianna_create(const arianna_config *cfg, arianna_handle **out);
ARIANNA_API int32_t arianna_destroy(arianna_handle *h);

/* Chain state.  set: `[System(x, β) for ...]` (MC_harmonic_oscillator.jl:13); e = potential(x) is derived.
 * init_synthetic: x0 = 4u - 2 from the engine's counter-based stream (same expression, :13).
 * get: what store_trajectory / callback_energy read, `system.x`, `system.e` (particle_1d.jl:63-70);
 * either pointer may be NULL.  Resets nothing. */
ARIANNA_API int32_t arianna_set_state(arianna_handle *h, const double *x);
ARIANNA_API int32_t arianna_init_synthetic(arianna_handle *h, int64_t seed);
ARIANNA_API int32_t arianna_get_state(arianna_handle *h, double *x, double *e);
/* The same for ARIANNA_F32 handles in their own element type (the Float64 entry points above also work on them:
 * set rounds to Float32, get widens exactly). */
ARIANNA_API int32_t arianna_set_state_f32(arianna_handle *h, const float *x);
ARIANNA_API int32_t arianna_get_state_f32(arianna_handle *h, float *x, float *e);
/* Asynchronous variant for StoreTrajectories at scale (algorithms.jl:198-203): snapshots x on the device and
 * drains the snapshot into caller-pinned memory on a second stream, so the PCIe transfer overlaps the next sweep;
 * arianna_copy_wait() / arianna_synchronize() complete it. */
ARIANNA_API int32_t arianna_get_state_async(arianna_handle *h, double *x_pinned);
/* Waits for the LAST arianna_get_state_async frame only (not for sweeps queued after it): the host writes frame i to
 * disk while sweep i + 1 runs. */
ARIANNA_API int32_t arianna_copy_wait(arianna_handle *h);
ARIANNA_API int32_t arianna_set_beta(arianna_handle *h, double beta);
ARIANNA_API int32_t arianna_set_betas(arianna_handle *h, const double *betas); /* per-chain β, [n_chains] host */

/* Replica exchange (parallel tempering) across per-chain β ladders.  A ladder is L consecutive chains by GLOBAL index
 * (2 <= L <= ARIANNA_MAX_LADDER); global chain g is rung g % L of ladder g / L.
 * arianna_set_ladder writes per-chain β = betas[g % L] ([L] host), with the same effect as arianna_set_betas; the shard
 * must hold whole ladders (chain_offset % L == 0 and n_chains % L == 0, ARIANNA_ERR_INVALID otherwise).  Calling it
 * with another L resets the round index and the swap counters; later arianna_set_beta(s) calls are allowed (the
 * exchange always reads the per-chain β).
 * arianna_replica_exchange runs ONE round R (per handle, from 0): rungs (r, r + 1) with r ≡ R (mod 2) of every local
 * ladder swap their positions x iff min(1, exp(Δ)) > u, Δ = (β_g − β_{g+1})·(e_g − e_{g+1}), e = potential(x) in exact
 * binary64, u = (A >> 11)·2^-53 from the Philox stream tag 4 (sid = seed + g, p = R, sub 0), strict >, NaN rejects.  β,
 * the Move counters and the chain's Metropolis stream stay with the slot (the temperature).  Asynchronous.
 * arianna_exchange_counters: accepted swaps per rung pair [L − 1] (local shard) and the number of rounds; pair k was
 * attempted n_ladders_local × #{R' < rounds : R' ≡ k (mod 2)} times.
 * arianna_ladder_sums: the callback record restricted to each rung, [L][2 + n_moves] = (Σ e, Σ_c acc_ck/tot_ck per
 * move, chain count) over the local shard, in a fixed reduction order; multi-GPU hosts sum them across ranks.
 * Float64 ensembles with the native Philox stream (ARIANNA_ERR_UNSUPPORTED otherwise). */
#define ARIANNA_MAX_LADDER 256
ARIANNA_API int32_t arianna_set_ladder(arianna_handle *h, int32_t L, const double *betas);
ARIANNA_API int32_t arianna_replica_exchange(arianna_handle *h);
ARIANNA_API int32_t arianna_exchange_counters(arianna_handle *h, int64_t *accepted, int64_t *rounds);
ARIANNA_API int32_t arianna_ladder_sums(arianna_handle *h, double *sums);

/* Histograms and moments of the chains' current state, reduced on the device (StoreTrajectories + a host histogram
 * without the download).  observable: ARIANNA_OBS_X the position, ARIANNA_OBS_E the energy potential(x) (Float64
 * handles: exact binary64; Float32 handles: Float64(potential_f32(x)), i.e. what arianna_get_state_f32 returns, widened).
 * Global chain g = chain_offset + c belongs to group g % n_groups (1 <= n_groups <= ARIANNA_MAX_LADDER; 1 = the whole
 * ensemble, L = the rungs of a replica-exchange ladder); counts of any sharding sum to the one-handle counts.
 * Bin rule (a formula, not edges): inv_w = n_bins / (hi − lo) in binary64, computed once by arianna_set_histogram;
 * k = floor((v − lo)·inv_w) with the subtraction and the product rounded separately (no contraction).  NaN -> the nan
 * cell, k < 0 -> underflow, k >= n_bins -> overflow (±inf land there), otherwise bin k.
 * counts [n_groups][n_bins + 3] int64 = [n_bins regular][underflow][overflow][nan]; moments [n_groups][3] =
 * (n, Σv, Σv²) over the finite v, binary64 sums in a fixed order (deterministic for a handle).
 * arianna_set_histogram allocates and zeroes the accumulators (a second call replaces the binning);
 * n_groups·(n_bins + 3) <= ARIANNA_MAX_HISTOGRAM_CELLS, n_bins >= 1, lo and hi finite, lo < hi, inv_w finite and > 0.
 * arianna_histogram_accumulate adds one sample of every local chain (asynchronous; reads x only: no callback record,
 * series record, counter, β, σ or step count changes).  arianna_histogram_read returns the local-shard accumulators
 * and the number of accumulate calls (any pointer may be NULL; synchronises); multi-GPU hosts sum counts and moments
 * across ranks.  arianna_histogram_reset zeroes counts, moments and the call count and keeps the binning.
 * ARIANNA_ERR_INVALID for bad arguments and for accumulate / read / reset before arianna_set_histogram. */
#define ARIANNA_MAX_HISTOGRAM_CELLS 16384
enum arianna_observable { ARIANNA_OBS_X = 0, ARIANNA_OBS_E = 1 };
ARIANNA_API int32_t arianna_set_histogram(arianna_handle *h, int32_t observable, double lo, double hi, int32_t n_bins,
                                          int32_t n_groups);
ARIANNA_API int32_t arianna_histogram_accumulate(arianna_handle *h);
ARIANNA_API int32_t arianna_histogram_read(arianna_handle *h, int64_t *counts, double *moments, int64_t *n_samples);
ARIANNA_API int32_t arianna_histogram_reset(arianna_handle *h);

/* Policy parameters θ = (σ) of move `move_id` (0-based): the shared `parameters` array every chain's Move
 * aliases (metropolis.jl:253-260), mutated in place by learning_step! (learning.jl:33).  P must be 1.
 * log_norm (optional, may be NULL) lets the host pass its own binary64 value of log(2π·σ²)/2
 * (particle_1d.jl:53) so that replay is bit-exact with the host language's `log`. */
ARIANNA_API int32_t arianna_set_params(arianna_handle *h, int32_t move_id, const double *theta, int32_t P,
                           const double *log_norm);
ARIANNA_API int32_t arianna_get_params(arianna_handle *h, int32_t move_id, double *theta, int32_t P);

/* K fused Metropolis steps for every local chain, native RNG (cfg.rng_mode).  Replaces K consecutive
 * make_step!(sim, ::Metropolis) calls with sweepstep = 1 (metropolis.jl:302-309 -> mc_sweep! :203-212 ->
 * mc_step! :176-190).  Asynchronous. */
ARIANNA_API int32_t arianna_sweep(arianna_handle *h, int64_t K, uint32_t flags);

/* A whole stretch of the schedule in one call: n_stores consecutive store intervals of K[i] Metropolis steps each,
 * with the StoreCallbacks record (algorithms.jl:97-102: callback_energy, callback_acceptance) taken after every
 * interval ON THE DEVICE.  Equivalent to  for i: arianna_sweep(h, K[i], ARIANNA_SWEEP_REDUCE); arianna_callback_sums
 * but the chains stay in registers across up to ARIANNA_MAX_SERIES intervals per launch, nothing is copied to the
 * host between stores and the multi-GPU host all-reduces the whole series at once.  records (optional, host):
 * [n_stores][2 + n_moves] = (Σ e, Σ_c acc_ck/tot_ck for every move k, local chain count) per store, local shard --
 * callback_acceptance is a per-move vector (metropolis.jl:319-321), NaN while some chain never tried a move; NULL =
 * leave them on the device (arianna_series_device; asynchronous).  arianna_series_global all-reduces the device
 * records of the LAST arianna_sweep_series call over the communicator (arianna_comm_init) and returns ensemble-wide
 * records.  Native Philox stream only (ARIANNA_ERR_UNSUPPORTED otherwise: use arianna_sweep). */
#define ARIANNA_MAX_SERIES 64
ARIANNA_API int32_t arianna_sweep_series(arianna_handle *h, int32_t n_stores, const int64_t *K, double *records);
ARIANNA_API int32_t arianna_series_device(arianna_handle *h, double **dptr, int32_t *n_doubles);
ARIANNA_API int32_t arianna_series_global(arianna_handle *h, int32_t n_stores, double *records);
/* How many store intervals one launch of arianna_sweep_series fuses for this ensemble (longer series are chunked):
 * callers that can choose the length of a stretch should use a multiple of it. */
ARIANNA_API int32_t arianna_series_per_launch(arianna_handle *h, int32_t *n);

/* The same stretch as a complete job with HOST buffers: chains in (x_in, [n_chains], NULL = keep the resident state),
 * n_stores store intervals, records out ([n_stores][2 + n_moves] local-shard sums, may be NULL), chains out (x_out, may be
 * NULL) -- i.e. `chains = [...]; run!(Simulation(chains, (Metropolis, StoreCallbacks, StoreLastFrames), steps))`
 * (src/simulation.jl:175-204) in one call.  The ensemble is cut into slices of chains that go through ALL the store
 * intervals one slice after the other, so that the upload of the next slice (H2D stream) and the download of the
 * previous one (D2H stream) overlap the sweep of the current one (pass page-locked buffers -- arianna_host_alloc -- for
 * the copies to be asynchronous).  n_slices is the number of REGULAR slices (size n_chains / n_slices); the plan starts
 * with smaller slices (1/64 of the ensemble, doubling) and, when x_out is given, ends with slices that halve again, so
 * that the exposed first upload and last download are short.  Chains are independent: the final chains and counters
 * are bit-identical to arianna_set_state + arianna_sweep_series + arianna_get_state, the records equal up to the order
 * of the slice sums.  Synchronous: host buffers are complete / reusable on return.  Multi-GPU hosts all-reduce the
 * device records afterwards (arianna_series_global). */
ARIANNA_API int32_t arianna_run_host_job(arianna_handle *h, const double *x_in, int32_t n_stores, const int64_t *K,
                                         double *records, double *x_out, int32_t n_slices);
/* PCIe view of the LAST arianna_run_host_job call: device time (ms, first copy start -> last copy end on the upload /
 * download stream, so it includes the waits on the sweeps in between) and the achieved GB/s of each direction; NaN for
 * a direction the job did not use.  Any pointer may be NULL. */
ARIANNA_API int32_t arianna_job_timing(arianna_handle *h, double *h2d_ms, double *h2d_gbs, double *d2h_ms, double *d2h_gbs);

/* Replay mode: the same K steps consuming caller-supplied draws instead of the native RNG, always in EXACT
 * arithmetic.  u_cat / z / u_acc are step-major [K][n_chains] (u_cat may be NULL when n_moves == 1);
 * `on_device` != 0 means the three pointers (and decisions_out) are device pointers.  decisions_out
 * (optional) receives mc_step!'s return value (metropolis.jl:185,188) per step and chain. */
ARIANNA_API int32_t arianna_sweep_replay(arianna_handle *h, int64_t K, const double *u_cat, const double *z,
                             const double *u_acc, uint8_t *decisions_out, int32_t on_device);

/* XOSHIRO mode: per-chain generator states [n_chains][4] uint64 -- the fields s0..s3 of the reference's
 * `Xoshiro(seed + c - 1)` (metropolis.jl:262-263; Random stdlib [EXT]).  The engine's default ziggurat tables are
 * Julia's literal ki / wi / fi (normal.jl [EXT]), so with those states the device draws the uniforms and normals Julia
 * draws (pinned by the known answers printed in the Julia manual, DESIGN.md section 3).
 * arianna_set_ziggurat_tables overrides the three 256-entry tables (a host whose randn uses other tables). */
ARIANNA_API int32_t arianna_set_rng_state(arianna_handle *h, const uint64_t *states);
ARIANNA_API int32_t arianna_get_rng_state(arianna_handle *h, uint64_t *states);
ARIANNA_API int32_t arianna_set_ziggurat_tables(arianna_handle *h, const uint64_t *ki, const double *wi, const double *fi);

/* Callbacks.  callback_energy (particle_1d.jl:68-70) and callback_acceptance (metropolis.jl:319-321: per
 * move, the mean over chains of accepted_calls/total_calls, NaN while some chain never tried the move).
 * arianna_callbacks returns the means over THIS handle's chains (the local shard); multi-GPU hosts use the
 * *_sums variants and combine across shards:
 *   sums[0] = Σ e,  sums[1 + k] = Σ_c acc_ck / tot_ck,  sums[1 + n_moves] = local chain count.
 * arianna_callback_sums_device exposes the device buffer holding those 2 + n_moves doubles (valid until the
 * next sweep) for an NCCL all-reduce without a host round trip; the host finishes the division. */
ARIANNA_API int32_t arianna_callbacks(arianna_handle *h, double *mean_energy, double *acc_per_move);
ARIANNA_API int32_t arianna_callback_sums(arianna_handle *h, double *sums);
ARIANNA_API int32_t arianna_callback_sums_device(arianna_handle *h, double **dptr, int32_t *n);

/* Move counters summed over the local chains (what a single-ensemble host `Move` would hold), and the raw
 * per-chain counters [n_moves][n_chains]. */
ARIANNA_API int32_t arianna_get_counters(arianna_handle *h, int64_t *accepted, int64_t *total);
ARIANNA_API int32_t arianna_get_chain_counters(arianna_handle *h, uint32_t *accepted, uint32_t *total);

/* PGMC.  One make_step!(sim, ::PolicyGradientEstimator) (estimator.jl:111-134): for each learnable move
 * (0-based ids, in order) and each chain, q_batch samples of sample_gradient_data/pgmc_estimate
 * (gradients.jl:93-121) with the analytic ∂σ log q = δ²/σ³ − 1/σ, summed into the per-move accumulators
 * gradients_data[k] (estimator.jl:130).  Asynchronous.
 * arianna_pgmc_read returns the accumulated SUMS (local shard); arianna_pgmc_reset zeroes them
 * (update.jl:55).  arianna_pgmc_sums_device exposes the [n_learn][5] device buffer for an all-reduce. */
ARIANNA_API int32_t arianna_pgmc_estimate(arianna_handle *h, int32_t q_batch, const int32_t *learn_ids, int32_t n_learn);
ARIANNA_API int32_t arianna_pgmc_estimate_replay(arianna_handle *h, int32_t q_batch, const int32_t *learn_ids,
                                     int32_t n_learn, const double *z /* [n_learn][q_batch][n_chains] */,
                                     int32_t on_device);
ARIANNA_API int32_t arianna_pgmc_read(arianna_handle *h, arianna_gradient_data *out, int32_t n_learn);
ARIANNA_API int32_t arianna_pgmc_reset(arianna_handle *h);
ARIANNA_API int32_t arianna_pgmc_sums_device(arianna_handle *h, double **dptr, int32_t *n);

/* PolicyGradientUpdate ON THE DEVICE (update.jl:50-57 + learning_step!, learning.jl:32-164): averages the accumulated
 * GradientData of every learnable move (all-reduced over the communicator first when there is one), applies the move's
 * optimiser, stores the new σ in a device-resident parameter block that every following sweep / estimator launch of
 * this handle reads, and zeroes the accumulators -- no host round trip per update (asynchronous).  The host copy of θ
 * is refreshed by arianna_params_sync / arianna_get_params, which also report (ARIANNA_ERR_INVALID) a step that left
 * σ outside (0, ∞), as Normal(0, σ) would throw in the reference.  p1 = η (VPG, BLPG, NPG) or δ (BLAPG, ANPG,
 * BLANPG); p2 = ϵid.  Float64 ensembles with the native Philox stream. */
enum arianna_optimiser_kind {
    ARIANNA_OPT_STATIC = 0, ARIANNA_OPT_VPG = 1, ARIANNA_OPT_BLPG = 2, ARIANNA_OPT_BLAPG = 3, ARIANNA_OPT_NPG = 4,
    ARIANNA_OPT_ANPG = 5, ARIANNA_OPT_BLANPG = 6
};
typedef struct arianna_optimiser {
    int32_t kind;                /* enum arianna_optimiser_kind                                            */
    int32_t reserved;
    double p1;
    double p2;
} arianna_optimiser;
ARIANNA_API int32_t arianna_pgmc_update_device(arianna_handle *h, const int32_t *learn_ids, const arianna_optimiser *opts,
                                               int32_t n_learn);
ARIANNA_API int32_t arianna_params_sync(arianna_handle *h);

/* Page-locked host memory for hosts without a CUDA binding of their own: what arianna_run_host_job and
 * arianna_get_state_async need for their copies to be asynchronous.  write_combined != 0: memory the host only WRITES
 * and the GPU reads (x_in) -- not snooped, faster over PCIe, very slow to read back on the CPU. */
ARIANNA_API int32_t arianna_host_alloc(int64_t bytes, int32_t write_combined, void **out);
ARIANNA_API int32_t arianna_host_free(void *p);

/* Plumbing. */
ARIANNA_API int32_t arianna_get_stream(arianna_handle *h, void **stream);
ARIANNA_API int32_t arianna_synchronize(arianna_handle *h);
/* Device time (CUDA events on the engine's stream, milliseconds) of the LAST arianna_sweep / arianna_sweep_series /
 * arianna_run_host_job call (sweep_ms: kernels + fused reductions + record folds; for a host job also the waits on the
 * slice uploads) and of the last estimator pass (pgmc_ms).  NaN when there was none; either pointer may be NULL.
 * Synchronises with the end of that work.  The reference only has a wall-clock `@elapsed` around its t-loop
 * (src/simulation.jl:184). */
ARIANNA_API int32_t arianna_timing(arianna_handle *h, double *sweep_ms, double *pgmc_ms);
ARIANNA_API int32_t arianna_launch_count(arianna_handle *h, int64_t *n_launches);
ARIANNA_API int32_t arianna_steps_done(arianna_handle *h, int64_t *steps);
ARIANNA_API int32_t arianna_device_info(arianna_handle *h, int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor,
                            int64_t *hbm_bytes);

/* FP64 pipe peak of the handle's device by a dependent-chain-free DFMA microbenchmark (flop/s); used as the
 * FP64 roofline denominator because MEASURED_PEAKS.json holds none. */
ARIANNA_API int32_t arianna_measure_fp64_peak(arianna_handle *h, double *flops_per_s);

/* Multi-GPU for hosts without their own collective library (the Julia shim): one handle per rank, chains sharded
 * by (chain_offset, n_chains, n_chains_total).  Rank 0 obtains a 128-byte NCCL unique id, the host distributes it
 * (MPI, sockets, a file ...) and every rank calls arianna_comm_init.  libnccl.so.2 is resolved with dlopen at the
 * first call (override with ARIANNA_NCCL_LIB), so single-GPU users never need it.  The *_global calls all-reduce
 * the 2 + n_moves callback sums / the 5 n_learn estimator sums over NVLink on the engine's stream and return
 * ensemble-wide values on every rank; without a communicator they equal the local calls. */
ARIANNA_API int32_t arianna_nccl_unique_id(void *id128);
ARIANNA_API int32_t arianna_comm_init(arianna_handle *h, const void *id128, int32_t rank, int32_t n_ranks);
ARIANNA_API int32_t arianna_callbacks_global(arianna_handle *h, double *mean_energy, double *acc_per_move);
/* arianna_series_global without stalling the compute stream: the records of the last series call are snapshotted and
 * the all-reduce + the copy into `records_pinned` (page-locked host memory, [n_stores][2 + n_moves]) run on a side stream while
 * the NEXT sweep already executes -- the next launch does not depend on the callback means of this one.
 * arianna_series_global_wait (or arianna_synchronize) completes it; one operation in flight per handle. */
ARIANNA_API int32_t arianna_series_global_begin(arianna_handle *h, int32_t n_stores, double *records_pinned);
ARIANNA_API int32_t arianna_series_global_wait(arianna_handle *h);
ARIANNA_API int32_t arianna_pgmc_read_global(arianna_handle *h, arianna_gradient_data *out, int32_t n_learn);

/* Diagnostic: evaluates the device FP64 math layer (csrc/math64.cuh) on host arrays so that tests can compare
 * the device code paths with extended-precision references.  kind: 0 min(1,exp(a)) | 1 -2 ln(b 2^-53) | 2 sqrt(a) |
 * 3 sin/cos(2 pi b 2^-53) -> out[2i], out[2i+1] | 4 Box-Muller(b, c) -> out[2i], out[2i+1] | 5 accept test of
 * x = a with the 11-bit prefix word b and refinement word c -> out[2i] = FP32-filtered, out[2i+1] = plain FP64
 * decision (8: the same with a 12-bit prefix) | 9 -2 ln(b 2^-52), b < 2^52 (the Box-Muller radius form) |
 * 6 / 7 Philox4x32-10 block of the Metropolis stream for (sid = b, p = c[, sub = a]) through the per-chain hoisted
 * form (sub 0) / the general form -> out[4i .. 4i+3] = the four 32-bit output words. */
ARIANNA_API int32_t arianna_debug_math(arianna_handle *h, int32_t kind, const double *a, const uint64_t *b,
                                       const uint64_t *c, double *out, int64_t n);

#ifdef __cplusplus
}
#endif
#endif /* ARIANNA_CUDA_H */
