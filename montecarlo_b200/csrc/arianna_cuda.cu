// arianna_cuda.cu -- C ABI of libarianna_cuda.so (declared in include/arianna_cuda.h).
//
// Host side of the engine: owns the HBM-resident ensemble, picks the kernel instantiation, keeps the draw
// indices (steps_done / estimator samples) and hands out device pointers of the small reduction buffers for
// the per-store NCCL all-reduce.  There is NO CPU fallback anywhere in this file: without a CUDA device
// arianna_create fails with ARIANNA_ERR_NO_DEVICE.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include <cuda_runtime.h>
#include <dlfcn.h>

#include "../../include/arianna_cuda.h"
#include "kernels.cuh"
#include "kernels_exchange.cuh"
#include "kernels_histogram.cuh"

using namespace arianna;

// ---- NCCL, resolved at run time (dlopen) so the library has no link-time dependency on it ------------------------
// Only the five entry points below are used; ABI of NCCL 2.x: ncclUniqueId is a 128-byte POD passed BY VALUE,
// ncclDouble == 8, ncclSum == 0.
namespace nccl {
struct UniqueId { char internal[128]; };
using Comm = void *;
struct Api {
    void *lib = nullptr;
    int (*GetUniqueId)(UniqueId *) = nullptr;
    int (*CommInitRank)(Comm *, int, UniqueId, int) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, Comm, cudaStream_t) = nullptr;
    int (*CommDestroy)(Comm) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
static Api g_api;
static const char *load(std::string &err)
{
    if (g_api.lib) return nullptr;
    const char *names[] = {getenv("ARIANNA_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void *lib = nullptr;
    for (const char *n : names)
        if (n && (lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break;
    if (!lib) { err = std::string("dlopen(libnccl.so.2) failed: ") + dlerror(); return err.c_str(); }
    Api a;
    a.lib = lib;
    a.GetUniqueId = (decltype(a.GetUniqueId))dlsym(lib, "ncclGetUniqueId");
    a.CommInitRank = (decltype(a.CommInitRank))dlsym(lib, "ncclCommInitRank");
    a.AllReduce = (decltype(a.AllReduce))dlsym(lib, "ncclAllReduce");
    a.CommDestroy = (decltype(a.CommDestroy))dlsym(lib, "ncclCommDestroy");
    a.GetErrorString = (decltype(a.GetErrorString))dlsym(lib, "ncclGetErrorString");
    if (!a.GetUniqueId || !a.CommInitRank || !a.AllReduce || !a.CommDestroy || !a.GetErrorString) {
        err = "libnccl is missing a required symbol";
        return err.c_str();
    }
    g_api = a;
    return nullptr;
}
}  // namespace nccl

static_assert(ARIANNA_MAX_MOVES == kMaxMoves, "header / kernel pool size mismatch");
static_assert(ARIANNA_MAX_SERIES == kMaxSeries, "header / kernel series size mismatch");
static_assert(ARIANNA_MAX_LADDER == kMaxLadder, "header / kernel ladder size mismatch");
static_assert(ARIANNA_MAX_HISTOGRAM_CELLS == kHistMaxCells, "header / kernel histogram size mismatch");
static_assert(kHistBlock >= kMaxLadder, "every group needs a thread in every CTA of histogram_kernel");
static_assert(sizeof(arianna_gradient_data) == 5 * sizeof(double), "gradient record layout");

struct arianna_handle {
    arianna_config cfg{};
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream = nullptr;   // D2H: trajectory frames / host-job downloads overlap the next sweep
    cudaStream_t h2d_stream = nullptr;    // H2D: host-job uploads (PCIe is full duplex: the two directions get a stream each)
    cudaEvent_t ev_snap = nullptr, ev_copy = nullptr;
    cudaEvent_t ev_job[4] = {nullptr, nullptr, nullptr, nullptr};   // [0,1] first/last upload, [2,3] first/last download of the last host job
    bool job_timed[2] = {false, false};
    int64_t job_bytes[2] = {0, 0};
    cudaStream_t coll_stream = nullptr;   // the tiny all-reduces of a series run beside the next sweep
    cudaEvent_t ev_coll_src = nullptr, ev_coll_done = nullptr;
    double *d_coll_series = nullptr;      // snapshot of d_series the asynchronous all-reduce works on
    int64_t coll_series_cap = 0;
    cudaEvent_t ev_t[4] = {nullptr, nullptr, nullptr, nullptr};   // device-time brackets: [0,1] last sweep/series/job, [2,3] last estimator pass
    bool timed[2] = {false, false};
    double *d_snap = nullptr;             // device snapshot of x the copy stream reads from
    int sm_count = 0, cc_major = 0, cc_minor = 0;
    size_t hbm_bytes = 0;
    size_t smem_per_sm = 0;
    int grid = 0;        // grid of the light streaming kernels: 8 CTAs per SM x SM count

    int64_t M = 0;
    bool f32 = false;               // ARIANNA_F32: the state lives in d_xf (4 B per chain), d_x is not allocated
    float *d_xf = nullptr;
    float *d_betas_f = nullptr;
    double lognorm_f32 = 0.0;       // log(2π·Float64(σ32·σ32))/2
    double *d_x = nullptr;
    uint32_t *d_acc = nullptr, *d_tot = nullptr;
    double *d_betas = nullptr;
    uint64_t *d_rng = nullptr;
    uint64_t *d_ki = nullptr;
    double *d_wi = nullptr, *d_fi = nullptr;
    double *d_partials = nullptr;
    unsigned int *d_ticket = nullptr;
    double *d_sums = nullptr;       // [kMaxOut]
    double *d_gd = nullptr;         // [kMaxMoves][5]
    double *d_pgmc_partials = nullptr;     // [n_learn][grid][5] of the estimator kernel (grow-only)
    size_t pgmc_partials_cap = 0;
    unsigned int *d_pgmc_ticket = nullptr; // [kMaxMoves]
    unsigned long long *d_csum = nullptr;  // [2 * kMaxMoves]
    m64::MathTables *d_tables = nullptr;   // exp/log tables of csrc/math64.cuh
    double *d_scratch = nullptr;    // e[] staging for get_state / dfma out
    size_t scratch_bytes = 0;

    double *d_series = nullptr;     // [series_cap][3] callback records of the last arianna_sweep_series call
    int64_t series_cap = 0, series_n = 0;
    double *d_series_partials = nullptr;   // single-move: [grid][n + 1][2]; multi-move: [grid][n][1 + n_moves] (grow-only)
    size_t series_partials_cap = 0;        // doubles
    uint8_t *d_cat_table = nullptr;        // multi-move pools: move index by the top 12 bits of the categorical word
    uint32_t cat_thr[kMaxMoves] = {};      // T_j = min(ceil(cp_j 2^32), 2^32 - 1)
    int cat_n = 0;                         // thresholds below 2^32 (the reachable ones)

    nccl::Comm comm = nullptr;      // optional: set by arianna_comm_init
    int comm_rank = 0, comm_size = 1;
    double *d_coll = nullptr;       // [kMaxMoves * 5] staging of the tiny all-reduces

    PoolParams pool{};
    DevTheta *d_theta = nullptr;    // device-resident θ block (on-device optimiser); mirrors `pool` when active
    bool theta_active = false;      // the kernels read θ from d_theta
    bool theta_dirty = false;       // the device copy is ahead of `pool` (arianna_params_sync pulls it)
    int64_t steps_done = 0;         // MC steps done per chain == draw index base == total_calls (single move)
    int64_t pgmc_samples = 0;       // estimator samples drawn per chain
    int64_t launches = 0;
    bool sums_valid = false;

    int ladder_L = 0;                      // replica exchange: rungs per ladder (0 = no ladder set)
    int64_t ex_rounds = 0;                 // exchange rounds done (the round index R of the next one)
    unsigned long long *d_xacc = nullptr;  // [kMaxLadder] accepted swaps per rung pair
    double *d_ladder = nullptr;            // [L] the β ladder
    double *d_ladder_partials = nullptr;   // [grid][L][1 + n_moves] of ladder_reduce_kernel
    double *d_ladder_sums = nullptr;       // [L][2 + n_moves]

    int hist_obs = -1;                     // on-device histogram: observable (-1 = none set)
    int hist_bins = 0, hist_groups = 0, hist_grid = 0;
    size_t hist_smem = 0;                  // dynamic shared memory of histogram_kernel: G·(n_bins + 3) u32
    double hist_lo = 0.0, hist_inv_w = 0.0;
    int64_t hist_samples = 0;              // accumulate calls since set / reset
    unsigned long long *d_hist_counts = nullptr;   // [G][n_bins + 3]
    double *d_hist_moments = nullptr;      // [G][3]
    double *d_hist_partials = nullptr;     // [hist_grid][G][3]
    std::string err;
};

static thread_local std::string g_create_err;

static int32_t fail(arianna_handle *h, int32_t code, const std::string &msg)
{
    if (h) h->err = msg; else g_create_err = msg;
    return code;
}

#define CU_TRY(h, expr)                                                                                       \
    do {                                                                                                      \
        cudaError_t _e = (expr);                                                                              \
        if (_e != cudaSuccess)                                                                                \
            return fail((h), _e == cudaErrorMemoryAllocation ? ARIANNA_ERR_NOMEM : ARIANNA_ERR_CUDA,          \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                                  \
    } while (0)

#define REQUIRE(h, cond, msg)                                                                                 \
    do {                                                                                                      \
        if (!(cond)) return fail((h), ARIANNA_ERR_INVALID, (msg));                                            \
    } while (0)

namespace {

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

double host_lognorm(double sigma)
{
    // log((2π)*(σ*σ))/2 with 2π = 6.283185307179586 (particle_1d.jl:53)
    const double s2 = sigma * sigma;
    return std::log(6.283185307179586 * s2) / 2.0;
}

// RN(1 / (2·(σ·σ))) for kernels.cuh:exact_div, or 0 when 2σ² is outside the range its error analysis covers
double host_inv2s2(double sigma)
{
    const double d = 2.0 * (sigma * sigma);
    return (d >= 0x1p-300 && d <= 0x1p300) ? 1.0 / d : 0.0;
}

// host pool -> device θ block (whole block; tiny)
int32_t push_theta(arianna_handle *h)
{
    DevTheta t{};
    for (int k = 0; k < kMaxMoves; ++k) {
        t.sigma[k] = h->pool.sigma[k];
        t.lognorm[k] = h->pool.lognorm[k];
        t.inv2s2[k] = h->pool.inv2s2[k];
    }
    if (!h->d_theta && cudaMalloc(&h->d_theta, sizeof(DevTheta)) != cudaSuccess) {
        cudaGetLastError();
        h->err = "device parameter block allocation failed";
        return ARIANNA_ERR_NOMEM;
    }
    // (synchronous on purpose: `t` lives on this stack frame)
    if (cudaMemcpyAsync(h->d_theta, &t, sizeof t, cudaMemcpyHostToDevice, h->stream) != cudaSuccess ||
        cudaStreamSynchronize(h->stream) != cudaSuccess) {
        h->err = std::string("device parameter upload: ") + cudaGetErrorString(cudaGetLastError());
        return ARIANNA_ERR_CUDA;
    }
    return ARIANNA_OK;
}

// device θ block -> host pool (synchronises); reports an optimiser step that left (0, ∞)
int32_t pull_theta(arianna_handle *h)
{
    if (!h->theta_active || !h->theta_dirty) return ARIANNA_OK;
    DevTheta t{};
    if (cudaMemcpyAsync(&t, h->d_theta, sizeof t, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
        cudaStreamSynchronize(h->stream) != cudaSuccess) {
        h->err = std::string("device parameter download: ") + cudaGetErrorString(cudaGetLastError());
        return ARIANNA_ERR_CUDA;
    }
    for (int k = 0; k < h->pool.n_moves; ++k) {
        h->pool.sigma[k] = t.sigma[k];
        h->pool.lognorm[k] = t.lognorm[k];
        h->pool.inv2s2[k] = t.inv2s2[k];
    }
    h->theta_dirty = false;
    if (t.bad) {
        h->err = "arianna_pgmc_update_device: an optimiser step left sigma outside (0, inf) (Normal(0, sigma) throws in the reference)";
        return ARIANNA_ERR_INVALID;
    }
    return ARIANNA_OK;
}

int grid_for(const arianna_handle *h, int64_t M, int ctas_per_sm)
{
    // at most `cap` CTAs, and every thread gets the same number of chains (to within one): with only a few chains
    // per thread a grid of exactly `cap` CTAs leaves a ragged last round (3.46 chains per thread = 13 % imbalance)
    const int64_t need = (M + kBlock - 1) / kBlock;
    const int64_t cap = (int64_t)h->sm_count * ctas_per_sm;
    if (need <= cap) return (int)need;
    const int64_t per_thread = (need + cap - 1) / cap;
    int64_t grid = (need + per_thread - 1) / per_thread;
    // ... rounded up to whole resident waves (one wave = ctas_per_sm / waves CTAs per SM; callers pass a multiple of
    // the SM count): a partial last wave costs more than a 2 % spread in chains per thread
    const int64_t wave = (int64_t)h->sm_count * 4;
    grid = (grid + wave - 1) / wave * wave;
    return (int)(grid < cap ? grid : cap);
}

size_t ensure_scratch(arianna_handle *h, size_t bytes)
{
    if (h->scratch_bytes >= bytes) return bytes;
    if (h->d_scratch) cudaFree(h->d_scratch);
    h->d_scratch = nullptr;
    h->scratch_bytes = 0;
    if (cudaMalloc(&h->d_scratch, bytes) != cudaSuccess) { cudaGetLastError(); return 0; }
    h->scratch_bytes = bytes;
    return bytes;
}

// Ziggurat tables of Julia's randn [EXT: stdlib Random, normal.jl]: Julia's literal constants, i.e. the randmtzig
// recursion evaluated exactly and rounded once (scripts/make_zig_tables.py) -- randmtzig.c's own double-precision recipe
// is 3e-12..3e-10 away from them.  With these defaults and Xoshiro(seed + c - 1) states (julia_rng.py, uploaded through
// arianna_set_rng_state) the XOSHIRO mode draws the very normals Julia draws (known answers of the Julia manual: tests/test_host.py, tests/test_oracle.py); the host may
// still override the tables (arianna_set_ziggurat_tables), e.g. for a Julia whose tables ever change.
#include "zig_tables_julia.inc"
void make_zig_tables(uint64_t *ki, double *wi, double *fi)
{
    std::memcpy(ki, kZigKiJulia, sizeof kZigKiJulia);
    std::memcpy(wi, kZigWiJulia, sizeof kZigWiJulia);
    std::memcpy(fi, kZigFiJulia, sizeof kZigFiJulia);
}

// Doubles per callback record: [Σe, Σ_c acc/tot per move, count]
inline int record_stride(const arianna_handle *h) { return 2 + h->pool.n_moves; }

// Categorical(weights) as integer thresholds + a bucket table (kernels_multi.cuh).  cp_j is summed in binary64 exactly
// as Distributions' scan does (`cp += p[i += 1]` [EXT]); cp <= w 2^-32  <=>  w >= ceil(cp 2^32).  Table entry of the
// bucket of the top 12 bits: k (no threshold inside) | 0x80 + j (exactly one, T_j) | 0xFF (several).
int build_cat_table(const double *weight, int nm, uint32_t *thr32, uint8_t *table)
{
    unsigned long long thr[kMaxMoves];
    double cp = weight[0];
    int n_reach = 0;
    for (int j = 0; j < kMaxMoves; ++j) thr32[j] = 0xffffffffu;
    for (int j = 0; j < nm - 1; ++j) {
        if (j > 0) cp = cp + weight[j];
        const double t = std::ceil(cp * 4294967296.0);
        thr[j] = t <= 0.0 ? 0ull : (t >= 4294967296.0 ? (1ull << 32) : (unsigned long long)t);
        if (thr[j] < (1ull << 32)) { thr32[j] = (uint32_t)thr[j]; n_reach = j + 1; }   // non-decreasing: a prefix
    }
    auto pick = [&](unsigned long long w) {
        int k = 0;
        for (int j = 0; j < nm - 1; ++j) k += (w >= thr[j]) ? 1 : 0;
        return k;
    };
    for (int b = 0; b < kCatBuckets; ++b) {
        const unsigned long long lo = (unsigned long long)b << 20, hi = lo + ((1ull << 20) - 1);
        const int k0 = pick(lo), k1 = pick(hi);
        table[b] = k0 == k1 ? (uint8_t)k0 : (k1 == k0 + 1 ? (uint8_t)(0x80 | k0) : (uint8_t)0xff);
    }
    return n_reach;
}

int32_t ensure_series_partials(arianna_handle *h, size_t n_doubles);

// Grid of the grid-stride kernels: an integer number of FULL resident waves (occupancy API x SM count x kGridWaves).
// One wave is the worst choice for these kernels: all CTAs start together, their warps run the Philox phase and the
// FP64 phase in lockstep (bursts of contention on one pipe at a time) and the SM drains unevenly at the end.  With
// 16 waves the hardware CTA scheduler staggers the phases and balances the tail; measured on M = 2^27, K = 10:
// 1 / 2 / 4 / 8 / 16 / 32 / 64 / 256 waves -> 5.57 / 5.28 / 5.15 / 5.09 / 5.06 / 5.07 / 5.11 / 5.36 ms.
constexpr int kGridWaves = 16;
template <typename K>
int wave_grid(const arianna_handle *h, K kernel, size_t smem, int64_t M)
{
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kBlock, smem) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        per_sm = 2;
    }
    if (per_sm > 8) per_sm = 8;
    return grid_for(h, M, per_sm * kGridWaves);
}

// the largest grid wave_grid() can return: what the per-CTA partial buffers are sized for
int max_wave_grid(const arianna_handle *h) { return h->sm_count * 8 * kGridWaves; }

int32_t ensure_series_partials(arianna_handle *h, size_t n_doubles)
{
    if (h->series_partials_cap >= n_doubles) return ARIANNA_OK;
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) cudaGetLastError();
    cudaFree(h->d_series_partials);
    h->d_series_partials = nullptr;
    h->series_partials_cap = 0;
    if (cudaMalloc(&h->d_series_partials, sizeof(double) * n_doubles) != cudaSuccess) {
        cudaGetLastError();
        h->err = "series partials allocation failed";
        return ARIANNA_ERR_NOMEM;
    }
    h->series_partials_cap = n_doubles;
    return ARIANNA_OK;
}

template <typename F>
int32_t dispatch_pot(int pot, F &&f)
{
    switch (pot) {
    case POT_HARMONIC: return f(std::integral_constant<int, POT_HARMONIC>{});
    case POT_QUARTIC: return f(std::integral_constant<int, POT_QUARTIC>{});
    default: return f(std::integral_constant<int, POT_DOUBLE_WELL>{});
    }
}

// f(kernel) with the histogram_kernel instantiation of the handle's element type, the observable and the potential
template <typename F>
int32_t dispatch_histogram(const arianna_handle *h, int observable, F &&f)
{
    auto pick = [&](auto zero) -> int32_t {
        using T = decltype(zero);
        if (observable == ARIANNA_OBS_X) return f(histogram_kernel<T, kHistPosition>);
        return dispatch_pot(h->cfg.potential, [&](auto pot) -> int32_t { return f(histogram_kernel<T, decltype(pot)::value>); });
    };
    return h->f32 ? pick(0.0f) : pick(0.0);
}

}  // namespace

extern "C" {

uint32_t arianna_abi_version(void) { return ARIANNA_ABI_VERSION; }

const char *arianna_last_error(const arianna_handle *h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int32_t arianna_create(const arianna_config *cfg, arianna_handle **out)
{
    if (!cfg || !out) return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: NULL argument");
    *out = nullptr;
    if (cfg->struct_size != sizeof(arianna_config))
        return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: struct_size does not match this ABI");
    if (cfg->n_chains < 1) return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: n_chains must be >= 1");
    if (cfg->n_moves < 1 || cfg->n_moves > ARIANNA_MAX_MOVES)
        return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: n_moves must be in 1..ARIANNA_MAX_MOVES");
    if (cfg->potential < 0 || cfg->potential > ARIANNA_POT_DOUBLE_WELL)
        return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: unknown potential");
    if (cfg->rng_mode != ARIANNA_RNG_PHILOX && cfg->rng_mode != ARIANNA_RNG_XOSHIRO)
        return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: unknown rng_mode");
    if (cfg->arith_mode != ARIANNA_ARITH_EXACT && cfg->arith_mode != ARIANNA_ARITH_FAST)
        return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: unknown arith_mode");
    if (cfg->dtype != ARIANNA_F64 && cfg->dtype != ARIANNA_F32)
        return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: unknown dtype");
    if (cfg->dtype == ARIANNA_F32 && (cfg->n_moves != 1 || cfg->rng_mode != ARIANNA_RNG_PHILOX))
        return fail(nullptr, ARIANNA_ERR_UNSUPPORTED,
                    "arianna_create: Float32 ensembles support single-move pools with the native Philox stream (or replay)");
    double wsum = 0.0;
    for (int k = 0; k < cfg->n_moves; ++k) {
        if (!(cfg->sigma[k] > 0.0) || !std::isfinite(cfg->sigma[k]))
            return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: sigma must be finite and > 0");
        if (!(cfg->weight[k] >= 0.0))
            return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: weights must be >= 0");
        wsum += cfg->weight[k];
    }
    // Distributions.Categorical rejects probability vectors that do not sum to one [EXT] (metropolis.jl:206)
    if (std::fabs(wsum - 1.0) > 1e-10 * std::sqrt((double)cfg->n_moves))
        return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: move weights must sum to 1 (Categorical)");

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, ARIANNA_ERR_NO_DEVICE,
                    "arianna_create: no CUDA device visible; libarianna_cuda has no CPU fallback");
    }
    int dev = cfg->device;
    if (dev < 0) {
        if (cudaGetDevice(&dev) != cudaSuccess) return fail(nullptr, ARIANNA_ERR_CUDA, "cudaGetDevice failed");
    }
    if (dev >= ndev) return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_create: device ordinal out of range");

    arianna_handle *h = new (std::nothrow) arianna_handle();
    if (!h) return fail(nullptr, ARIANNA_ERR_NOMEM, "arianna_create: host allocation failed");
    h->cfg = *cfg;
    if (h->cfg.n_chains_total <= 0) h->cfg.n_chains_total = cfg->n_chains;
    h->device = dev;
    h->M = cfg->n_chains;
    DeviceGuard guard(dev);

    auto bail = [&](int32_t code, const std::string &msg) {
        g_create_err = msg;
        arianna_destroy(h);
        return code;
    };
#define CU_CREATE(expr)                                                                                       \
    do {                                                                                                      \
        cudaError_t _e = (expr);                                                                              \
        if (_e != cudaSuccess)                                                                                \
            return bail(_e == cudaErrorMemoryAllocation ? ARIANNA_ERR_NOMEM : ARIANNA_ERR_CUDA,               \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                                  \
    } while (0)

    cudaDeviceProp prop{};
    CU_CREATE(cudaGetDeviceProperties(&prop, dev));
    h->sm_count = prop.multiProcessorCount;
    h->cc_major = prop.major;
    h->cc_minor = prop.minor;
    h->hbm_bytes = prop.totalGlobalMem;
    h->smem_per_sm = prop.sharedMemPerMultiprocessor;
    if (prop.major != 10)
        return bail(ARIANNA_ERR_UNSUPPORTED, "arianna_create: this library is built for sm_100a (B200) only");
    // persistent-style grid: 8 resident CTAs of 256 threads per SM cover the 64-warp SM limit
    h->grid = grid_for(h, h->M, 8);
    if (cfg->stream) {
        h->stream = (cudaStream_t)cfg->stream;
    } else {
        CU_CREATE(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        h->own_stream = true;
    }

    const int nm = cfg->n_moves;
    h->pool.n_moves = nm;
    for (int k = 0; k < kMaxMoves; ++k) {
        h->pool.sigma[k] = k < nm ? cfg->sigma[k] : 1.0;
        h->pool.weight[k] = k < nm ? cfg->weight[k] : 0.0;
        h->pool.lognorm[k] = host_lognorm(h->pool.sigma[k]);
        h->pool.inv2s2[k] = host_inv2s2(h->pool.sigma[k]);
    }

    h->f32 = cfg->dtype == ARIANNA_F32;
    if (h->f32) {
        CU_CREATE(cudaMalloc(&h->d_xf, sizeof(float) * h->M));
        CU_CREATE(cudaMemsetAsync(h->d_xf, 0, sizeof(float) * h->M, h->stream));
        const float s32 = (float)h->pool.sigma[0], s2 = s32 * s32;
        h->lognorm_f32 = std::log(6.283185307179586 * (double)s2) / 2.0;
    } else {
        CU_CREATE(cudaMalloc(&h->d_x, sizeof(double) * h->M));
    }
    CU_CREATE(cudaMalloc(&h->d_acc, sizeof(uint32_t) * h->M * nm));
    CU_CREATE(cudaMemsetAsync(h->d_acc, 0, sizeof(uint32_t) * h->M * nm, h->stream));
    if (nm > 1) {
        CU_CREATE(cudaMalloc(&h->d_tot, sizeof(uint32_t) * h->M * nm));
        CU_CREATE(cudaMemsetAsync(h->d_tot, 0, sizeof(uint32_t) * h->M * nm, h->stream));
        std::vector<uint8_t> table(kCatBuckets);
        h->cat_n = build_cat_table(h->pool.weight, nm, h->cat_thr, table.data());
        CU_CREATE(cudaMalloc(&h->d_cat_table, kCatBuckets));
        CU_CREATE(cudaMemcpyAsync(h->d_cat_table, table.data(), kCatBuckets, cudaMemcpyHostToDevice, h->stream));
        CU_CREATE(cudaStreamSynchronize(h->stream));
    }
    if (!h->f32) CU_CREATE(cudaMemsetAsync(h->d_x, 0, sizeof(double) * h->M, h->stream));
    CU_CREATE(cudaMalloc(&h->d_partials, sizeof(double) * (size_t)max_wave_grid(h) * kMaxOut));
    CU_CREATE(cudaMalloc(&h->d_ticket, sizeof(unsigned int)));
    CU_CREATE(cudaMemsetAsync(h->d_ticket, 0, sizeof(unsigned int), h->stream));
    CU_CREATE(cudaMalloc(&h->d_sums, sizeof(double) * kMaxOut));
    CU_CREATE(cudaMemsetAsync(h->d_sums, 0, sizeof(double) * kMaxOut, h->stream));
    CU_CREATE(cudaMalloc(&h->d_gd, sizeof(double) * kMaxMoves * 5));
    CU_CREATE(cudaMemsetAsync(h->d_gd, 0, sizeof(double) * kMaxMoves * 5, h->stream));
    CU_CREATE(cudaMalloc(&h->d_csum, sizeof(unsigned long long) * 2 * kMaxMoves));
    {
        m64::MathTables T;
        m64::build_math_tables(T);
        CU_CREATE(cudaMalloc(&h->d_tables, sizeof T));
        CU_CREATE(cudaMemcpyAsync(h->d_tables, &T, sizeof T, cudaMemcpyHostToDevice, h->stream));
        CU_CREATE(cudaStreamSynchronize(h->stream));
    }

    if (cfg->rng_mode == ARIANNA_RNG_XOSHIRO) {
        CU_CREATE(cudaMalloc(&h->d_rng, sizeof(uint64_t) * 4 * h->M));
        CU_CREATE(cudaMemsetAsync(h->d_rng, 0, sizeof(uint64_t) * 4 * h->M, h->stream));
        CU_CREATE(cudaMalloc(&h->d_ki, sizeof(uint64_t) * 256));
        CU_CREATE(cudaMalloc(&h->d_wi, sizeof(double) * 256));
        CU_CREATE(cudaMalloc(&h->d_fi, sizeof(double) * 256));
        uint64_t ki[256];
        double wi[256], fi[256];
        make_zig_tables(ki, wi, fi);
        CU_CREATE(cudaMemcpyAsync(h->d_ki, ki, sizeof ki, cudaMemcpyHostToDevice, h->stream));
        CU_CREATE(cudaMemcpyAsync(h->d_wi, wi, sizeof wi, cudaMemcpyHostToDevice, h->stream));
        CU_CREATE(cudaMemcpyAsync(h->d_fi, fi, sizeof fi, cudaMemcpyHostToDevice, h->stream));
        CU_CREATE(cudaStreamSynchronize(h->stream));  // stack tables must outlive the copies
    }
    // opt in to large dynamic shared memory for the multi-move kernels (2 * n_moves * 256 * 4 B <= 32 KB: default ok)
    CU_CREATE(cudaStreamSynchronize(h->stream));
#undef CU_CREATE
    *out = h;
    return ARIANNA_OK;
}

int32_t arianna_destroy(arianna_handle *h)
{
    if (!h) return ARIANNA_OK;
    DeviceGuard guard(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    cudaFree(h->d_xf); cudaFree(h->d_betas_f);
    cudaFree(h->d_x); cudaFree(h->d_acc); cudaFree(h->d_tot); cudaFree(h->d_betas); cudaFree(h->d_rng);
    cudaFree(h->d_ki); cudaFree(h->d_wi); cudaFree(h->d_fi); cudaFree(h->d_partials); cudaFree(h->d_ticket);
    cudaFree(h->d_sums); cudaFree(h->d_gd); cudaFree(h->d_csum); cudaFree(h->d_scratch); cudaFree(h->d_tables);
    cudaFree(h->d_series); cudaFree(h->d_series_partials); cudaFree(h->d_cat_table);
    cudaFree(h->d_pgmc_partials); cudaFree(h->d_pgmc_ticket); cudaFree(h->d_theta);
    cudaFree(h->d_xacc); cudaFree(h->d_ladder); cudaFree(h->d_ladder_partials); cudaFree(h->d_ladder_sums);
    cudaFree(h->d_hist_counts); cudaFree(h->d_hist_moments); cudaFree(h->d_hist_partials);
    if (h->coll_stream) cudaStreamSynchronize(h->coll_stream);
    if (h->comm) { nccl::g_api.CommDestroy(h->comm); h->comm = nullptr; }
    cudaFree(h->d_coll);
    if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
    if (h->h2d_stream) { cudaStreamSynchronize(h->h2d_stream); cudaStreamDestroy(h->h2d_stream); }
    if (h->coll_stream) { cudaStreamSynchronize(h->coll_stream); cudaStreamDestroy(h->coll_stream); }
    cudaFree(h->d_coll_series);
    if (h->ev_coll_src) cudaEventDestroy(h->ev_coll_src);
    if (h->ev_coll_done) cudaEventDestroy(h->ev_coll_done);
    for (auto &e : h->ev_job) if (e) cudaEventDestroy(e);
    for (auto &e : h->ev_t) if (e) cudaEventDestroy(e);
    if (h->ev_snap) cudaEventDestroy(h->ev_snap);
    if (h->ev_copy) cudaEventDestroy(h->ev_copy);
    cudaFree(h->d_snap);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    cudaGetLastError();
    delete h;
    return ARIANNA_OK;
}

int32_t arianna_set_state(arianna_handle *h, const double *x)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, x != nullptr, "arianna_set_state: x is NULL");
    DeviceGuard guard(h->device);
    if (h->f32) {        // Float64 view of a Float32 ensemble: upload, round to nearest
        if (!ensure_scratch(h, sizeof(double) * h->M)) return fail(h, ARIANNA_ERR_NOMEM, "arianna_set_state: scratch allocation failed");
        CU_TRY(h, cudaMemcpyAsync(h->d_scratch, x, sizeof(double) * h->M, cudaMemcpyHostToDevice, h->stream));
        f32_from_f64_kernel<<<h->grid, kBlock, 0, h->stream>>>(h->d_xf, h->d_scratch, h->M);
        CU_TRY(h, cudaGetLastError());
        ++h->launches;
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        h->sums_valid = false;
        return ARIANNA_OK;
    }
    CU_TRY(h, cudaMemcpyAsync(h->d_x, x, sizeof(double) * h->M, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    h->sums_valid = false;
    return ARIANNA_OK;
}

int32_t arianna_init_synthetic(arianna_handle *h, int64_t seed)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    if (h->f32)
        init_kernel_f32<<<h->grid, kBlock, 0, h->stream>>>(h->d_xf, h->M, (uint64_t)(seed + h->cfg.chain_offset));
    else
    init_kernel<<<h->grid, kBlock, 0, h->stream>>>(h->d_x, h->M, (uint64_t)(seed + h->cfg.chain_offset));
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    h->sums_valid = false;
    return ARIANNA_OK;
}

int32_t arianna_get_state(arianna_handle *h, double *x, double *e)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    if (h->f32) {        // Float64 view of a Float32 ensemble: widen exactly on the device, then download
        if (!ensure_scratch(h, sizeof(double) * h->M)) return fail(h, ARIANNA_ERR_NOMEM, "arianna_get_state: scratch allocation failed");
        double *out[2] = {x, e};
        for (int w = 0; w < 2; ++w) {
            if (!out[w]) continue;
            f64_from_f32_kernel<<<h->grid, kBlock, 0, h->stream>>>(h->d_scratch, h->d_xf, h->M, h->cfg.potential, w);
            CU_TRY(h, cudaGetLastError());
            ++h->launches;
            CU_TRY(h, cudaMemcpyAsync(out[w], h->d_scratch, sizeof(double) * h->M, cudaMemcpyDeviceToHost, h->stream));
        }
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        return ARIANNA_OK;
    }
    if (x) CU_TRY(h, cudaMemcpyAsync(x, h->d_x, sizeof(double) * h->M, cudaMemcpyDeviceToHost, h->stream));
    if (e) {
        if (!ensure_scratch(h, sizeof(double) * h->M))
            return fail(h, ARIANNA_ERR_NOMEM, "arianna_get_state: scratch allocation failed");
        energy_kernel<<<h->grid, kBlock, 0, h->stream>>>(h->d_x, h->d_scratch, h->M, h->cfg.potential);
        CU_TRY(h, cudaGetLastError());
        ++h->launches;
        CU_TRY(h, cudaMemcpyAsync(e, h->d_scratch, sizeof(double) * h->M, cudaMemcpyDeviceToHost, h->stream));
    }
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

int32_t arianna_set_state_f32(arianna_handle *h, const float *x)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, x != nullptr, "arianna_set_state_f32: x is NULL");
    if (!h->f32) return fail(h, ARIANNA_ERR_UNSUPPORTED, "arianna_set_state_f32: the handle was not created with ARIANNA_F32");
    DeviceGuard guard(h->device);
    CU_TRY(h, cudaMemcpyAsync(h->d_xf, x, sizeof(float) * h->M, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    h->sums_valid = false;
    return ARIANNA_OK;
}

int32_t arianna_get_state_f32(arianna_handle *h, float *x, float *e)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (!h->f32) return fail(h, ARIANNA_ERR_UNSUPPORTED, "arianna_get_state_f32: the handle was not created with ARIANNA_F32");
    DeviceGuard guard(h->device);
    if (x) CU_TRY(h, cudaMemcpyAsync(x, h->d_xf, sizeof(float) * h->M, cudaMemcpyDeviceToHost, h->stream));
    if (e) {
        if (!ensure_scratch(h, sizeof(float) * h->M)) return fail(h, ARIANNA_ERR_NOMEM, "arianna_get_state_f32: scratch allocation failed");
        energy_kernel_f32<<<h->grid, kBlock, 0, h->stream>>>(h->d_xf, reinterpret_cast<float *>(h->d_scratch), h->M, h->cfg.potential);
        CU_TRY(h, cudaGetLastError());
        ++h->launches;
        CU_TRY(h, cudaMemcpyAsync(e, h->d_scratch, sizeof(float) * h->M, cudaMemcpyDeviceToHost, h->stream));
    }
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

// Device-time bracket `which` (0 sweeps, 1 estimator) on the compute stream; read by arianna_timing.
static void time_mark(arianna_handle *h, int which, bool begin)
{
    cudaEvent_t &e = h->ev_t[2 * which + (begin ? 0 : 1)];
    if (!e && cudaEventCreate(&e) != cudaSuccess) { cudaGetLastError(); e = nullptr; return; }
    if (cudaEventRecord(e, h->stream) != cudaSuccess) { cudaGetLastError(); return; }
    if (!begin) h->timed[which] = true;
}

// The copy stream and its two events (trajectory frames, pipelined host jobs), created on first use.
static int32_t ensure_copy_stream(arianna_handle *h)
{
    if (h->copy_stream) return ARIANNA_OK;
    CU_TRY(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CU_TRY(h, cudaStreamCreateWithFlags(&h->h2d_stream, cudaStreamNonBlocking));
    for (auto &e : h->ev_job) CU_TRY(h, cudaEventCreate(&e));
    CU_TRY(h, cudaEventCreateWithFlags(&h->ev_snap, cudaEventDisableTiming));
    CU_TRY(h, cudaEventCreateWithFlags(&h->ev_copy, cudaEventDisableTiming));
    CU_TRY(h, cudaEventRecord(h->ev_copy, h->copy_stream));
    return ARIANNA_OK;
}

int32_t arianna_get_state_async(arianna_handle *h, double *x_pinned)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, x_pinned != nullptr, "arianna_get_state_async: destination is NULL");
    if (h->f32) return fail(h, ARIANNA_ERR_UNSUPPORTED, "arianna_get_state_async: Float64 ensembles only (use arianna_get_state_f32)");
    DeviceGuard guard(h->device);
    int32_t rc = ensure_copy_stream(h);
    if (rc) return rc;
    if (!h->d_snap) CU_TRY(h, cudaMalloc(&h->d_snap, sizeof(double) * h->M));
    // snapshot x on the compute stream (D2D, ~0.1 ms/GiB-scale) so the next sweep can start at once, then drain the
    // snapshot over PCIe on the copy stream; the previous frame must have left the snapshot first
    CU_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_copy, 0));
    CU_TRY(h, cudaMemcpyAsync(h->d_snap, h->d_x, sizeof(double) * h->M, cudaMemcpyDeviceToDevice, h->stream));
    CU_TRY(h, cudaEventRecord(h->ev_snap, h->stream));
    CU_TRY(h, cudaStreamWaitEvent(h->copy_stream, h->ev_snap, 0));
    CU_TRY(h, cudaMemcpyAsync(x_pinned, h->d_snap, sizeof(double) * h->M, cudaMemcpyDeviceToHost, h->copy_stream));
    CU_TRY(h, cudaEventRecord(h->ev_copy, h->copy_stream));
    return ARIANNA_OK;
}

// Page-locked host memory for hosts without a CUDA binding of their own (the Julia shim): the buffers
// arianna_run_host_job / arianna_get_state_async need for their copies to be asynchronous.  write_combined: memory the
// host only writes and the GPU reads (x_in) -- not snooped, faster over PCIe, very slow to read back on the CPU.
int32_t arianna_host_alloc(int64_t bytes, int32_t write_combined, void **out)
{
    if (!out || bytes <= 0) return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_host_alloc: bad arguments");
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, (size_t)bytes, cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0));
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, e == cudaErrorMemoryAllocation ? ARIANNA_ERR_NOMEM : ARIANNA_ERR_CUDA,
                    std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
    }
    return ARIANNA_OK;
}

int32_t arianna_host_free(void *p)
{
    if (!p) return ARIANNA_OK;
    cudaError_t e = cudaFreeHost(p);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(nullptr, ARIANNA_ERR_CUDA, std::string("cudaFreeHost: ") + cudaGetErrorString(e)); }
    return ARIANNA_OK;
}

int32_t arianna_copy_wait(arianna_handle *h)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (!h->copy_stream) return ARIANNA_OK;
    DeviceGuard guard(h->device);
    CU_TRY(h, cudaEventSynchronize(h->ev_copy));
    return ARIANNA_OK;
}

int32_t arianna_set_beta(arianna_handle *h, double beta)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    h->cfg.beta = beta;
    if (h->d_betas) { cudaStreamSynchronize(h->stream); cudaFree(h->d_betas); h->d_betas = nullptr; }
    if (h->d_betas_f) { cudaStreamSynchronize(h->stream); cudaFree(h->d_betas_f); h->d_betas_f = nullptr; }
    return ARIANNA_OK;
}

int32_t arianna_set_betas(arianna_handle *h, const double *betas)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, betas != nullptr, "arianna_set_betas: betas is NULL");
    DeviceGuard guard(h->device);
    if (h->f32) {        // Particle{Float32}.β is a Float32
        if (!h->d_betas_f) CU_TRY(h, cudaMalloc(&h->d_betas_f, sizeof(float) * h->M));
        if (!ensure_scratch(h, sizeof(double) * h->M)) return fail(h, ARIANNA_ERR_NOMEM, "arianna_set_betas: scratch allocation failed");
        CU_TRY(h, cudaMemcpyAsync(h->d_scratch, betas, sizeof(double) * h->M, cudaMemcpyHostToDevice, h->stream));
        f32_from_f64_kernel<<<h->grid, kBlock, 0, h->stream>>>(h->d_betas_f, h->d_scratch, h->M);
        CU_TRY(h, cudaGetLastError());
        ++h->launches;
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        return ARIANNA_OK;
    }
    if (!h->d_betas) CU_TRY(h, cudaMalloc(&h->d_betas, sizeof(double) * h->M));
    CU_TRY(h, cudaMemcpyAsync(h->d_betas, betas, sizeof(double) * h->M, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

int32_t arianna_set_params(arianna_handle *h, int32_t move_id, const double *theta, int32_t P,
                           const double *log_norm)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, move_id >= 0 && move_id < h->pool.n_moves, "arianna_set_params: move_id out of range");
    REQUIRE(h, theta != nullptr && P == 1, "arianna_set_params: StandardGaussian has exactly one parameter (σ)");
    REQUIRE(h, std::isfinite(theta[0]) && theta[0] > 0.0, "arianna_set_params: σ must be finite and > 0 (Normal(0, σ))");
    // kernel parameters are passed by value at launch: updating the host copy is all that is needed
    h->pool.sigma[move_id] = theta[0];
    h->pool.lognorm[move_id] = log_norm ? *log_norm : host_lognorm(theta[0]);
    h->pool.inv2s2[move_id] = host_inv2s2(theta[0]);
    if (h->theta_active) {          // keep the device-resident block coherent (pull first: other moves may be ahead there)
        DeviceGuard guard(h->device);
        const double s0 = h->pool.sigma[move_id], l0 = h->pool.lognorm[move_id], i0 = h->pool.inv2s2[move_id];
        int32_t rc = pull_theta(h);
        if (rc) return rc;
        h->pool.sigma[move_id] = s0; h->pool.lognorm[move_id] = l0; h->pool.inv2s2[move_id] = i0;
        rc = push_theta(h);
        if (rc) return rc;
    }
    if (h->f32) {
        const float s32 = (float)theta[0], s2 = s32 * s32;
        h->lognorm_f32 = log_norm ? *log_norm : std::log(6.283185307179586 * (double)s2) / 2.0;
    }
    return ARIANNA_OK;
}

int32_t arianna_get_params(arianna_handle *h, int32_t move_id, double *theta, int32_t P)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, move_id >= 0 && move_id < h->pool.n_moves, "arianna_get_params: move_id out of range");
    REQUIRE(h, theta != nullptr && P == 1, "arianna_get_params: StandardGaussian has exactly one parameter (σ)");
    {
        DeviceGuard guard(h->device);
        const int32_t rc = pull_theta(h);       // the on-device optimiser may be ahead of the host copy
        if (rc) return rc;
    }
    theta[0] = h->pool.sigma[move_id];
    return ARIANNA_OK;
}

static int32_t launch_callback_reduce(arianna_handle *h)
{
    if (h->f32) {
        callback_reduce_f32_kernel<<<h->grid, kBlock, 0, h->stream>>>(h->d_xf, h->d_acc, h->M, h->steps_done, h->cfg.potential,
                                                                      h->d_partials, h->d_ticket, h->d_sums);
        CU_TRY(h, cudaGetLastError());
        ++h->launches;
        h->sums_valid = true;
        return ARIANNA_OK;
    }
    ReduceParams rp{h->d_x, h->d_acc, h->d_tot, h->M, h->steps_done, h->pool.n_moves, h->cfg.potential,
                    h->d_partials, h->d_ticket, h->d_sums};
    callback_reduce_kernel<<<h->grid, kBlock, 0, h->stream>>>(rp);
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    h->sums_valid = true;
    return ARIANNA_OK;
}

// One launch of the multi-move sweep over chains [off, off + m): n_int intervals of K[i] steps starting at MC step t0,
// with a callback record after each when `out` != NULL (records go to out[0 .. n_int) x record_stride, added when
// `accumulate`; the last one is also copied to `sums` when given).  Asynchronous on h->stream.
static int32_t launch_multi(arianna_handle *h, int64_t off, int64_t m, int64_t t0, int n_int, const int64_t *K,
                            double *out, double *sums, int accumulate)
{
    const bool exact = h->cfg.arith_mode == ARIANNA_ARITH_EXACT;
    const int nm = h->pool.n_moves;
    MultiParams mp{};
    mp.x = h->d_x + off; mp.acc = h->d_acc + off; mp.tot = h->d_tot + off;
    mp.betas = h->d_betas ? h->d_betas + off : nullptr; mp.beta = h->cfg.beta;
    // the per-move counter arrays are [n_moves][M] of the WHOLE handle: a slice keeps that row pitch
    mp.M = m; mp.t0 = t0;
    mp.sid0 = (uint64_t)(h->cfg.seed + h->cfg.chain_offset + off);
    mp.tables = h->d_tables;
    mp.cat_table = h->d_cat_table;
    for (int j = 0; j < kMaxMoves; ++j) mp.cat_thr[j] = h->cat_thr[j];
    mp.cat_n = h->cat_n;
    mp.pool = h->pool;
    mp.theta = h->theta_active ? h->d_theta : nullptr;
    mp.n_int = n_int; mp.record = out ? 1 : 0;
    bool even = (t0 & 1) == 0;
    for (int i = 0; i < n_int; ++i) {
        mp.K[i] = (int)K[i];
        even = even && K[i] > 0 && (K[i] & 1) == 0;
    }
    mp.K[n_int] = 0;
    mp.even = even ? 1 : 0;
    mp.pitch = h->M;
    // two counter buffers (prefetch of the next chain's counters) when that still leaves kMultiMinBlocks CTAs per SM
    mp.dbuf = multi_smem_bytes(nm, n_int, mp.record, 1) + 1024 <= h->smem_per_sm / kMultiMinBlocks ? 1 : 0;
    const size_t smem = multi_smem_bytes(nm, n_int, mp.record, mp.dbuf);
    int grid = 0;
    int32_t rc = dispatch_pot(h->cfg.potential, [&](auto pot) -> int32_t {
        constexpr int POT = decltype(pot)::value;
        auto go = [&](auto kernel) -> int32_t {
            CU_TRY(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            grid = wave_grid(h, kernel, smem, m);
            if (mp.record) {
                const int32_t r = ensure_series_partials(h, (size_t)grid * n_int * (1 + nm));
                if (r) return r;
                mp.partials = h->d_series_partials;
            }
            kernel<<<grid, kBlock, smem, h->stream>>>(mp);
            return ARIANNA_OK;
        };
        if (h->d_betas)
            return exact ? go(sweep_multi_kernel<POT, ARITH_EXACT, true>) : go(sweep_multi_kernel<POT, ARITH_FAST, true>);
        return exact ? go(sweep_multi_kernel<POT, ARITH_EXACT, false>) : go(sweep_multi_kernel<POT, ARITH_FAST, false>);
    });
    if (rc) return rc;
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    if (mp.record) {
        series_fold_multi_kernel<<<n_int, kBlock, 0, h->stream>>>(h->d_series_partials, grid, n_int, nm, m, out, sums,
                                                                 accumulate);
        CU_TRY(h, cudaGetLastError());
        ++h->launches;
    }
    return ARIANNA_OK;
}

int32_t arianna_sweep(arianna_handle *h, int64_t K, uint32_t flags)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, K >= 0, "arianna_sweep: K must be >= 0");
    REQUIRE(h, h->steps_done + K <= 0xFFFFFFFFll, "arianna_sweep: per-chain counters are 32-bit (2^32-1 steps max)");
    DeviceGuard guard(h->device);
    const bool multi = h->pool.n_moves > 1;
    const bool want_reduce = (flags & ARIANNA_SWEEP_REDUCE) != 0;
    if (K == 0) return want_reduce ? launch_callback_reduce(h) : ARIANNA_OK;
    if (h->f32 || h->cfg.rng_mode != ARIANNA_RNG_PHILOX) {           // (these paths pass θ by value)
        const int32_t rcp = pull_theta(h);
        if (rcp) return rcp;
    }
    const size_t smem = multi ? sizeof(uint32_t) * 2 * h->pool.n_moves * kBlock : 0;
    const bool exact = h->cfg.arith_mode == ARIANNA_ARITH_EXACT;
    time_mark(h, 0, true);

    if (h->f32) {
        F32Params fp{};
        fp.x = h->d_xf; fp.acc = h->d_acc; fp.betas = h->d_betas_f; fp.beta = (float)h->cfg.beta;
        fp.M = h->M; fp.K = K; fp.t0 = h->steps_done;
        fp.sid0 = (uint64_t)(h->cfg.seed + h->cfg.chain_offset);
        fp.sigma = (float)h->pool.sigma[0]; fp.lognorm = h->lognorm_f32;
        fp.reduce = want_reduce ? 1 : 0;
        fp.partials = h->d_partials; fp.ticket = h->d_ticket; fp.sums = h->d_sums;
        fp.tables = h->d_tables;
        const int32_t rc = dispatch_pot(h->cfg.potential, [&](auto pot) -> int32_t {
            constexpr int POT = decltype(pot)::value;
            auto go = [&](auto kernel) -> int32_t {
                kernel<<<wave_grid(h, kernel, 0, h->M), kBlock, 0, h->stream>>>(fp);
                return ARIANNA_OK;
            };
            return exact ? go(sweep_f32_kernel<POT, ARITH_EXACT>) : go(sweep_f32_kernel<POT, ARITH_FAST>);
        });
        if (rc) return rc;
        CU_TRY(h, cudaGetLastError());
        ++h->launches;
        h->steps_done += K;
        h->sums_valid = want_reduce;
        time_mark(h, 0, false);
        return ARIANNA_OK;
    }
    if (h->cfg.rng_mode == ARIANNA_RNG_PHILOX && multi) {
        // multi-move pools: the record (when asked for) is reduced inside the sweep, per move
        REQUIRE(h, K < (int64_t(1) << 31), "arianna_sweep: K must be < 2^31");
        const int32_t rc = launch_multi(h, 0, h->M, h->steps_done, 1, &K, want_reduce ? h->d_sums : nullptr, nullptr, 0);
        if (rc) return rc;
        h->steps_done += K;
        h->sums_valid = want_reduce;
        time_mark(h, 0, false);
        return ARIANNA_OK;
    }
    if (h->cfg.rng_mode == ARIANNA_RNG_PHILOX) {

        SweepParams sp{};
        sp.x = h->d_x; sp.acc = h->d_acc; sp.tot = h->d_tot; sp.betas = h->d_betas; sp.beta = h->cfg.beta;
        sp.M = h->M; sp.K = K; sp.t0 = h->steps_done;
        sp.sid0 = (uint64_t)(h->cfg.seed + h->cfg.chain_offset);
        sp.reduce = want_reduce ? 1 : 0;
        sp.partials = h->d_partials; sp.ticket = h->d_ticket; sp.sums = h->d_sums;
        sp.tables = h->d_tables;
        sp.pool = h->pool;
        sp.theta = h->theta_active ? h->d_theta : nullptr;
        // the Philox sweep keeps its math tables in dynamic shared memory (one pinned base register, kernels.cuh)
        const size_t psmem = sizeof(m64::MathTables);
        auto launch = [&](auto kernel) -> int32_t {
            if (psmem > 48 * 1024)
                CU_TRY(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem));
            kernel<<<wave_grid(h, kernel, psmem, h->M), kBlock, psmem, h->stream>>>(sp);
            return ARIANNA_OK;
        };
        const int32_t rc = dispatch_pot(h->cfg.potential, [&](auto pot) -> int32_t {
            constexpr int POT = decltype(pot)::value;
            const bool generic = h->d_betas || h->theta_active;     // per-chain β and / or σ read from the device
            if (exact) {
                if (generic) return launch(sweep_philox_kernel<POT, ARITH_EXACT>);
                return launch(sweep_philox_kernel<POT, ARITH_EXACT, false, false>);
            }
            if (generic) return launch(sweep_philox_kernel<POT, ARITH_FAST>);
            return launch(sweep_philox_kernel<POT, ARITH_FAST, false, false>);
        });
        if (rc) return rc;
    } else {
        XoshiroParams xp{};
        xp.x = h->d_x; xp.acc = h->d_acc; xp.tot = h->d_tot; xp.betas = h->d_betas; xp.beta = h->cfg.beta;
        xp.M = h->M; xp.K = K; xp.rng = h->d_rng; xp.ki = h->d_ki; xp.wi = h->d_wi; xp.fi = h->d_fi;
        xp.tables = h->d_tables;
        xp.pool = h->pool;
        // static tables (~25 KB) + 2 KB of counters per move: pools of 12+ moves pass the 48 KB default and must opt in
        auto launch = [&](auto kernel, size_t dyn) -> int32_t {
            cudaFuncAttributes fa{};
            CU_TRY(h, cudaFuncGetAttributes(&fa, kernel));
            if (fa.sharedSizeBytes + dyn > 48 * 1024)
                CU_TRY(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
            kernel<<<wave_grid(h, kernel, dyn, h->M), kBlock, dyn, h->stream>>>(xp);
            return ARIANNA_OK;
        };
        const int32_t rc = dispatch_pot(h->cfg.potential, [&](auto pot) -> int32_t {
            constexpr int POT = decltype(pot)::value;
            if (exact) return multi ? launch(sweep_xoshiro_kernel<POT, ARITH_EXACT, true>, smem)
                                    : launch(sweep_xoshiro_kernel<POT, ARITH_EXACT, false>, 0);
            return multi ? launch(sweep_xoshiro_kernel<POT, ARITH_FAST, true>, smem)
                         : launch(sweep_xoshiro_kernel<POT, ARITH_FAST, false>, 0);
        });
        if (rc) return rc;
    }
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    h->steps_done += K;
    h->sums_valid = false;
    int32_t rc_red = ARIANNA_OK;
    if (want_reduce) {
        if (h->cfg.rng_mode == ARIANNA_RNG_PHILOX) h->sums_valid = true;  // fused at the sweep's tail
        else rc_red = launch_callback_reduce(h);
    }
    time_mark(h, 0, false);
    return rc_red;
}

// Store intervals fused per series launch.  Each interval costs kSeriesBytesPerStore (3 KB) of shared memory per CTA
// on top of the kernel's math tables (~19 KB, mostly the sin/cos directions): as many intervals as keep the
// sweep's 4 resident CTAs per SM (11 on B200's 228 KB); an ensemble that fits one CTA per SM anyway (M <= 256 x SM
// count: the reference's own small-M configurations) fuses up to ARIANNA_MAX_SERIES per launch.
static int series_per_launch(const arianna_handle *h)
{
    // test hook (with ARIANNA_REPLAY_STAGE_BYTES): a small value forces the multi-launch splits the tests cover
    const char *e = getenv("ARIANNA_SERIES_PER_LAUNCH");
    const int env = e ? atoi(e) : 0;
    if (env > 0) return env < kMaxSeries ? env : kMaxSeries;
    if (h->pool.n_moves > 1) {
        // multi-move pools: one warp-accumulator row of (1 + n_moves) doubles per interval and warp; as many intervals
        // as keep kMultiMinBlocks CTAs per SM, at most 32 (the per-CTA partials grow with it)
        const long budget = (long)(h->smem_per_sm / kMultiMinBlocks) - 1024 - (long)multi_smem_bytes(h->pool.n_moves, 0, 0, 1);
        long n = budget / (long)(kWarpsPerBlock * (1 + h->pool.n_moves) * 8);
        if (n < 1) n = 1;
        if (n > 32) n = 32;
        return (int)n;
    }
    if (h->M <= (int64_t)kBlock * h->sm_count) return kMaxSeries;
    cudaFuncAttributes fa{};
    size_t stat = 1024;
    if (cudaFuncGetAttributes(&fa, sweep_philox_kernel<POT_HARMONIC, ARITH_FAST, true, false>) == cudaSuccess)
        stat = fa.sharedSizeBytes;
    else
        cudaGetLastError();
    const long per_cta = (long)(h->smem_per_sm / kSweepMinBlocks) - 1024 - (long)stat - (long)sizeof(m64::MathTables) -
                         (long)(sizeof(unsigned long long) * kBlock);
    long n = per_cta / kSeriesBytesPerStore;
    if (n < 1) n = 1;
    if (n > 16) n = 16;
    return (int)n;
}

int32_t arianna_series_per_launch(arianna_handle *h, int32_t *n)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, n != nullptr, "arianna_series_per_launch: NULL output");
    DeviceGuard guard(h->device);
    *n = series_per_launch(h);
    return ARIANNA_OK;
}

// n_stores store intervals over the chains [off, off + m) of this handle, starting at MC step t0; records are written
// to (accumulate = 0) or added into (1) d_series[0 .. n_stores).  Asynchronous on h->stream.
static int32_t series_range(arianna_handle *h, int64_t off, int64_t m, int64_t t0, int32_t n_stores, const int64_t *K,
                            int accumulate)
{
    const bool exact = h->cfg.arith_mode == ARIANNA_ARITH_EXACT;
    const int per_launch = series_per_launch(h);
    const int stride = record_stride(h);
    for (int32_t s0 = 0; s0 < n_stores; s0 += per_launch) {
        const int ns = n_stores - s0 < per_launch ? n_stores - s0 : per_launch;
        if (h->pool.n_moves > 1) {
            const int32_t rc = launch_multi(h, off, m, t0, ns, K + s0, h->d_series + (size_t)stride * s0, h->d_sums, accumulate);
            if (rc) return rc;
            for (int i = 0; i < ns; ++i) t0 += K[s0 + i];
            continue;
        }
        SweepParams sp{};
        sp.x = h->d_x + off; sp.acc = h->d_acc + off; sp.tot = nullptr;
        sp.betas = h->d_betas ? h->d_betas + off : nullptr; sp.beta = h->cfg.beta;
        sp.M = m; sp.t0 = t0;
        sp.sid0 = (uint64_t)(h->cfg.seed + h->cfg.chain_offset + off);
        sp.tables = h->d_tables;
        sp.pool = h->pool;
        sp.theta = h->theta_active ? h->d_theta : nullptr;
        sp.n_series = ns;
        SeriesK sk{};
        int64_t k_launch = 0;
        bool even = (t0 & 1) == 0;
        for (int i = 0; i < ns; ++i) {
            sp.series_K[i] = sk.k[i] = (int)K[s0 + i];
            k_launch += K[s0 + i];
            even = even && K[s0 + i] > 0 && (K[s0 + i] & 1) == 0;
        }
        sp.series_K[ns] = 0;
        sp.series_even = even ? 1 : 0;
        sp.K = k_launch;
        const size_t smem = sizeof(m64::MathTables) + (size_t)ns * kSeriesBytesPerStore + sizeof(unsigned long long) * kBlock;
        int grid = 0;
        int32_t rc = dispatch_pot(h->cfg.potential, [&](auto pot) -> int32_t {
            constexpr int POT = decltype(pot)::value;
            auto go = [&](auto kernel) -> int32_t {
                CU_TRY(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                grid = wave_grid(h, kernel, smem, m);
                const int32_t r = ensure_series_partials(h, (size_t)grid * (ns + 1) * 2);
                if (r) return r;
                sp.series_partials = h->d_series_partials;
                kernel<<<grid, kBlock, smem, h->stream>>>(sp);
                return ARIANNA_OK;
            };
            if (h->d_betas || h->theta_active)
                return exact ? go(sweep_philox_kernel<POT, ARITH_EXACT, true, true>)
                             : go(sweep_philox_kernel<POT, ARITH_FAST, true, true>);
            return exact ? go(sweep_philox_kernel<POT, ARITH_EXACT, true, false>)
                         : go(sweep_philox_kernel<POT, ARITH_FAST, true, false>);
        });
        if (rc) return rc;
        CU_TRY(h, cudaGetLastError());
        series_fold_kernel<<<ns, kBlock, 0, h->stream>>>(h->d_series_partials, grid, ns, t0, sk, m,
                                                       h->d_series + 3 * (size_t)s0, h->d_sums, accumulate);
        CU_TRY(h, cudaGetLastError());
        h->launches += 2;
        t0 += k_launch;
    }
    return ARIANNA_OK;
}

static int32_t series_prepare(arianna_handle *h, const char *who, int32_t n_stores, const int64_t *K, int64_t *total_out)
{
    REQUIRE(h, n_stores >= 0 && (n_stores == 0 || K != nullptr), std::string(who) + ": bad arguments");
    if (h->cfg.rng_mode != ARIANNA_RNG_PHILOX || h->f32)
        return fail(h, ARIANNA_ERR_UNSUPPORTED, std::string(who) + ": Float64 ensembles with the native Philox stream only (use arianna_sweep)");
    int64_t total = 0;
    for (int32_t i = 0; i < n_stores; ++i) {
        REQUIRE(h, K[i] >= 0 && K[i] < (int64_t(1) << 31), std::string(who) + ": K[i] must be in [0, 2^31)");
        total += K[i];
    }
    REQUIRE(h, h->steps_done + total <= 0xFFFFFFFFll, std::string(who) + ": per-chain counters are 32-bit (2^32-1 steps max)");
    *total_out = total;
    h->series_n = 0;
    if (n_stores == 0) return ARIANNA_OK;
    if (h->series_cap < n_stores) {
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        cudaFree(h->d_series);
        h->d_series = nullptr;
        h->series_cap = 0;
        const int64_t cap = n_stores < 1024 ? 1024 : n_stores;
        CU_TRY(h, cudaMalloc(&h->d_series, sizeof(double) * record_stride(h) * cap));
        h->series_cap = cap;
    }
    // The per-CTA partials for the LARGEST grid any launch of this call can use, allocated NOW: growing the buffer in the
    // middle of a pipelined host job means cudaFree, i.e. a device-wide synchronisation that waits for every queued
    // upload (measured: the regular slices of a job started only after the whole ensemble had been uploaded).
    {
        const int per_launch = series_per_launch(h);
        const size_t per_cta = h->pool.n_moves > 1 ? (size_t)per_launch * (1 + h->pool.n_moves) : (size_t)(per_launch + 1) * 2;
        const int32_t rc = ensure_series_partials(h, (size_t)max_wave_grid(h) * per_cta);
        if (rc) return rc;
    }
    return ARIANNA_OK;
}

int32_t arianna_sweep_series(arianna_handle *h, int32_t n_stores, const int64_t *K, double *records)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    int64_t total = 0;
    int32_t rc = series_prepare(h, "arianna_sweep_series", n_stores, K, &total);
    if (rc || n_stores == 0) return rc;
    time_mark(h, 0, true);
    rc = series_range(h, 0, h->M, h->steps_done, n_stores, K, 0);
    if (rc) {   // a launch failed after earlier ones were queued: drain them; the chains are part-way through the stretch
        cudaStreamSynchronize(h->stream);
        h->sums_valid = false;
        h->err += " (arianna_sweep_series was partly executed: chain state is undefined, steps_done was not advanced)";
        return rc;
    }
    time_mark(h, 0, false);
    h->steps_done += total;
    h->series_n = n_stores;
    h->sums_valid = true;   // the last record doubles as the callback sums of the current state
    if (records) {
        CU_TRY(h, cudaMemcpyAsync(records, h->d_series, sizeof(double) * record_stride(h) * n_stores, cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
    }
    return ARIANNA_OK;
}

// Slice plan of a host job: slice i = chains [cuts[i], cuts[i + 1]).  The sweep of a slice can only start when its
// upload has landed and its download only when its sweep is done, so the FIRST upload and the LAST download are
// exposed.  The plan therefore starts with small slices (1/64 of the ensemble, at least one resident wave of the sweep
// kernel) that double up to the regular size M / n_slices and, when the chains are downloaded, ends with slices that
// halve again: the per-launch overheads (a partial last wave per launch) are paid by the few regular slices while the
// exposed copies shrink to 1/64 of the ensemble.  Every cut except the last is a multiple of the CTA size.
static std::vector<int64_t> slice_cuts(int64_t M, int n_slices, bool ramp_head, bool ramp_tail, int64_t wave)
{
    auto down = [](int64_t v) { return v / kBlock * kBlock; };
    std::vector<int64_t> cuts{0};
    if (n_slices <= 1 || M <= 2 * kBlock) { cuts.push_back(M); return cuts; }
    int64_t cap = down((M + n_slices - 1) / n_slices + kBlock - 1);
    if (cap < kBlock) cap = kBlock;
    int64_t small = down(M / 64);
    if (small < wave) small = wave < cap ? wave : cap;
    std::vector<int64_t> ramp;      // small, small, 2 small, 2 small, 4 small, ... below the regular size
    {
        int64_t sum = 0;
        int rep = 0;
        for (int64_t sz = small; sz < cap && sum + sz <= M / 4;) {
            ramp.push_back(sz);
            sum += sz;
            if (rep) sz *= 2;
            rep ^= 1;
        }
    }
    int64_t tail = 0;
    if (ramp_tail) for (auto v : ramp) tail += v;
    if (ramp_head) for (auto v : ramp) cuts.push_back(cuts.back() + v);
    const int64_t body_end = (ramp_tail && !ramp.empty()) ? down(M - tail) : M;
    while (cuts.back() < body_end) {
        const int64_t left = body_end - cuts.back();
        cuts.push_back(cuts.back() + (left < cap + cap / 4 ? left : cap));       // no tiny remainder slice
    }
    if (ramp_tail && !ramp.empty()) {
        for (size_t i = ramp.size(); i-- > 1;) cuts.push_back(cuts.back() + ramp[i]);   // largest first ...
        cuts.push_back(M);                                                               // ... smallest (+ rounding) last
    }
    return cuts;
}

// A whole callbacks-only job with HOST buffers, pipelined over slices of the chains: the upload of slice i+1 (H2D
// stream) and the download of slice i-1 (D2H stream) run while slice i sweeps through ALL the store intervals on the
// compute stream (chains are independent, so slice-major order gives the same chains and the same records as
// time-major).  PCIe is full duplex: uploads and downloads never queue behind each other.
int32_t arianna_run_host_job(arianna_handle *h, const double *x_in, int32_t n_stores, const int64_t *K, double *records,
                             double *x_out, int32_t n_slices)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, n_slices >= 1 && n_slices <= 1024, "arianna_run_host_job: n_slices must be in 1..1024");
    DeviceGuard guard(h->device);
    int64_t total = 0;
    int32_t rc = series_prepare(h, "arianna_run_host_job", n_stores, K, &total);
    if (rc) return rc;
    rc = ensure_copy_stream(h);
    if (rc) return rc;
    // Slices: whole CTAs' worth of chains each (see slice_cuts)
    const std::vector<int64_t> cuts = slice_cuts(h->M, n_slices, x_in != nullptr, x_out != nullptr,
                                                 (int64_t)h->sm_count * 4 * kBlock);
    const int ns = (int)cuts.size() - 1;
    std::vector<cudaEvent_t> up(ns, nullptr), done(ns, nullptr);
    bool queued = false;
    auto cleanup = [&]() {
        if (queued) {   // a failure after work was queued: drain it so that no copy outlives the caller's buffers
            cudaStreamSynchronize(h->h2d_stream); cudaStreamSynchronize(h->stream); cudaStreamSynchronize(h->copy_stream);
            h->sums_valid = false;
        }
        for (auto e : up) if (e) cudaEventDestroy(e);
        for (auto e : done) if (e) cudaEventDestroy(e);
    };
#define JOB_TRY(expr)                                                                                         \
    do {                                                                                                      \
        cudaError_t _e = (expr);                                                                              \
        if (_e != cudaSuccess) {                                                                              \
            cleanup();                                                                                        \
            return fail(h, ARIANNA_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e) +             \
                        (queued ? " (the job was partly executed: chain state is undefined)" : ""));          \
        }                                                                                                     \
    } while (0)
    h->job_timed[0] = h->job_timed[1] = false;
    h->job_bytes[0] = x_in ? (int64_t)sizeof(double) * h->M : 0;
    h->job_bytes[1] = x_out ? (int64_t)sizeof(double) * h->M : 0;
    // everything already queued on the compute stream must be done with x before the uploads overwrite it
    JOB_TRY(cudaEventRecord(h->ev_snap, h->stream));
    JOB_TRY(cudaStreamWaitEvent(h->h2d_stream, h->ev_snap, 0));
    JOB_TRY(cudaStreamWaitEvent(h->copy_stream, h->ev_snap, 0));
    for (int i = 0; i < ns; ++i) {
        JOB_TRY(cudaEventCreateWithFlags(&up[i], cudaEventDisableTiming));
        JOB_TRY(cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming));
    }
    if (x_in) {
        JOB_TRY(cudaEventRecord(h->ev_job[0], h->h2d_stream));
        for (int i = 0; i < ns; ++i) {
            const int64_t off = cuts[i], m = cuts[i + 1] - cuts[i];
            queued = true;
            JOB_TRY(cudaMemcpyAsync(h->d_x + off, x_in + off, sizeof(double) * m, cudaMemcpyHostToDevice, h->h2d_stream));
            JOB_TRY(cudaEventRecord(up[i], h->h2d_stream));
        }
        JOB_TRY(cudaEventRecord(h->ev_job[1], h->h2d_stream));
        h->job_timed[0] = true;
    }
    time_mark(h, 0, true);
    for (int i = 0; i < ns; ++i) {
        const int64_t off = cuts[i], m = cuts[i + 1] - cuts[i];
        if (x_in) JOB_TRY(cudaStreamWaitEvent(h->stream, up[i], 0));
        if (n_stores > 0) {
            queued = true;
            rc = series_range(h, off, m, h->steps_done, n_stores, K, i > 0);
            if (rc) { cleanup(); return rc; }
        }
        if (x_out) {
            JOB_TRY(cudaEventRecord(done[i], h->stream));
            JOB_TRY(cudaStreamWaitEvent(h->copy_stream, done[i], 0));
            if (i == 0) JOB_TRY(cudaEventRecord(h->ev_job[2], h->copy_stream));
            JOB_TRY(cudaMemcpyAsync(x_out + off, h->d_x + off, sizeof(double) * m, cudaMemcpyDeviceToHost, h->copy_stream));
        }
    }
    if (x_out) {
        JOB_TRY(cudaEventRecord(h->ev_job[3], h->copy_stream));
        h->job_timed[1] = true;
    }
    time_mark(h, 0, false);
    h->steps_done += total;
    h->series_n = n_stores;
    h->sums_valid = n_stores > 0;
    if (records && n_stores > 0)
        JOB_TRY(cudaMemcpyAsync(records, h->d_series, sizeof(double) * record_stride(h) * n_stores, cudaMemcpyDeviceToHost, h->stream));
    JOB_TRY(cudaEventRecord(h->ev_copy, h->copy_stream));
    JOB_TRY(cudaStreamSynchronize(h->stream));
    JOB_TRY(cudaStreamSynchronize(h->copy_stream));
    JOB_TRY(cudaStreamSynchronize(h->h2d_stream));
#undef JOB_TRY
    queued = false;
    cleanup();
    return ARIANNA_OK;
}

int32_t arianna_job_timing(arianna_handle *h, double *h2d_ms, double *h2d_gbs, double *d2h_ms, double *d2h_gbs)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    double *ms[2] = {h2d_ms, d2h_ms}, *gbs[2] = {h2d_gbs, d2h_gbs};
    for (int w = 0; w < 2; ++w) {
        if (ms[w]) *ms[w] = std::nan("");
        if (gbs[w]) *gbs[w] = std::nan("");
        if (!h->job_timed[w]) continue;
        CU_TRY(h, cudaEventSynchronize(h->ev_job[2 * w + 1]));
        float t = 0.f;
        CU_TRY(h, cudaEventElapsedTime(&t, h->ev_job[2 * w], h->ev_job[2 * w + 1]));
        if (ms[w]) *ms[w] = t;
        if (gbs[w]) *gbs[w] = t > 0.f ? (double)h->job_bytes[w] / (t * 1e-3) / 1e9 : std::nan("");
    }
    return ARIANNA_OK;
}

int32_t arianna_series_device(arianna_handle *h, double **dptr, int32_t *n_doubles)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, dptr && n_doubles, "arianna_series_device: NULL output");
    *dptr = h->d_series;
    *n_doubles = (int32_t)(record_stride(h) * h->series_n);
    return ARIANNA_OK;
}

int32_t arianna_sweep_replay(arianna_handle *h, int64_t K, const double *u_cat, const double *z,
                             const double *u_acc, uint8_t *decisions_out, int32_t on_device)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, K >= 0, "arianna_sweep_replay: K must be >= 0");
    if (K == 0) return ARIANNA_OK;
    REQUIRE(h, z != nullptr && u_acc != nullptr, "arianna_sweep_replay: z and u_acc are required");
    const bool multi = h->pool.n_moves > 1;
    REQUIRE(h, !multi || u_cat != nullptr, "arianna_sweep_replay: u_cat is required for multi-move pools");
    REQUIRE(h, h->steps_done + K <= 0xFFFFFFFFll, "arianna_sweep_replay: per-chain counters are 32-bit");
    DeviceGuard guard(h->device);
    { const int32_t rcp = pull_theta(h); if (rcp) return rcp; }      // (this path passes θ by value)
    const size_t smem = multi ? sizeof(uint32_t) * 2 * h->pool.n_moves * kBlock : 0;

    auto launch = [&](int64_t k, const double *duc, const double *dz, const double *dua, uint8_t *ddec) -> int32_t {
        if (h->f32) {       // Float32 ensemble: the same Float64 draws, z rounded to Float32 as randn(rng, Float32) does
            F32Params fp{};
            fp.x = h->d_xf; fp.acc = h->d_acc; fp.betas = h->d_betas_f; fp.beta = (float)h->cfg.beta;
            fp.M = h->M; fp.K = k;
            fp.sigma = (float)h->pool.sigma[0]; fp.lognorm = h->lognorm_f32;
            fp.tables = h->d_tables;
            fp.z = dz; fp.u_acc = dua; fp.decisions = ddec;
            dispatch_pot(h->cfg.potential, [&](auto pot) -> int32_t {
                constexpr int POT = decltype(pot)::value;
                sweep_replay_f32_kernel<POT><<<wave_grid(h, sweep_replay_f32_kernel<POT>, 0, h->M), kBlock, 0, h->stream>>>(fp);
                return ARIANNA_OK;
            });
            CU_TRY(h, cudaGetLastError());
            ++h->launches;
            return ARIANNA_OK;
        }
        ReplayParams rp{};
        rp.x = h->d_x; rp.acc = h->d_acc; rp.tot = h->d_tot; rp.betas = h->d_betas; rp.beta = h->cfg.beta;
        rp.M = h->M; rp.K = k; rp.u_cat = multi ? duc : nullptr; rp.z = dz; rp.u_acc = dua; rp.decisions = ddec;
        rp.tables = h->d_tables;
        rp.pool = h->pool;
        auto go = [&](auto kernel, size_t dyn) -> int32_t {
            cudaFuncAttributes fa{};
            CU_TRY(h, cudaFuncGetAttributes(&fa, kernel));
            if (fa.sharedSizeBytes + dyn > 48 * 1024)
                CU_TRY(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
            kernel<<<wave_grid(h, kernel, dyn, h->M), kBlock, dyn, h->stream>>>(rp);
            return ARIANNA_OK;
        };
        // bulk-copy (TMA) path: cp.async.bulk needs 16-byte aligned rows, i.e. an even number of chains and 16-byte
        // aligned arrays; ragged shapes take the per-thread-load kernel (same arithmetic, same results)
        auto aligned16 = [](const void *q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
        const bool tma = (h->M % 2 == 0) && aligned16(dz) && aligned16(dua) && (!multi || aligned16(duc));
        auto go_tma = [&](auto kernel) -> int32_t {
            const size_t dyn = replay_tma_smem_bytes(h->pool.n_moves);
            CU_TRY(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
            int per_sm = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kReplayThreads, dyn) != cudaSuccess || per_sm < 1) {
                cudaGetLastError();
                per_sm = 1;
            }
            const int64_t nblocks = (h->M + kReplayChains - 1) / kReplayChains, cap = (int64_t)h->sm_count * per_sm;
            kernel<<<(int)(nblocks < cap ? nblocks : cap), kReplayThreads, dyn, h->stream>>>(rp);   // persistent CTAs
            return ARIANNA_OK;
        };
        const int32_t rc = dispatch_pot(h->cfg.potential, [&](auto pot) -> int32_t {
            constexpr int POT = decltype(pot)::value;
            if (tma) return multi ? go_tma(sweep_replay_tma_kernel<POT, true>) : go_tma(sweep_replay_tma_kernel<POT, false>);
            return multi ? go(sweep_replay_kernel<POT, true>, smem) : go(sweep_replay_kernel<POT, false>, 0);
        });
        if (rc) return rc;
        CU_TRY(h, cudaGetLastError());
        ++h->launches;
        return ARIANNA_OK;
    };

    if (on_device) {
        int32_t rc = launch(K, u_cat, z, u_acc, decisions_out);
        if (rc) return rc;
    } else {
        // stage host draws through a bounded device buffer, chunked over steps (<= 1 GiB per array)
        const size_t per_step = sizeof(double) * (size_t)h->M;
        size_t stage = size_t(1) << 30;
        // test hook (with ARIANNA_SERIES_PER_LAUNCH): a small value forces the chunking the tests cover
        if (const char *env = getenv("ARIANNA_REPLAY_STAGE_BYTES")) stage = (size_t)strtoull(env, nullptr, 10);
        int64_t kc = (int64_t)(stage / per_step);
        if (kc < 1) kc = 1;
        if (kc > K) kc = K;
        const size_t narr = multi ? 3 : 2;
        const size_t need = narr * per_step * kc + (decisions_out ? (size_t)h->M * kc : 0);
        if (!ensure_scratch(h, need)) return fail(h, ARIANNA_ERR_NOMEM, "arianna_sweep_replay: staging allocation failed");
        double *dz = h->d_scratch;
        double *dua = dz + (size_t)h->M * kc;
        double *duc = multi ? dua + (size_t)h->M * kc : nullptr;
        uint8_t *ddec = decisions_out ? reinterpret_cast<uint8_t *>(h->d_scratch + narr * (size_t)h->M * kc) : nullptr;
        for (int64_t s0 = 0; s0 < K; s0 += kc) {
            const int64_t k = (K - s0 < kc) ? K - s0 : kc;
            const size_t off = (size_t)s0 * h->M;
            CU_TRY(h, cudaMemcpyAsync(dz, z + off, per_step * k, cudaMemcpyHostToDevice, h->stream));
            CU_TRY(h, cudaMemcpyAsync(dua, u_acc + off, per_step * k, cudaMemcpyHostToDevice, h->stream));
            if (multi) CU_TRY(h, cudaMemcpyAsync(duc, u_cat + off, per_step * k, cudaMemcpyHostToDevice, h->stream));
            int32_t rc = launch(k, duc, dz, dua, ddec);
            if (rc) return rc;
            if (ddec)
                CU_TRY(h, cudaMemcpyAsync(decisions_out + off, ddec, (size_t)h->M * k, cudaMemcpyDeviceToHost, h->stream));
            CU_TRY(h, cudaStreamSynchronize(h->stream));
        }
    }
    h->steps_done += K;
    h->sums_valid = false;
    return ARIANNA_OK;
}

int32_t arianna_set_rng_state(arianna_handle *h, const uint64_t *states)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, states != nullptr, "arianna_set_rng_state: states is NULL");
    if (h->cfg.rng_mode != ARIANNA_RNG_XOSHIRO)
        return fail(h, ARIANNA_ERR_UNSUPPORTED, "arianna_set_rng_state: handle was not created with ARIANNA_RNG_XOSHIRO");
    DeviceGuard guard(h->device);
    CU_TRY(h, cudaMemcpyAsync(h->d_rng, states, sizeof(uint64_t) * 4 * h->M, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

int32_t arianna_get_rng_state(arianna_handle *h, uint64_t *states)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, states != nullptr, "arianna_get_rng_state: states is NULL");
    if (h->cfg.rng_mode != ARIANNA_RNG_XOSHIRO)
        return fail(h, ARIANNA_ERR_UNSUPPORTED, "arianna_get_rng_state: handle was not created with ARIANNA_RNG_XOSHIRO");
    DeviceGuard guard(h->device);
    CU_TRY(h, cudaMemcpyAsync(states, h->d_rng, sizeof(uint64_t) * 4 * h->M, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

int32_t arianna_set_ziggurat_tables(arianna_handle *h, const uint64_t *ki, const double *wi, const double *fi)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, ki && wi && fi, "arianna_set_ziggurat_tables: NULL table");
    if (h->cfg.rng_mode != ARIANNA_RNG_XOSHIRO)
        return fail(h, ARIANNA_ERR_UNSUPPORTED, "arianna_set_ziggurat_tables: handle was not created with ARIANNA_RNG_XOSHIRO");
    DeviceGuard guard(h->device);
    CU_TRY(h, cudaMemcpyAsync(h->d_ki, ki, sizeof(uint64_t) * 256, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaMemcpyAsync(h->d_wi, wi, sizeof(double) * 256, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaMemcpyAsync(h->d_fi, fi, sizeof(double) * 256, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

int32_t arianna_callback_sums_device(arianna_handle *h, double **dptr, int32_t *n)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, dptr && n, "arianna_callback_sums_device: NULL output");
    DeviceGuard guard(h->device);
    if (!h->sums_valid) {
        int32_t rc = launch_callback_reduce(h);
        if (rc) return rc;
    }
    *dptr = h->d_sums;
    *n = 2 + h->pool.n_moves;
    return ARIANNA_OK;
}

int32_t arianna_callback_sums(arianna_handle *h, double *sums)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, sums != nullptr, "arianna_callback_sums: sums is NULL");
    double *d = nullptr;
    int32_t n = 0;
    int32_t rc = arianna_callback_sums_device(h, &d, &n);
    if (rc) return rc;
    DeviceGuard guard(h->device);
    CU_TRY(h, cudaMemcpyAsync(sums, d, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

int32_t arianna_callbacks(arianna_handle *h, double *mean_energy, double *acc_per_move)
{
    if (!h) return ARIANNA_ERR_INVALID;
    double sums[kMaxOut];
    int32_t rc = arianna_callback_sums(h, sums);
    if (rc) return rc;
    const int nm = h->pool.n_moves;
    const double cnt = sums[1 + nm];
    if (mean_energy) *mean_energy = sums[0] / cnt;
    if (acc_per_move)
        for (int k = 0; k < nm; ++k) acc_per_move[k] = sums[1 + k] / cnt;
    return ARIANNA_OK;
}

// ---- replica exchange (parallel tempering) across per-chain β ladders (csrc/kernels_exchange.cuh) -----------------
static int32_t ladder_supported(arianna_handle *h, const char *who)
{
    if (h->f32 || h->cfg.rng_mode != ARIANNA_RNG_PHILOX)
        return fail(h, ARIANNA_ERR_UNSUPPORTED,
                    std::string(who) + ": replica exchange needs a Float64 ensemble with the native Philox stream");
    return ARIANNA_OK;
}

int32_t arianna_set_ladder(arianna_handle *h, int32_t L, const double *betas)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (int32_t rc = ladder_supported(h, "arianna_set_ladder")) return rc;
    REQUIRE(h, L >= 2 && L <= ARIANNA_MAX_LADDER, "arianna_set_ladder: L must be in 2..ARIANNA_MAX_LADDER");
    REQUIRE(h, betas != nullptr, "arianna_set_ladder: betas is NULL");
    REQUIRE(h, h->cfg.chain_offset % L == 0 && h->M % L == 0,
            "arianna_set_ladder: the shard must hold whole ladders (chain_offset and n_chains multiples of L)");
    DeviceGuard guard(h->device);
    const int nm = h->pool.n_moves;
    if (L != h->ladder_L) {             // another ladder shape: new buffers, fresh round index and counters
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        cudaFree(h->d_ladder); cudaFree(h->d_ladder_partials); cudaFree(h->d_ladder_sums);
        h->d_ladder = h->d_ladder_partials = h->d_ladder_sums = nullptr;
        h->ladder_L = 0;
        if (!h->d_xacc) CU_TRY(h, cudaMalloc(&h->d_xacc, sizeof(unsigned long long) * kMaxLadder));
        CU_TRY(h, cudaMalloc(&h->d_ladder, sizeof(double) * L));
        CU_TRY(h, cudaMalloc(&h->d_ladder_partials, sizeof(double) * (size_t)h->grid * L * (1 + nm)));
        CU_TRY(h, cudaMalloc(&h->d_ladder_sums, sizeof(double) * (size_t)L * (2 + nm)));
        CU_TRY(h, cudaMemsetAsync(h->d_xacc, 0, sizeof(unsigned long long) * kMaxLadder, h->stream));
        h->ex_rounds = 0;
    }
    if (!h->d_betas) CU_TRY(h, cudaMalloc(&h->d_betas, sizeof(double) * h->M));
    CU_TRY(h, cudaMemcpyAsync(h->d_ladder, betas, sizeof(double) * L, cudaMemcpyHostToDevice, h->stream));
    ladder_betas_kernel<<<h->grid, kBlock, 0, h->stream>>>(h->d_betas, h->d_ladder, L, h->M);
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    CU_TRY(h, cudaStreamSynchronize(h->stream));     // `betas` is borrowed for the call only
    h->ladder_L = L;
    return ARIANNA_OK;
}

int32_t arianna_replica_exchange(arianna_handle *h)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (int32_t rc = ladder_supported(h, "arianna_replica_exchange")) return rc;
    REQUIRE(h, h->ladder_L >= 2, "arianna_replica_exchange: no ladder (call arianna_set_ladder first)");
    DeviceGuard guard(h->device);
    const int L = h->ladder_L;
    ExchangeParams p{};
    p.x = h->d_x;
    p.betas = h->d_betas;
    p.beta = h->cfg.beta;
    p.n_ladders = h->M / L;
    p.L = L;
    p.pairs = (L - (int)(h->ex_rounds & 1)) / 2;
    p.R = h->ex_rounds;
    p.sid0 = (uint64_t)(h->cfg.seed + h->cfg.chain_offset);
    p.tables = h->d_tables;
    p.accepted = h->d_xacc;
    if (p.pairs > 0) {
        dispatch_pot(h->cfg.potential, [&](auto pot) -> int32_t {
            exchange_kernel<decltype(pot)::value><<<h->grid, kBlock, 0, h->stream>>>(p);
            return ARIANNA_OK;
        });
        CU_TRY(h, cudaGetLastError());
        ++h->launches;
        h->sums_valid = false;
    }
    ++h->ex_rounds;
    return ARIANNA_OK;
}

int32_t arianna_exchange_counters(arianna_handle *h, int64_t *accepted, int64_t *rounds)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (int32_t rc = ladder_supported(h, "arianna_exchange_counters")) return rc;
    REQUIRE(h, h->ladder_L >= 2, "arianna_exchange_counters: no ladder (call arianna_set_ladder first)");
    DeviceGuard guard(h->device);
    if (accepted) {
        unsigned long long a[kMaxLadder];
        CU_TRY(h, cudaMemcpyAsync(a, h->d_xacc, sizeof(unsigned long long) * (h->ladder_L - 1), cudaMemcpyDeviceToHost,
                                  h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        for (int k = 0; k < h->ladder_L - 1; ++k) accepted[k] = (int64_t)a[k];
    }
    if (rounds) *rounds = h->ex_rounds;
    return ARIANNA_OK;
}

int32_t arianna_ladder_sums(arianna_handle *h, double *sums)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (int32_t rc = ladder_supported(h, "arianna_ladder_sums")) return rc;
    REQUIRE(h, h->ladder_L >= 2, "arianna_ladder_sums: no ladder (call arianna_set_ladder first)");
    REQUIRE(h, sums != nullptr, "arianna_ladder_sums: sums is NULL");
    DeviceGuard guard(h->device);
    const int L = h->ladder_L, nm = h->pool.n_moves;
    LadderReduceParams p{h->d_x, h->d_acc, h->d_tot, h->M, h->M, h->steps_done, nm, h->cfg.potential, L,
                         h->d_ladder_partials};
    if (nm == 1) ladder_reduce_kernel<1><<<h->grid, kBlock, 0, h->stream>>>(p);
    else ladder_reduce_kernel<kMaxMoves><<<h->grid, kBlock, 0, h->stream>>>(p);
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    ladder_fold_kernel<<<L, kBlock, 0, h->stream>>>(h->d_ladder_partials, h->grid, L, nm, (double)(h->M / L),
                                                    h->d_ladder_sums);
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    CU_TRY(h, cudaMemcpyAsync(sums, h->d_ladder_sums, sizeof(double) * L * (2 + nm), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

// ---- on-device histograms and moments of x or e (csrc/kernels_histogram.cuh) ---------------------------------------
static int32_t histogram_set(arianna_handle *h, const char *who)
{
    REQUIRE(h, h->hist_obs >= 0, std::string(who) + ": no histogram (call arianna_set_histogram first)");
    return ARIANNA_OK;
}

int32_t arianna_set_histogram(arianna_handle *h, int32_t observable, double lo, double hi, int32_t n_bins, int32_t n_groups)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, observable == ARIANNA_OBS_X || observable == ARIANNA_OBS_E, "arianna_set_histogram: unknown observable");
    REQUIRE(h, n_bins >= 1, "arianna_set_histogram: n_bins must be >= 1");
    REQUIRE(h, n_groups >= 1 && n_groups <= ARIANNA_MAX_LADDER, "arianna_set_histogram: n_groups must be in 1..ARIANNA_MAX_LADDER");
    REQUIRE(h, (int64_t)n_groups * ((int64_t)n_bins + 3) <= ARIANNA_MAX_HISTOGRAM_CELLS,
            "arianna_set_histogram: n_groups * (n_bins + 3) exceeds ARIANNA_MAX_HISTOGRAM_CELLS");
    REQUIRE(h, std::isfinite(lo) && std::isfinite(hi) && lo < hi, "arianna_set_histogram: lo and hi must be finite, lo < hi");
    const double inv_w = (double)n_bins / (hi - lo);
    REQUIRE(h, std::isfinite(inv_w) && inv_w > 0.0, "arianna_set_histogram: n_bins / (hi - lo) must be finite and > 0");
    DeviceGuard guard(h->device);
    CU_TRY(h, cudaStreamSynchronize(h->stream));   // an accumulate in flight still uses the old buffers
    cudaFree(h->d_hist_counts); cudaFree(h->d_hist_moments); cudaFree(h->d_hist_partials);
    h->d_hist_counts = nullptr;
    h->d_hist_moments = h->d_hist_partials = nullptr;
    h->hist_obs = -1;
    const int G = n_groups, cells = n_groups * (n_bins + 3);
    const size_t smem = sizeof(unsigned int) * cells;
    int per_sm = 0;
    int32_t rc = dispatch_histogram(h, observable, [&](auto kernel) -> int32_t {
        CU_TRY(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(sizeof(unsigned int) * kHistMaxCells)));
        CU_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kHistBlock, smem));
        return ARIANNA_OK;
    });
    if (rc) return rc;
    if (per_sm < 1) return fail(h, ARIANNA_ERR_CUDA, "arianna_set_histogram: histogram_kernel cannot be resident");
    // one resident wave: every CTA flushes its whole histogram once, so more CTAs only cost more global atomics
    const int64_t need = (h->M + kHistBlock - 1) / kHistBlock;
    const int64_t wave = (int64_t)h->sm_count * per_sm;
    const int grid = (int)(need < wave ? need : wave);
    CU_TRY(h, cudaMalloc(&h->d_hist_counts, sizeof(unsigned long long) * cells));
    CU_TRY(h, cudaMalloc(&h->d_hist_moments, sizeof(double) * G * 3));
    CU_TRY(h, cudaMalloc(&h->d_hist_partials, sizeof(double) * (size_t)grid * G * 3));
    CU_TRY(h, cudaMemsetAsync(h->d_hist_counts, 0, sizeof(unsigned long long) * cells, h->stream));
    CU_TRY(h, cudaMemsetAsync(h->d_hist_moments, 0, sizeof(double) * G * 3, h->stream));
    h->hist_obs = observable;
    h->hist_bins = n_bins;
    h->hist_groups = G;
    h->hist_grid = grid;
    h->hist_smem = smem;
    h->hist_lo = lo;
    h->hist_inv_w = inv_w;
    h->hist_samples = 0;
    return ARIANNA_OK;
}

int32_t arianna_histogram_accumulate(arianna_handle *h)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (int32_t rc = histogram_set(h, "arianna_histogram_accumulate")) return rc;
    DeviceGuard guard(h->device);
    const int G = h->hist_groups;
    HistogramParams p{};
    p.x = h->f32 ? static_cast<const void *>(h->d_xf) : static_cast<const void *>(h->d_x);
    p.M = h->M;
    p.g0 = (int)(((h->cfg.chain_offset % G) + G) % G);
    p.G = G;
    p.n_bins = h->hist_bins;
    p.lo = h->hist_lo;
    p.inv_w = h->hist_inv_w;
    p.counts = h->d_hist_counts;
    p.partials = h->d_hist_partials;
    dispatch_histogram(h, h->hist_obs, [&](auto kernel) -> int32_t {
        kernel<<<h->hist_grid, kHistBlock, h->hist_smem, h->stream>>>(p);
        return ARIANNA_OK;
    });
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    histogram_fold_kernel<<<G, kBlock, 0, h->stream>>>(h->d_hist_partials, h->hist_grid, G, h->d_hist_moments);
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    ++h->hist_samples;
    return ARIANNA_OK;
}

int32_t arianna_histogram_read(arianna_handle *h, int64_t *counts, double *moments, int64_t *n_samples)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (int32_t rc = histogram_set(h, "arianna_histogram_read")) return rc;
    DeviceGuard guard(h->device);
    const size_t G = (size_t)h->hist_groups;
    if (counts)
        CU_TRY(h, cudaMemcpyAsync(counts, h->d_hist_counts, sizeof(int64_t) * G * (h->hist_bins + 3), cudaMemcpyDeviceToHost,
                                  h->stream));
    if (moments) CU_TRY(h, cudaMemcpyAsync(moments, h->d_hist_moments, sizeof(double) * G * 3, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    if (n_samples) *n_samples = h->hist_samples;
    return ARIANNA_OK;
}

int32_t arianna_histogram_reset(arianna_handle *h)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (int32_t rc = histogram_set(h, "arianna_histogram_reset")) return rc;
    DeviceGuard guard(h->device);
    const size_t G = (size_t)h->hist_groups;
    CU_TRY(h, cudaMemsetAsync(h->d_hist_counts, 0, sizeof(unsigned long long) * G * (h->hist_bins + 3), h->stream));
    CU_TRY(h, cudaMemsetAsync(h->d_hist_moments, 0, sizeof(double) * G * 3, h->stream));
    h->hist_samples = 0;
    return ARIANNA_OK;
}

// ---- multi-GPU without a Python host: NCCL all-reduce of the tiny sum vectors inside the library ------------------
#define NCCL_TRY(h, expr)                                                                                     \
    do {                                                                                                      \
        int _r = (expr);                                                                                      \
        if (_r != 0) return fail((h), ARIANNA_ERR_NCCL, std::string(#expr) + ": " + nccl::g_api.GetErrorString(_r)); \
    } while (0)

int32_t arianna_nccl_unique_id(void *id128)
{
    if (!id128) return fail(nullptr, ARIANNA_ERR_INVALID, "arianna_nccl_unique_id: NULL output");
    std::string err;
    if (nccl::load(err)) return fail(nullptr, ARIANNA_ERR_NCCL, err);
    nccl::UniqueId id;
    int r = nccl::g_api.GetUniqueId(&id);
    if (r != 0) return fail(nullptr, ARIANNA_ERR_NCCL, std::string("ncclGetUniqueId: ") + nccl::g_api.GetErrorString(r));
    std::memcpy(id128, &id, sizeof id);
    return ARIANNA_OK;
}

int32_t arianna_comm_init(arianna_handle *h, const void *id128, int32_t rank, int32_t n_ranks)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, id128 != nullptr && n_ranks >= 1 && rank >= 0 && rank < n_ranks, "arianna_comm_init: bad arguments");
    REQUIRE(h, h->comm == nullptr, "arianna_comm_init: communicator already initialised");
    std::string err;
    if (nccl::load(err)) return fail(h, ARIANNA_ERR_NCCL, err);
    DeviceGuard guard(h->device);
    nccl::UniqueId id;
    std::memcpy(&id, id128, sizeof id);
    NCCL_TRY(h, nccl::g_api.CommInitRank(&h->comm, n_ranks, id, rank));
    h->comm_rank = rank;
    h->comm_size = n_ranks;
    if (!h->d_coll) CU_TRY(h, cudaMalloc(&h->d_coll, sizeof(double) * kMaxMoves * 5));
    return ARIANNA_OK;
}

static int32_t allreduce_small(arianna_handle *h, const double *d_src, int n, double *host_out)
{
    CU_TRY(h, cudaMemcpyAsync(h->d_coll, d_src, sizeof(double) * n, cudaMemcpyDeviceToDevice, h->stream));
    if (h->comm)
        NCCL_TRY(h, nccl::g_api.AllReduce(h->d_coll, h->d_coll, (size_t)n, /*ncclDouble*/ 8, /*ncclSum*/ 0, h->comm, h->stream));
    CU_TRY(h, cudaMemcpyAsync(host_out, h->d_coll, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

int32_t arianna_callbacks_global(arianna_handle *h, double *mean_energy, double *acc_per_move)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    if (!h->d_coll) CU_TRY(h, cudaMalloc(&h->d_coll, sizeof(double) * kMaxMoves * 5));
    double *d = nullptr;
    int32_t n = 0;
    int32_t rc = arianna_callback_sums_device(h, &d, &n);
    if (rc) return rc;
    double sums[kMaxOut];
    rc = allreduce_small(h, d, n, sums);
    if (rc) return rc;
    const int nm = h->pool.n_moves;
    const double cnt = sums[1 + nm];
    if (mean_energy) *mean_energy = sums[0] / cnt;
    if (acc_per_move)
        for (int k = 0; k < nm; ++k) acc_per_move[k] = sums[1 + k] / cnt;
    return ARIANNA_OK;
}

int32_t arianna_series_global(arianna_handle *h, int32_t n_stores, double *records)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, records != nullptr && n_stores >= 0 && n_stores <= h->series_n,
            "arianna_series_global: n_stores exceeds the last arianna_sweep_series call");
    if (n_stores == 0) return ARIANNA_OK;
    DeviceGuard guard(h->device);
    // in place on the series buffer: ONE all-reduce for the whole stretch of the schedule
    if (h->comm)
        NCCL_TRY(h, nccl::g_api.AllReduce(h->d_series, h->d_series, (size_t)record_stride(h) * n_stores, /*ncclDouble*/ 8,
                                          /*ncclSum*/ 0, h->comm, h->stream));
    CU_TRY(h, cudaMemcpyAsync(records, h->d_series, sizeof(double) * record_stride(h) * n_stores, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

// The same all-reduce without stalling the compute stream: the records of the last series are snapshotted (D2D on the
// compute stream, microseconds), and the all-reduce + the D2H copy into page-locked `records` run on a side stream
// while the NEXT sweep already executes -- the next launch does not depend on callback means (SURVEY.md §5).
// arianna_series_global_wait() (or arianna_synchronize) completes it.  One operation in flight per handle: a second
// begin waits (on the device) for the first.
int32_t arianna_series_global_begin(arianna_handle *h, int32_t n_stores, double *records_pinned)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, records_pinned != nullptr && n_stores >= 0 && n_stores <= h->series_n,
            "arianna_series_global_begin: n_stores exceeds the last arianna_sweep_series call");
    if (n_stores == 0) return ARIANNA_OK;
    DeviceGuard guard(h->device);
    if (!h->coll_stream) {
        CU_TRY(h, cudaStreamCreateWithFlags(&h->coll_stream, cudaStreamNonBlocking));
        CU_TRY(h, cudaEventCreateWithFlags(&h->ev_coll_src, cudaEventDisableTiming));
        CU_TRY(h, cudaEventCreateWithFlags(&h->ev_coll_done, cudaEventDisableTiming));
        CU_TRY(h, cudaEventRecord(h->ev_coll_done, h->coll_stream));
    }
    if (h->coll_series_cap < h->series_cap) {
        CU_TRY(h, cudaStreamSynchronize(h->coll_stream));
        cudaFree(h->d_coll_series);
        h->d_coll_series = nullptr;
        h->coll_series_cap = 0;
        CU_TRY(h, cudaMalloc(&h->d_coll_series, sizeof(double) * record_stride(h) * h->series_cap));
        h->coll_series_cap = h->series_cap;
    }
    const size_t n = (size_t)record_stride(h) * n_stores;
    CU_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_coll_done, 0));     // the previous operation has left the snapshot
    CU_TRY(h, cudaMemcpyAsync(h->d_coll_series, h->d_series, sizeof(double) * n, cudaMemcpyDeviceToDevice, h->stream));
    CU_TRY(h, cudaEventRecord(h->ev_coll_src, h->stream));
    CU_TRY(h, cudaStreamWaitEvent(h->coll_stream, h->ev_coll_src, 0));
    if (h->comm)
        NCCL_TRY(h, nccl::g_api.AllReduce(h->d_coll_series, h->d_coll_series, n, /*ncclDouble*/ 8, /*ncclSum*/ 0, h->comm,
                                          h->coll_stream));
    CU_TRY(h, cudaMemcpyAsync(records_pinned, h->d_coll_series, sizeof(double) * n, cudaMemcpyDeviceToHost, h->coll_stream));
    CU_TRY(h, cudaEventRecord(h->ev_coll_done, h->coll_stream));
    return ARIANNA_OK;
}

int32_t arianna_series_global_wait(arianna_handle *h)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (!h->coll_stream) return ARIANNA_OK;
    DeviceGuard guard(h->device);
    CU_TRY(h, cudaEventSynchronize(h->ev_coll_done));
    return ARIANNA_OK;
}

int32_t arianna_pgmc_read_global(arianna_handle *h, arianna_gradient_data *out, int32_t n_learn)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, out != nullptr && n_learn >= 0 && n_learn <= kMaxMoves, "arianna_pgmc_read_global: bad arguments");
    if (n_learn == 0) return ARIANNA_OK;
    DeviceGuard guard(h->device);
    if (!h->d_coll) CU_TRY(h, cudaMalloc(&h->d_coll, sizeof(double) * kMaxMoves * 5));
    return allreduce_small(h, h->d_gd, 5 * n_learn, reinterpret_cast<double *>(out));
}

int32_t arianna_get_counters(arianna_handle *h, int64_t *accepted, int64_t *total)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    const int nm = h->pool.n_moves;
    CU_TRY(h, cudaMemsetAsync(h->d_csum, 0, sizeof(unsigned long long) * 2 * kMaxMoves, h->stream));
    counter_sum_kernel<<<h->grid, kBlock, 0, h->stream>>>(h->d_acc, h->d_tot, h->M, nm, h->steps_done, h->d_csum);
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    unsigned long long out[2 * kMaxMoves];
    CU_TRY(h, cudaMemcpyAsync(out, h->d_csum, sizeof(unsigned long long) * 2 * nm, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    for (int k = 0; k < nm; ++k) {
        if (accepted) accepted[k] = (int64_t)out[k];
        if (total) total[k] = (int64_t)out[nm + k];
    }
    return ARIANNA_OK;
}

int32_t arianna_get_chain_counters(arianna_handle *h, uint32_t *accepted, uint32_t *total)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    const size_t n = (size_t)h->M * h->pool.n_moves;
    if (accepted) CU_TRY(h, cudaMemcpyAsync(accepted, h->d_acc, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, h->stream));
    if (total && h->d_tot)
        CU_TRY(h, cudaMemcpyAsync(total, h->d_tot, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    if (total && !h->d_tot)
        for (size_t i = 0; i < n; ++i) total[i] = (uint32_t)h->steps_done;
    return ARIANNA_OK;
}

static int32_t pgmc_impl(arianna_handle *h, int32_t q_batch, const int32_t *learn_ids, int32_t n_learn,
                         const double *z, int32_t on_device, bool replay)
{
    if (h->f32) return fail(h, ARIANNA_ERR_UNSUPPORTED, "arianna_pgmc_estimate: Float64 ensembles only");
    REQUIRE(h, q_batch >= 1, "arianna_pgmc_estimate: q_batch must be >= 1");
    REQUIRE(h, n_learn >= 0 && n_learn <= kMaxMoves && (n_learn == 0 || learn_ids != nullptr),
            "arianna_pgmc_estimate: bad learn_ids");
    for (int l = 0; l < n_learn; ++l)
        REQUIRE(h, learn_ids[l] >= 0 && learn_ids[l] < h->pool.n_moves, "arianna_pgmc_estimate: learn id out of range");
    if (n_learn == 0) return ARIANNA_OK;
    REQUIRE(h, replay || h->pgmc_samples + (int64_t)n_learn * q_batch < (int64_t(1) << 33),
            "arianna_pgmc_estimate: the estimator stream holds 2^33 samples per chain");
    DeviceGuard guard(h->device);
    const bool exact = replay || h->cfg.arith_mode == ARIANNA_ARITH_EXACT;
    const double *dz = z;
    if (replay && !on_device) {
        const size_t bytes = sizeof(double) * (size_t)n_learn * q_batch * h->M;
        if (!ensure_scratch(h, bytes)) return fail(h, ARIANNA_ERR_NOMEM, "arianna_pgmc_estimate_replay: staging allocation failed");
        CU_TRY(h, cudaMemcpyAsync(h->d_scratch, z, bytes, cudaMemcpyHostToDevice, h->stream));
        dz = h->d_scratch;
    }
    time_mark(h, 1, true);
    {
        // ONE launch for all the learnable moves (the loop over moves runs inside the kernel)
        PgmcParams pp{};
        pp.x = h->d_x; pp.betas = h->d_betas; pp.beta = h->cfg.beta; pp.M = h->M; pp.q_batch = q_batch;
        pp.n_learn = n_learn;
        pp.q0 = h->pgmc_samples;
        pp.sid0 = (uint64_t)(h->cfg.seed + h->cfg.chain_offset);
        for (int l = 0; l < n_learn; ++l) {
            pp.sigma[l] = h->pool.sigma[learn_ids[l]];
            pp.lognorm[l] = h->pool.lognorm[learn_ids[l]];
            pp.learn_id[l] = learn_ids[l];
        }
        pp.theta = h->theta_active ? h->d_theta : nullptr;
        pp.z = replay ? dz : nullptr;
        pp.gd = h->d_gd;
        pp.tables = h->d_tables;
        if (!h->d_pgmc_ticket) {
            CU_TRY(h, cudaMalloc(&h->d_pgmc_ticket, sizeof(unsigned int) * kMaxMoves));
            CU_TRY(h, cudaMemsetAsync(h->d_pgmc_ticket, 0, sizeof(unsigned int) * kMaxMoves, h->stream));
        }
        pp.ticket = h->d_pgmc_ticket;
        const int32_t rc = dispatch_pot(h->cfg.potential, [&](auto pot) -> int32_t {
            constexpr int POT = decltype(pot)::value;
            auto go = [&](auto kernel) -> int32_t {
                const int grid = wave_grid(h, kernel, 0, h->M);
                const size_t need = (size_t)n_learn * grid * 5;
                if (h->pgmc_partials_cap < need) {
                    CU_TRY(h, cudaStreamSynchronize(h->stream));
                    cudaFree(h->d_pgmc_partials);
                    h->d_pgmc_partials = nullptr;
                    h->pgmc_partials_cap = 0;
                    CU_TRY(h, cudaMalloc(&h->d_pgmc_partials, sizeof(double) * need));
                    h->pgmc_partials_cap = need;
                }
                pp.partials = h->d_pgmc_partials;
                kernel<<<grid, kBlock, 0, h->stream>>>(pp);
                return ARIANNA_OK;
            };
            if (replay) return go(pgmc_kernel<POT, ARITH_EXACT, true>);
            return exact ? go(pgmc_kernel<POT, ARITH_EXACT, false>) : go(pgmc_kernel<POT, ARITH_FAST, false>);
        });
        if (rc) return rc;
        CU_TRY(h, cudaGetLastError());
        ++h->launches;
    }
    time_mark(h, 1, false);
    if (!replay) h->pgmc_samples += (int64_t)n_learn * q_batch;
    if (replay && !on_device) CU_TRY(h, cudaStreamSynchronize(h->stream));
    if (exact) h->sums_valid = false;  // chain state drifted by the perform/undo rounding
    return ARIANNA_OK;
}

int32_t arianna_pgmc_estimate(arianna_handle *h, int32_t q_batch, const int32_t *learn_ids, int32_t n_learn)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (h->cfg.rng_mode != ARIANNA_RNG_PHILOX)
        return fail(h, ARIANNA_ERR_UNSUPPORTED, "arianna_pgmc_estimate: native estimator draws need ARIANNA_RNG_PHILOX");
    return pgmc_impl(h, q_batch, learn_ids, n_learn, nullptr, 0, false);
}

int32_t arianna_pgmc_estimate_replay(arianna_handle *h, int32_t q_batch, const int32_t *learn_ids, int32_t n_learn,
                                     const double *z, int32_t on_device)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, z != nullptr, "arianna_pgmc_estimate_replay: z is NULL");
    return pgmc_impl(h, q_batch, learn_ids, n_learn, z, on_device, true);
}

int32_t arianna_pgmc_read(arianna_handle *h, arianna_gradient_data *out, int32_t n_learn)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, out != nullptr && n_learn >= 0 && n_learn <= kMaxMoves, "arianna_pgmc_read: bad arguments");
    DeviceGuard guard(h->device);
    CU_TRY(h, cudaMemcpyAsync(out, h->d_gd, sizeof(double) * 5 * n_learn, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

int32_t arianna_pgmc_reset(arianna_handle *h)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    CU_TRY(h, cudaMemsetAsync(h->d_gd, 0, sizeof(double) * kMaxMoves * 5, h->stream));
    return ARIANNA_OK;
}

int32_t arianna_pgmc_update_device(arianna_handle *h, const int32_t *learn_ids, const arianna_optimiser *opts, int32_t n_learn)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, n_learn >= 0 && n_learn <= kMaxMoves && (n_learn == 0 || (learn_ids && opts)),
            "arianna_pgmc_update_device: bad arguments");
    if (h->f32) return fail(h, ARIANNA_ERR_UNSUPPORTED, "arianna_pgmc_update_device: Float64 ensembles only");
    if (n_learn == 0) return ARIANNA_OK;
    UpdateParams u{};
    u.n_learn = n_learn;
    for (int l = 0; l < n_learn; ++l) {
        REQUIRE(h, learn_ids[l] >= 0 && learn_ids[l] < h->pool.n_moves, "arianna_pgmc_update_device: learn id out of range");
        REQUIRE(h, opts[l].kind >= ARIANNA_OPT_STATIC && opts[l].kind <= ARIANNA_OPT_BLANPG,
                "arianna_pgmc_update_device: unknown optimiser");
        u.learn_id[l] = learn_ids[l]; u.kind[l] = opts[l].kind; u.p1[l] = opts[l].p1; u.p2[l] = opts[l].p2;
    }
    DeviceGuard guard(h->device);
    if (!h->theta_active) {
        const int32_t rc = push_theta(h);
        if (rc) return rc;
        h->theta_active = true;
    }
    // gradients_data summed over all ranks, in place (every rank then applies the same step to its own θ block)
    if (h->comm)
        NCCL_TRY(h, nccl::g_api.AllReduce(h->d_gd, h->d_gd, (size_t)5 * n_learn, /*ncclDouble*/ 8, /*ncclSum*/ 0, h->comm, h->stream));
    pgmc_update_kernel<<<1, 32, 0, h->stream>>>(h->d_theta, h->d_gd, u);
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    h->theta_dirty = true;
    return ARIANNA_OK;
}

int32_t arianna_params_sync(arianna_handle *h)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    return pull_theta(h);
}

int32_t arianna_pgmc_sums_device(arianna_handle *h, double **dptr, int32_t *n)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, dptr && n, "arianna_pgmc_sums_device: NULL output");
    *dptr = h->d_gd;
    *n = kMaxMoves * 5;
    return ARIANNA_OK;
}

int32_t arianna_get_stream(arianna_handle *h, void **stream)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, stream != nullptr, "arianna_get_stream: NULL output");
    *stream = (void *)h->stream;
    return ARIANNA_OK;
}

int32_t arianna_synchronize(arianna_handle *h)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    if (h->copy_stream) CU_TRY(h, cudaStreamSynchronize(h->copy_stream));
    if (h->h2d_stream) CU_TRY(h, cudaStreamSynchronize(h->h2d_stream));
    if (h->coll_stream) CU_TRY(h, cudaStreamSynchronize(h->coll_stream));
    return ARIANNA_OK;
}

int32_t arianna_timing(arianna_handle *h, double *sweep_ms, double *pgmc_ms)
{
    if (!h) return ARIANNA_ERR_INVALID;
    DeviceGuard guard(h->device);
    double *out[2] = {sweep_ms, pgmc_ms};
    for (int w = 0; w < 2; ++w) {
        if (!out[w]) continue;
        *out[w] = std::nan("");
        if (!h->timed[w]) continue;
        CU_TRY(h, cudaEventSynchronize(h->ev_t[2 * w + 1]));
        float ms = 0.f;
        CU_TRY(h, cudaEventElapsedTime(&ms, h->ev_t[2 * w], h->ev_t[2 * w + 1]));
        *out[w] = ms;
    }
    return ARIANNA_OK;
}

int32_t arianna_launch_count(arianna_handle *h, int64_t *n_launches)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, n_launches != nullptr, "arianna_launch_count: NULL output");
    *n_launches = h->launches;
    return ARIANNA_OK;
}

int32_t arianna_steps_done(arianna_handle *h, int64_t *steps)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, steps != nullptr, "arianna_steps_done: NULL output");
    *steps = h->steps_done;
    return ARIANNA_OK;
}

int32_t arianna_device_info(arianna_handle *h, int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor,
                            int64_t *hbm_bytes)
{
    if (!h) return ARIANNA_ERR_INVALID;
    if (sm_count) *sm_count = h->sm_count;
    if (cc_major) *cc_major = h->cc_major;
    if (cc_minor) *cc_minor = h->cc_minor;
    if (hbm_bytes) *hbm_bytes = (int64_t)h->hbm_bytes;
    return ARIANNA_OK;
}

int32_t arianna_debug_math(arianna_handle *h, int32_t kind, const double *a, const uint64_t *b, const uint64_t *c,
                           double *out, int64_t n)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, kind >= 0 && kind <= 11 && out != nullptr && n >= 0, "arianna_debug_math: bad arguments");
    if (n == 0) return ARIANNA_OK;
    DeviceGuard guard(h->device);
    const int64_t nout = (kind == 6 || kind == 7) ? 4 * n : (kind == 9 || kind < 3) ? n : 2 * n;
    const size_t bytes = sizeof(double) * (size_t)(nout + 3 * n);
    if (!ensure_scratch(h, bytes)) return fail(h, ARIANNA_ERR_NOMEM, "arianna_debug_math: scratch allocation failed");
    double *d_out = h->d_scratch;
    double *d_a = d_out + nout;
    uint64_t *d_b = reinterpret_cast<uint64_t *>(d_a + n);
    uint64_t *d_c = d_b + n;
    if (a) CU_TRY(h, cudaMemcpyAsync(d_a, a, sizeof(double) * n, cudaMemcpyHostToDevice, h->stream));
    if (b) CU_TRY(h, cudaMemcpyAsync(d_b, b, sizeof(uint64_t) * n, cudaMemcpyHostToDevice, h->stream));
    if (c) CU_TRY(h, cudaMemcpyAsync(d_c, c, sizeof(uint64_t) * n, cudaMemcpyHostToDevice, h->stream));
    debug_math_kernel<<<h->grid > 0 ? h->sm_count * 4 : 1, kBlock, 0, h->stream>>>(kind, d_a, d_b, d_c, d_out, n, h->d_tables);
    CU_TRY(h, cudaGetLastError());
    ++h->launches;
    CU_TRY(h, cudaMemcpyAsync(out, d_out, sizeof(double) * nout, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ARIANNA_OK;
}

int32_t arianna_measure_fp64_peak(arianna_handle *h, double *flops_per_s)
{
    if (!h) return ARIANNA_ERR_INVALID;
    REQUIRE(h, flops_per_s != nullptr, "arianna_measure_fp64_peak: NULL output");
    DeviceGuard guard(h->device);
    const int grid = h->sm_count * 8;
    const int iters = 2048;
    if (!ensure_scratch(h, sizeof(double) * (size_t)grid * kBlock))
        return fail(h, ARIANNA_ERR_NOMEM, "arianna_measure_fp64_peak: scratch allocation failed");
    cudaEvent_t e0, e1;
    CU_TRY(h, cudaEventCreate(&e0));
    CU_TRY(h, cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        CU_TRY(h, cudaEventRecord(e0, h->stream));
        dfma_peak_kernel<<<grid, kBlock, 0, h->stream>>>(h->d_scratch, iters, 0.999999, 1e-9);
        CU_TRY(h, cudaEventRecord(e1, h->stream));
        CU_TRY(h, cudaEventSynchronize(e1));
        ++h->launches;
        float ms = 0.f;
        CU_TRY(h, cudaEventElapsedTime(&ms, e0, e1));
        const double flops = 2.0 * 64.0 * (double)iters * (double)grid * kBlock;  // 64 DFMA per iteration
        const double rate = flops / (ms * 1e-3);
        if (rep > 0 && rate > best) best = rate;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CU_TRY(h, cudaGetLastError());
    *flops_per_s = best;
    return ARIANNA_OK;
}

}  // extern "C"
