// kernels.cuh -- the fused Metropolis sweep, callback-reduction and PGMC kernels (sm_100a).
//
// Layout in HBM (struct-of-arrays, one chain per thread, coalesced 8-byte lanes):
//   x[M]                 f64   chain positions (Particle.x, particle_1d.jl:10); e = potential(x) is recomputed
//   acc[n_moves][M]      u32   Move.accepted_calls per chain and move (metropolis.jl:146)
//   tot[n_moves][M]      u32   Move.total_calls -- only materialised for multi-move pools; a single-move pool has
//                              tot == steps_done for every chain
//   betas[M]             f64   optional per-chain β
//   rng[M][4]            u64   only in XOSHIRO mode
// Each thread keeps its chain's (x, e, counters) in registers across the K fused steps of one launch and writes
// back once: algorithmic HBM traffic is 24/K bytes per chain-step (x r+w 16 B, acc r+w 8 B).
//
// Reference mapping: mc_step! (src/metropolis.jl:176-190), mc_sweep! (:203-212), the particle_1d methods
// (example/particle_1d/particle_1d.jl:20-59), callback_energy (:68-70), callback_acceptance
// (src/metropolis.jl:319-321), pgmc_estimate (src/PolicyGuided/gradients.jl:93-109).
#pragma once
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

#include "math64.cuh"
#include "rng.cuh"

namespace arianna {

// Launch shape of the fused sweep: kBlock threads per CTA (a multiple of 32) and kSweepMinBlocks resident CTAs per SM
// requested through __launch_bounds__, i.e. a cap of 65536 / (256·4) = 64 registers.  The measured optimum: 3, 5 or 6
// CTAs per SM and a software pipeline of pair p+1 over pair p were all slower (DESIGN.md §4).
constexpr int kBlock = 256;
constexpr int kSweepMinBlocks = 4;
constexpr int kPgmcMinBlocks = 3;   // the estimator (a full FP64 exp per sample) prefers 80 registers x 3 CTAs: 4.20 vs 4.39 ms (C4)
constexpr int kMaxMoves = 16;
constexpr int kMaxSeries = 64;              // store intervals one series launch can fuse (host picks <= this)
constexpr int kSeriesBytesPerStore = kBlock * (8 + 4);   // shared memory per fused interval: Σe f64 + ΣΔacc u32 per thread
constexpr int kWarpsPerBlock = kBlock / 32;

enum { POT_HARMONIC = 0, POT_QUARTIC = 1, POT_DOUBLE_WELL = 2 };
enum { ARITH_EXACT = 0, ARITH_FAST = 1 };

struct PoolParams {
    int n_moves;
    double sigma[kMaxMoves];
    double weight[kMaxMoves];
    double lognorm[kMaxMoves];  // log((2π)·(σ·σ))/2, host-computed (particle_1d.jl:53)
    double inv2s2[kMaxMoves];   // RN(1 / (2·(σ·σ))), host-computed, or 0 when σ is outside the range exact_div covers
};

// Device-resident policy parameters θ = (σ) of every move + the per-move constants derived from them: written by
// pgmc_update_kernel (on-device optimiser), read by the sweep / estimator kernels instead of the by-value PoolParams
// when a handle runs its PolicyGradientUpdate on the device (no host round trip per update).
struct DevTheta {
    double sigma[kMaxMoves];
    double lognorm[kMaxMoves];
    double inv2s2[kMaxMoves];
    int bad;                    // set when an update left σ outside (0, ∞) (Normal(0, σ) would throw in the reference)
};

struct SweepParams {
    double *x;
    uint32_t *acc;
    uint32_t *tot;          // nullptr for single-move pools
    const double *betas;    // nullptr -> beta
    double beta;
    int64_t M;
    int64_t K;
    int64_t t0;             // MC steps already done by every chain (draw index base)
    uint64_t sid0;          // seed + chain_offset: stream id of local chain 0
    int reduce;             // fuse the callback sums into the tail of the sweep (single-move kernels)
    double *partials;       // [gridDim.x][kMaxOut]
    unsigned int *ticket;
    double *sums;           // [2 + n_moves]
    const m64::MathTables *tables;  // exp/log tables in global memory (copied to shared by every CTA)
    PoolParams pool;
    const DevTheta *theta;          // non-null: σ lives on the device (read by the BETAS = true instantiations only)
    // series mode (sweep_philox_kernel<..., SERIES = true>): n_series store intervals fused into ONE launch
    int n_series;
    int series_even;                // every interval is a positive even number of steps starting on an even step
    int series_K[kMaxSeries + 1];   // MC steps of each interval (one spare slot: read past the last interval)
    double *series_partials;        // [gridDim.x][n_series + 1][2]: (Σe, ΣΔacc) per interval, then (Σacc at entry, 0)
};

constexpr int kMaxOut = 2 + kMaxMoves;

__device__ __forceinline__ void load_tables(m64::MathTables *dst, const m64::MathTables *src)
{
    const double *s = reinterpret_cast<const double *>(src);
    double *d = reinterpret_cast<double *>(dst);
    for (int i = threadIdx.x; i < (int)(sizeof(m64::MathTables) / sizeof(double)); i += blockDim.x) d[i] = s[i];
}

// Handle of a MathTables copy in shared memory (m64::Tab).  Call it AFTER the __syncthreads() that follows
// load_tables: the empty volatile asm makes the window address opaque to the optimiser, which (1) keeps it in ONE
// register across the sweep's loops instead of being re-derived next to every use and (2) orders every table load
// (plain, non-volatile ld.shared asm that the compiler may otherwise treat as a pure function of its address) after
// the barrier through a data dependency.
__device__ __forceinline__ m64::Tab shared_tab(const void *smem_ptr)
{
    uint32_t a = (uint32_t)__cvta_generic_to_shared(smem_ptr);
    asm volatile("" : "+r"(a));
    return m64::Tab{a};
}
// explicit shared-memory accesses relative to such an address (series accumulators of the sweep)
__device__ __forceinline__ double lds_f64(uint32_t a) { double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_f64(uint32_t a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned long long lds_u64(uint32_t a) { unsigned long long v; asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_u64(uint32_t a, unsigned long long v) { asm volatile("st.shared.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }

// ---------------------------------------------------------------------------------------------------------
// potential(x)
// ---------------------------------------------------------------------------------------------------------
template <int POT, int ARITH>
__device__ __forceinline__ double potential(double x)
{
    if constexpr (ARITH == ARITH_EXACT) {
        if constexpr (POT == POT_HARMONIC) {
            return __dmul_rn(x, x);
        } else if constexpr (POT == POT_QUARTIC) {
            double x2 = __dmul_rn(x, x);
            return __dmul_rn(x2, x2);
        } else {
            double w = __dsub_rn(__dmul_rn(x, x), 1.0);
            return __dmul_rn(w, w);
        }
    } else {
        if constexpr (POT == POT_HARMONIC) {
            return x * x;
        } else if constexpr (POT == POT_QUARTIC) {
            double x2 = x * x;
            return x2 * x2;
        } else {
            double w = fma(x, x, -1.0);
            return w * w;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// One Metropolis step (SURVEY.md Appendix A.1).  Returns mc_step!'s return value.
// EXACT: every statement is one round-to-nearest binary64 operation in the reference's order; the __d*_rn
// intrinsics are never contracted into FMAs.
// ---------------------------------------------------------------------------------------------------------
template <int POT>
__device__ __forceinline__ int mc_step_exact(double &x, double &e, double beta, double sigma, double lognorm,
                                             double inv2s2, double z, double u_acc, m64::Tab tb)
{
    double delta = __dadd_rn(0.0, __dmul_rn(sigma, z));                       // particle_1d.jl:57
    double s2 = __dmul_rn(sigma, sigma);
    double t1 = m64::exact_div(-__dmul_rn(delta, delta), __dmul_rn(2.0, s2), inv2s2);   // :53
    double lqf = __dsub_rn(t1, lognorm);                                      // metropolis.jl:178
    double e1 = e;                                                            // particle_1d.jl:31
    const double xn = __dadd_rn(x, delta);                                    // :32
    const double en = potential<POT, ARITH_EXACT>(xn);                        // :33
    double dlogp = __dsub_rn(__dmul_rn(-en, beta), __dmul_rn(-e1, beta));     // metropolis.jl:98
    delta = -delta;                                                           // particle_1d.jl:38
    double lqb = lqf;  // log_proposal_density of -δ: only (-δ)·(-δ) == δ·δ enters -> bitwise equal (metropolis.jl:182)
    double arg = __dsub_rn(__dadd_rn(dlogp, lqb), lqf);                       // :183, NOT simplified to dlogp
    // α = min(one(T), exp(arg)); α > rand(rng) (:183-184, strict >, NaN rejects) -- decided exactly as the FP64
    // evaluation of exp (≤1 ulp, like Julia's / glibc's) would, through the FP32 filter of m64::exp_accept
    float ulo, uhi;
    m64::ucell_from_double(u_acc, ulo, uhi);
    const bool a = m64::exp_accept(arg, ulo, uhi, [&]() { return u_acc; }, tb);
    // reject: the negated move is re-applied (:187), x = fl(fl(x+δ)-δ) -- not a restore.  Both outcomes are computed and
    // selected (no branch: two chains of one thread can then be interleaved by the scheduler)
    const double xr = __dadd_rn(xn, delta);
    const double er = potential<POT, ARITH_EXACT>(xr);
    x = a ? xn : xr;
    e = a ? en : er;
    return a ? 1 : 0;
}

// FAST: symmetric proposal => log q terms cancel; α > u  <=>  exp(β(e - e')) > u  because u < 1; reject restores x.
// The accept uniform arrives as (ulo, cell, exact_u): a float cell [ulo, ulo + cell) that contains u and a callable
// producing the exact 53-bit u on demand (see m64::exp_accept).
template <int PBITS>
struct CellP { uint32_t f; };     // PBITS-bit prefix of the accept uniform: u ∈ [f, f+1)·2^-PBITS
template <int PBITS>
struct CellM { uint32_t fm; };    // the same prefix as the filter's pre-assembled addend bits (m64::exp_prefix_bits);
                                  // the FAST step of a CellM caller must be given β·log2(e) for β (m64::exp_accept_prefix)
struct CellF { float ulo, cell; };

template <int PBITS, class ExactU>
__device__ __forceinline__ bool accept_in_cell(double arg, CellP<PBITS> c, ExactU exact_u, m64::Tab tb)
{
    return m64::exp_accept_prefix<PBITS>(arg, c.f, exact_u, tb);
}
template <int PBITS, class ExactU>
__device__ __forceinline__ bool accept_in_cell(double arg, CellM<PBITS> c, ExactU exact_u, m64::Tab tb)
{
    return m64::exp_accept_prefix<PBITS, true>(arg, c.fm, exact_u, tb);
}
// kFloorMagicBits in a register the compiler cannot fold back into an immediate
__device__ __forceinline__ uint32_t floor_magic_reg()
{
    uint32_t m;
    asm volatile("mov.u32 %0, 0xCB400000;" : "=r"(m));
    return m;
}
template <class ExactU>
__device__ __forceinline__ bool accept_in_cell(double arg, CellF c, ExactU exact_u, m64::Tab tb)
{
    return m64::exp_accept(arg, c.ulo, c.ulo + c.cell, exact_u, tb);   // ulo + cell is exact
}

template <int POT, class Cell, class ExactU>
__device__ __forceinline__ bool mc_step_fast(double &x, double &e, double beta, double sigma, double z, Cell cell,
                                             ExactU exact_u, m64::Tab tb)
{
    // e is re-derived from x (one DMUL on the idle FP64 pipe) instead of being carried through two more selects on
    // the ALU pipe, which is the busiest pipe of the sweep
    const double e0 = potential<POT, ARITH_FAST>(x);
    const double xn = fma(sigma, z, x);
    const double en = potential<POT, ARITH_FAST>(xn);
    const bool a = accept_in_cell(beta * (e0 - en), cell, exact_u, tb);
    x = a ? xn : x;
    (void)e;  // FAST never carries e: callers that need it (the fused reduction) evaluate potential(x)
    return a;
}

template <int POT, int ARITH, class Cell, class ExactU>
__device__ __forceinline__ bool mc_step(double &x, double &e, double beta, double sigma, double lognorm, double inv2s2,
                                        double z, Cell cell, ExactU exact_u, m64::Tab tb)
{
    if constexpr (ARITH == ARITH_EXACT)
        return mc_step_exact<POT>(x, e, beta, sigma, lognorm, inv2s2, z, exact_u(), tb) != 0;
    else
        return mc_step_fast<POT>(x, e, beta, sigma, z, cell, exact_u, tb);
}

// acc += flag as ONE predicated add (@p VIADD).  Written as `if (flag) ++acc` the compiler emits an add, a predicated
// move and a copy (three issue slots in an issue-bound loop); ptxas folds the setp below into the predicate that
// produced `flag`.
__device__ __forceinline__ void count_if(uint32_t &acc, uint32_t flag)
{
    asm("{\n .reg .pred p;\n setp.ne.u32 p, %1, 0;\n @p add.u32 %0, %0, 1;\n}" : "+r"(acc) : "r"(flag));
}

// Distributions.Categorical inverse-CDF scan [EXT] (metropolis.jl:206); weights in shared memory.
__device__ __forceinline__ int categorical(int n, const double *w, double u)
{
    int k = 0;
    double cp = w[0];
    while (cp <= u && k < n - 1) {
        ++k;
        cp = __dadd_rn(cp, w[k]);
    }
    return k;
}

__device__ __forceinline__ uint64_t u64_of(uint32_t lo, uint32_t hi) { return (uint64_t)lo | ((uint64_t)hi << 32); }

// ---------------------------------------------------------------------------------------------------------
// Block reduction of NOUT doubles per thread -> partials[blockIdx.x][*]; the last block to finish folds the
// partials in a fixed order (deterministic for a given grid) into out[] (+= when accumulate).
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int NOUT_MAX>
__device__ __forceinline__ void block_reduce_and_finish(const double *vals, int nout, double *partials,
                                                        unsigned int *ticket, double *out, bool accumulate)
{
    __shared__ double s_w[kWarpsPerBlock][NOUT_MAX];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < NOUT_MAX; ++i) {
        if (i < nout) {
            double v = warp_sum(vals[i]);
            if (lane == 0) s_w[warp][i] = v;
        }
    }
    __syncthreads();
    if (threadIdx.x < nout) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < kWarpsPerBlock; ++w) v += s_w[w][threadIdx.x];
        partials[(size_t)blockIdx.x * NOUT_MAX + threadIdx.x] = v;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = atomicAdd(ticket, 1u);
        s_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // fold: thread t sums blocks t, t+kBlock, ... for each output; then a block tree over threads
    for (int i = 0; i < nout; ++i) {
        double v = 0.0;
        for (unsigned int b = threadIdx.x; b < gridDim.x; b += kBlock)
            v += __ldcg(&partials[(size_t)b * NOUT_MAX + i]);
        v = warp_sum(v);
        __syncthreads();
        if (lane == 0) s_w[warp][0] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
#pragma unroll
            for (int w = 0; w < kWarpsPerBlock; ++w) t += s_w[w][0];
            out[i] = accumulate ? out[i] + t : t;
        }
    }
    if (threadIdx.x == 0) *ticket = 0u;  // re-arm for the next launch on this stream
}

// ---------------------------------------------------------------------------------------------------------
// K1: fused sweep, native Philox, single-move pools (multi-move pools: sweep_multi_kernel below).
// ---------------------------------------------------------------------------------------------------------
//
// SERIES (single-move pools): the launch covers n_series consecutive store intervals.  The chain stays in registers
// across ALL of them (HBM traffic 24/(ΣK) B per chain-step, per-chain prologue paid once) and the callback sums of
// every interval are accumulated per thread in shared memory -- Σe as f64, the accepted-count INCREMENT of the
// interval as u32 -- then block-reduced once at the end of the launch into series_partials; series_fold_kernel
// turns the partials into one [Σe, Σacc/t, count] record per store.  No host round trip and no second launch per
// store: StoreCallbacks at every 10th step costs the same as one K = 10·n_series sweep.
template <int POT, int ARITH, bool SERIES = false, bool BETAS = true>
__global__ void __launch_bounds__(kBlock, kSweepMinBlocks) sweep_philox_kernel(const SweepParams p)
{
    // dynamic shared memory: [MathTables][kernel-specific arrays] -- ONE symbol, so one pinned base register serves
    // the math tables and the series accumulators alike
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr uint32_t kTabBytes = (uint32_t)sizeof(m64::MathTables);
    load_tables(reinterpret_cast<m64::MathTables *>(smem_raw), p.tables);
    __syncthreads();
    const m64::Tab tb = shared_tab(smem_raw);
    // SERIES: [n_series][kBlock] f64 Σe, [n_series][kBlock] u32 ΣΔacc, [kBlock] u64 Σacc at entry, as byte addresses
    const uint32_t a_se = tb.s + kTabBytes + 8u * threadIdx.x;
    const uint32_t a_da = tb.s + kTabBytes + (SERIES ? 8u * kBlock * (uint32_t)p.n_series : 0u) + 4u * threadIdx.x;
    const uint32_t a_base = tb.s + kTabBytes + (SERIES ? 12u * kBlock * (uint32_t)p.n_series : 0u) + 8u * threadIdx.x;
    if constexpr (SERIES) {
        for (int s = 0; s < p.n_series; ++s) {
            sts_f64(a_se + 8u * kBlock * s, 0.0);
            sts_u32(a_da + 4u * kBlock * s, 0u);
        }
        sts_u64(a_base, 0ull);
    }

    const int64_t tend = p.t0 + p.K;
    double sum_e = 0.0;
    unsigned long long sum_acc = 0ull;   // Σ accepted_calls: exact in integers; every chain shares tot = tend
    uint32_t cnt = 0;
    // (the BETAS = false instantiation -- the headline kernel -- keeps σ as a constant-bank operand; a handle whose
    // optimiser runs on the device is routed to the BETAS = true one)
    const bool dev = BETAS && p.theta != nullptr;
    const double sigma0 = dev ? p.theta->sigma[0] : p.pool.sigma[0], lognorm0 = dev ? p.theta->lognorm[0] : p.pool.lognorm[0],
                 inv0 = dev ? p.theta->inv2s2[0] : p.pool.inv2s2[0];
    // Steps are consumed in Box-Muller pairs (pair index = step >> 1).  A run of steps [ta, tb) that starts on an odd
    // step uses only the sine half of its first pair and one that ends on an even step only the cosine half of its
    // last, so the result does not depend on how the steps are chunked into launches or store intervals.

    const uint32_t magic = floor_magic_reg();
    const int64_t stride = (int64_t)gridDim.x * kBlock;
    int64_t c = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    // the next chain's state is fetched while the current chain runs its K serial steps (hides the HBM latency
    // that would otherwise be exposed once per chain at the top of the loop)
    // (a series launch runs >= 100 steps per chain: there the load latency is noise and the three prefetch registers
    // are worth more to the loop body)
    constexpr bool PREFETCH = !SERIES;
    double x_next = (PREFETCH && c < p.M) ? p.x[c] : 0.0;
    uint32_t acc_next = (PREFETCH && c < p.M) ? p.acc[c] : 0u;
    for (; c < p.M; c += stride) {
        double x;
        uint32_t acc;
        if constexpr (PREFETCH) {
            x = x_next;
            acc = acc_next;
            if (c + stride < p.M) {
                x_next = p.x[c + stride];
                acc_next = p.acc[c + stride];
            }
        } else {
            x = p.x[c];
            acc = p.acc[c];
        }
        double e = potential<POT, ARITH>(x);
        // BETAS = false: β is a kernel-parameter constant (a constant-bank operand, no registers)
        const double beta_nat = BETAS ? (p.betas ? p.betas[c] : p.beta) : p.beta;
        // FAST: the accept argument is formed in binary-log units (CellM), β·log2e·(e − e')
        const double beta = ARITH == ARITH_FAST ? beta_nat * 1.4426950408889634 : beta_nat;
        const uint64_t sid = p.sid0 + (uint64_t)c;

        // chain-only halves of the first three Philox rounds (rng.cuh); the rare refinement block is generated unhoisted
        const PhiloxChain<kTagMetropolis, 0> ph(sid);
        // Draws of one pair of steps (a pure function of the pair index, independent of the chain state).
        // ONE Philox block feeds the pair: words B0/B1 give the two 53-bit Box-Muller uniforms (top 53 bits) and,
        // in their low 11 bits, the PREFIXES of the two accept uniforms.  The remaining 42 bits of an accept
        // uniform come from sub-block 1 of the pair and are only generated when the FP32 filter cannot decide (lazy refinement).
        struct PairDraws {
            double z0, z1;
            uint32_t f0, f1;   // 12-bit / 11-bit prefixes of u_acc(2p), u_acc(2p+1), OR-ed into the filter's magic bits
            uint64_t pr;
        };
        auto gen_pair = [&](uint64_t pr) {
            PairDraws d;
            const U64Pair b0 = ph.block((uint32_t)pr);
            m64::box_muller_u64(u64_of(b0.a_lo, b0.a_hi), u64_of(b0.b_lo, b0.b_hi), tb, d.z0, d.z1);
            d.f0 = m64::exp_prefix_bits<12>(b0.a_lo, magic);   // 12 bits: the radius uniform takes A >> 12
            d.f1 = m64::exp_prefix_bits<11>(b0.b_lo, magic);   // (as the accept filter's addend bits: magic | prefix)
            d.pr = pr;
            return d;
        };
        // the two (state-dependent, serial) Metropolis steps of a pair; DO0 / DO1 are compile-time
        auto do_steps = [&](const PairDraws &d, auto do0, auto do1) {
            if constexpr (decltype(do0)::value) {
                auto exact_u = [&]() {
                    const U64Pair r = philox_block<kTagMetropolis>(sid, d.pr, 1);
                    return m64::u53_prefix_refine<12>(d.f0 & 0xfffu, r.a_lo, r.a_hi);
                };
                const CellM<12> ulo{d.f0};
                const uint32_t a = mc_step<POT, ARITH>(x, e, beta, sigma0, lognorm0, inv0, d.z0, ulo, exact_u, tb);
                count_if(acc, a);
            }
            if constexpr (decltype(do1)::value) {
                auto exact_u = [&]() {
                    const U64Pair r = philox_block<kTagMetropolis>(sid, d.pr, 1);
                    return m64::u53_prefix_refine<11>(d.f1 & 0x7ffu, r.b_lo, r.b_hi);
                };
                const CellM<11> ulo{d.f1};
                const uint32_t a = mc_step<POT, ARITH>(x, e, beta, sigma0, lognorm0, inv0, d.z1, ulo, exact_u, tb);
                count_if(acc, a);
            }
        };
        using T_ = std::true_type;
        using F_ = std::false_type;
        auto run_steps = [&](uint32_t ta, uint32_t tb) {     // MC steps [ta, tb) of this chain; t < 2^32 (host check)
        if (tb <= ta) return;    // empty interval (two stores with no Metropolis step between them): with an odd ta
                                 // the lead step below would run and tb - tfull would wrap around
        const bool lead = (ta & 1u) != 0;
        const uint32_t tfull = ta + (lead ? 1u : 0u);
        const int npairs = (int)((tb - tfull) >> 1);
        const bool trail = ((tb - tfull) & 1u) != 0;
        uint64_t pr = (uint64_t)(ta >> 1);
        if (lead) { do_steps(gen_pair(pr), F_{}, T_{}); ++pr; }
#pragma unroll 1
        for (int i = 0; i < npairs; ++i, ++pr) do_steps(gen_pair(pr), T_{}, T_{});
        if (trail) do_steps(gen_pair(pr), T_{}, F_{});
        };
        if constexpr (SERIES) {
            sts_u64(a_base, lds_u64(a_base) + acc);
            uint32_t acc_prev = acc, ta = (uint32_t)p.t0;
            if (p.series_even) {
                // whole pairs only: ONE flat loop over the pairs of all intervals; a countdown marks the store points
                // (a nested interval/pair loop makes the compiler rebuild the per-chain Philox constants in every
                // interval's preheader: measured 6 % slower than this form)
                // Loop control is ONE add, compare and branch per pair: the pair index is compared with the index of the
                // next store point, and the end of the launch (always a store point) is tested inside that rare block
                // (a countdown + the loop's own counter cost seven instructions per pair in an issue-bound loop)
                int s = 0;
                uint32_t pr = ta >> 1;
                uint32_t next = pr + ((uint32_t)p.series_K[0] >> 1);
#pragma unroll 1
                for (;;) {
                    do_steps(gen_pair((uint64_t)pr), T_{}, T_{});
                    if (++pr == next) {
                        sts_f64(a_se + 8u * kBlock * s, lds_f64(a_se + 8u * kBlock * s) + potential<POT, ARITH>(x));
                        sts_u32(a_da + 4u * kBlock * s, lds_u32(a_da + 4u * kBlock * s) + (acc - acc_prev));
                        acc_prev = acc;
                        if (++s == p.n_series) break;
                        next += (uint32_t)p.series_K[s] >> 1;
                    }
                }
            } else
#pragma unroll 1
            for (int s = 0; s < p.n_series; ++s) {
                const uint32_t tb = ta + (uint32_t)p.series_K[s];
                run_steps(ta, tb);
                sts_f64(a_se + 8u * kBlock * s, lds_f64(a_se + 8u * kBlock * s) + potential<POT, ARITH>(x));  // Σ e
                sts_u32(a_da + 4u * kBlock * s, lds_u32(a_da + 4u * kBlock * s) + (acc - acc_prev));          // accepted here
                acc_prev = acc;
                ta = tb;
            }
        } else {
            run_steps((uint32_t)p.t0, (uint32_t)tend);
        }

        p.x[c] = x;
        p.acc[c] = acc;
        if (p.reduce) {
            sum_e += potential<POT, ARITH>(x);   // callback_energy: Σ system.e, e == potential(x) always
            sum_acc += acc;      // callback_acceptance: Σ_c acc_c/tot with tot == tend for every chain
            ++cnt;
        }
    }

    if constexpr (SERIES) {
        // one block reduction per interval, in a fixed order (deterministic for a given grid); integer-valued sums
        // are exact in binary64 (< 2^53)
        __shared__ double s_w[kWarpsPerBlock][2];
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        for (int s = 0; s <= p.n_series; ++s) {
            double v0, v1;
            if (s < p.n_series) {
                v0 = lds_f64(a_se + 8u * kBlock * s);
                v1 = (double)lds_u32(a_da + 4u * kBlock * s);
            } else {
                v0 = (double)lds_u64(a_base);
                v1 = 0.0;
            }
            v0 = warp_sum(v0);
            v1 = warp_sum(v1);
            __syncthreads();
            if (lane == 0) { s_w[warp][0] = v0; s_w[warp][1] = v1; }
            __syncthreads();
            if (threadIdx.x < 2) {
                double t = 0.0;
#pragma unroll
                for (int w = 0; w < kWarpsPerBlock; ++w) t += s_w[w][threadIdx.x];
                p.series_partials[((size_t)blockIdx.x * (p.n_series + 1) + s) * 2 + threadIdx.x] = t;
            }
        }
        return;
    }
    if (p.reduce) {
        // Σ acc_c / tot == (Σ acc_c) / tot exactly in real arithmetic; the integer sum is exact in binary64 (< 2^53)
        // and ONE division replaces a DDIV per chain.  0/0 = NaN at t = 0, like the reference's store_first record.
        double vals[3] = {sum_e, (double)sum_acc / (double)tend, (double)cnt};
        block_reduce_and_finish<3>(vals, 3, p.partials, p.ticket, p.sums, false);
    }
}

// Series fold: CTA s turns the per-CTA partials of a series launch into the callback record of store s,
//   out[s] = [Σ_c e_c(t_s), (Σ_c acc_c(t_s)) / t_s, M]   with  Σ acc(t_s) = Σ acc(entry) + Σ_{s' <= s} ΣΔacc(s')
// (same definition as the fused reduction of the plain sweep: Σ_c acc_c/tot with tot == t_s for every chain).
// The last CTA's record is also copied to `sums` so that arianna_callbacks() after a series needs no extra pass.
struct SeriesK { int k[kMaxSeries]; };
__global__ void __launch_bounds__(kBlock) series_fold_kernel(const double *partials, int n_ctas, int n_series,
                                                             int64_t t0, const SeriesK series_K, int64_t M,
                                                             double *out, double *sums, int accumulate)
{
    __shared__ double s_w[kWarpsPerBlock][2];
    __shared__ int64_t s_t;
    const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        int64_t t = t0;
        for (int i = 0; i <= s; ++i) t += series_K.k[i];
        s_t = t;
    }
    double e = 0.0, a = 0.0;
    for (int b = threadIdx.x; b < n_ctas; b += kBlock) {
        const double *row = partials + (size_t)b * (n_series + 1) * 2;
        e += row[2 * s];
        a += row[2 * n_series];                       // Σacc at entry
        for (int i = 0; i <= s; ++i) a += row[2 * i + 1];
    }
    e = warp_sum(e);
    a = warp_sum(a);
    if (lane == 0) { s_w[warp][0] = e; s_w[warp][1] = a; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double te = 0.0, ta = 0.0;
#pragma unroll
        for (int w = 0; w < kWarpsPerBlock; ++w) { te += s_w[w][0]; ta += s_w[w][1]; }
        // accumulate: this launch covered one SLICE of the chains (arianna_run_host_job); slices are folded one after
        // the other on one stream, so the sum order is fixed
        double r0 = te, r1 = ta / (double)s_t, r2 = (double)M;
        if (accumulate) { r0 += out[3 * s]; r1 += out[3 * s + 1]; r2 += out[3 * s + 2]; }
        out[3 * s] = r0; out[3 * s + 1] = r1; out[3 * s + 2] = r2;
        if (s == n_series - 1 && sums) { sums[0] = r0; sums[1] = r1; sums[2] = r2; }
    }
}

// ---------------------------------------------------------------------------------------------------------
// K6: replay sweep -- consumes caller-supplied draws, always EXACT arithmetic.  HBM-bound: 16 B (24 B with
// u_cat) of draws per chain-step.  Draws are streamed with evict-first loads, 4 steps prefetched ahead.
// ---------------------------------------------------------------------------------------------------------
struct ReplayParams {
    double *x;
    uint32_t *acc;
    uint32_t *tot;
    const double *betas;
    double beta;
    int64_t M;
    int64_t K;
    const double *u_cat;  // [K][M] or nullptr
    const double *z;      // [K][M]
    const double *u_acc;  // [K][M]
    uint8_t *decisions;   // [K][M] or nullptr
    const m64::MathTables *tables;
    PoolParams pool;
};

template <int POT, bool MULTI>
__global__ void __launch_bounds__(kBlock) sweep_replay_kernel(const ReplayParams p)
{
    extern __shared__ unsigned char smem_raw[];
    uint32_t *s_acc = reinterpret_cast<uint32_t *>(smem_raw);
    uint32_t *s_tot = s_acc + (MULTI ? p.pool.n_moves * kBlock : 0);
    __shared__ double s_sigma[kMaxMoves], s_weight[kMaxMoves], s_lognorm[kMaxMoves], s_inv[kMaxMoves];
    if (threadIdx.x < kMaxMoves) {
        s_sigma[threadIdx.x] = p.pool.sigma[threadIdx.x];
        s_weight[threadIdx.x] = p.pool.weight[threadIdx.x];
        s_lognorm[threadIdx.x] = p.pool.lognorm[threadIdx.x];
        s_inv[threadIdx.x] = p.pool.inv2s2[threadIdx.x];
    }
    __shared__ m64::MathTables s_T;
    load_tables(&s_T, p.tables);
    __syncthreads();
    const m64::Tab tb = shared_tab(&s_T);
    const int nm = p.pool.n_moves;
    constexpr int PF = 4;

    for (int64_t c = (int64_t)blockIdx.x * kBlock + threadIdx.x; c < p.M; c += (int64_t)gridDim.x * kBlock) {
        double x = p.x[c];
        double e = potential<POT, ARITH_EXACT>(x);
        const double beta = p.betas ? p.betas[c] : p.beta;
        uint32_t acc = 0;
        if constexpr (MULTI) {
            for (int k = 0; k < nm; ++k) {
                s_acc[k * kBlock + threadIdx.x] = p.acc[(size_t)k * p.M + c];
                s_tot[k * kBlock + threadIdx.x] = p.tot[(size_t)k * p.M + c];
            }
        } else {
            acc = p.acc[c];
        }
        // Bursts of PF steps: request the draws of PF steps, then run the PF serial steps.  (A rolling register queue
        // that re-requests a slot as soon as it is consumed was measured SLOWER on B200: +14..29 registers cost more
        // occupancy than the smoother request stream gained -- 4.5 vs 4.8 TB/s.)
        for (int64_t s0 = 0; s0 < p.K; s0 += PF) {
            double zz[PF], ua[PF], uc[PF];
#pragma unroll
            for (int i = 0; i < PF; ++i) {
                if (s0 + i < p.K) {
                    const size_t o = (size_t)(s0 + i) * p.M + c;
                    zz[i] = __ldcs(p.z + o);
                    ua[i] = __ldcs(p.u_acc + o);
                    uc[i] = (MULTI && p.u_cat) ? __ldcs(p.u_cat + o) : 0.0;
                }
            }
#pragma unroll
            for (int i = 0; i < PF; ++i) {
                if (s0 + i < p.K) {
                    int d;
                    if constexpr (MULTI) {
                        const int k = categorical(nm, s_weight, uc[i]);
                        d = mc_step_exact<POT>(x, e, beta, s_sigma[k], s_lognorm[k], s_inv[k], zz[i], ua[i], tb);
                        s_acc[k * kBlock + threadIdx.x] += d;
                        s_tot[k * kBlock + threadIdx.x] += 1;
                    } else {
                        d = mc_step_exact<POT>(x, e, beta, s_sigma[0], s_lognorm[0], s_inv[0], zz[i], ua[i], tb);
                        acc += d;
                    }
                    if (p.decisions) __stcs(p.decisions + (size_t)(s0 + i) * p.M + c, (uint8_t)d);
                }
            }
        }
        p.x[c] = x;
        if constexpr (MULTI) {
            for (int k = 0; k < nm; ++k) {
                p.acc[(size_t)k * p.M + c] = s_acc[k * kBlock + threadIdx.x];
                p.tot[(size_t)k * p.M + c] = s_tot[k * kBlock + threadIdx.x];
            }
        } else {
            p.acc[c] = acc;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// XOSHIRO sweep: the reference's own draw order per step -- u_cat = rand, z = randn, u_acc = rand
// (metropolis.jl:206, particle_1d.jl:57, metropolis.jl:184) -- from a per-chain xoshiro256++ state in HBM.
// ---------------------------------------------------------------------------------------------------------
struct XoshiroParams {
    double *x;
    uint32_t *acc;
    uint32_t *tot;
    const double *betas;
    double beta;
    int64_t M;
    int64_t K;
    uint64_t *rng;        // [M][4]
    const uint64_t *ki;   // ziggurat tables in global memory (copied to shared)
    const double *wi;
    const double *fi;
    const m64::MathTables *tables;
    PoolParams pool;
};

template <int POT, int ARITH, bool MULTI>
__global__ void __launch_bounds__(kBlock) sweep_xoshiro_kernel(const XoshiroParams p)
{
    extern __shared__ unsigned char smem_raw[];
    uint32_t *s_acc = reinterpret_cast<uint32_t *>(smem_raw);
    uint32_t *s_tot = s_acc + (MULTI ? p.pool.n_moves * kBlock : 0);
    __shared__ double s_sigma[kMaxMoves], s_weight[kMaxMoves], s_lognorm[kMaxMoves], s_inv[kMaxMoves];
    __shared__ uint64_t s_ki[256];
    __shared__ double s_wi[256], s_fi[256];
    __shared__ m64::MathTables s_T;
    load_tables(&s_T, p.tables);
    if (threadIdx.x < kMaxMoves) {
        s_sigma[threadIdx.x] = p.pool.sigma[threadIdx.x];
        s_weight[threadIdx.x] = p.pool.weight[threadIdx.x];
        s_lognorm[threadIdx.x] = p.pool.lognorm[threadIdx.x];
        s_inv[threadIdx.x] = p.pool.inv2s2[threadIdx.x];
    }
    for (int i = threadIdx.x; i < 256; i += kBlock) {
        s_ki[i] = p.ki[i];
        s_wi[i] = p.wi[i];
        s_fi[i] = p.fi[i];
    }
    __syncthreads();
    const m64::Tab tb = shared_tab(&s_T);
    const ZigTables T{s_ki, s_wi, s_fi};
    const int nm = p.pool.n_moves;

    for (int64_t c = (int64_t)blockIdx.x * kBlock + threadIdx.x; c < p.M; c += (int64_t)gridDim.x * kBlock) {
        double x = p.x[c];
        double e = potential<POT, ARITH>(x);
        const double beta = p.betas ? p.betas[c] : p.beta;
        const ulonglong2 r01 = *reinterpret_cast<const ulonglong2 *>(p.rng + 4 * c);
        const ulonglong2 r23 = *reinterpret_cast<const ulonglong2 *>(p.rng + 4 * c + 2);
        Xoshiro g{r01.x, r01.y, r23.x, r23.y};
        uint32_t acc = 0;
        if constexpr (MULTI) {
            for (int k = 0; k < nm; ++k) {
                s_acc[k * kBlock + threadIdx.x] = p.acc[(size_t)k * p.M + c];
                s_tot[k * kBlock + threadIdx.x] = p.tot[(size_t)k * p.M + c];
            }
        } else {
            acc = p.acc[c];
        }
        for (int64_t s = 0; s < p.K; ++s) {
            const double uc = g.rand();  // always consumed, even when n_moves == 1 (metropolis.jl:206)
            const double zz = xoshiro_randn(g, T);
            const uint64_t uaw = g.next();  // rand(rng) = (next >> 11)·2^-53 [EXT]
            const uint32_t ua_lo = (uint32_t)uaw, ua_hi = (uint32_t)(uaw >> 32);
            auto exact_u = [&]() { return u53(ua_lo, ua_hi); };
            const CellF ulo{m64::ulo_from_word23(ua_hi), 0x1p-23f};
            if constexpr (MULTI) {
                const int k = categorical(nm, s_weight, uc);
                const bool d = mc_step<POT, ARITH>(x, e, beta, s_sigma[k], s_lognorm[k], s_inv[k], zz, ulo, exact_u,
                                                   tb);
                if (d) s_acc[k * kBlock + threadIdx.x] += 1;
                s_tot[k * kBlock + threadIdx.x] += 1;
            } else {
                (void)uc;
                if (mc_step<POT, ARITH>(x, e, beta, s_sigma[0], s_lognorm[0], s_inv[0], zz, ulo, exact_u, tb))
                    ++acc;
            }
        }
        p.x[c] = x;
        *reinterpret_cast<ulonglong2 *>(p.rng + 4 * c) = make_ulonglong2(g.s0, g.s1);
        *reinterpret_cast<ulonglong2 *>(p.rng + 4 * c + 2) = make_ulonglong2(g.s2, g.s3);
        if constexpr (MULTI) {
            for (int k = 0; k < nm; ++k) {
                p.acc[(size_t)k * p.M + c] = s_acc[k * kBlock + threadIdx.x];
                p.tot[(size_t)k * p.M + c] = s_tot[k * kBlock + threadIdx.x];
            }
        } else {
            p.acc[c] = acc;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// K2 (standalone): callback sums over the resident state.  sums = [Σ e, Σ_c acc_ck/tot_ck (k < n_moves), count].
// Used for multi-move pools and whenever callbacks are requested without a preceding fused-reduce sweep.
// ---------------------------------------------------------------------------------------------------------
struct ReduceParams {
    const double *x;
    const uint32_t *acc;
    const uint32_t *tot;   // nullptr -> steps_done
    int64_t M;
    int64_t steps_done;
    int n_moves;
    int potential;
    double *partials;
    unsigned int *ticket;
    double *sums;
};

__global__ void __launch_bounds__(kBlock) callback_reduce_kernel(const ReduceParams p)
{
    double vals[kMaxOut];
#pragma unroll
    for (int i = 0; i < kMaxOut; ++i) vals[i] = 0.0;
    for (int64_t c = (int64_t)blockIdx.x * kBlock + threadIdx.x; c < p.M; c += (int64_t)gridDim.x * kBlock) {
        const double x = p.x[c];
        double e;
        if (p.potential == POT_HARMONIC) e = potential<POT_HARMONIC, ARITH_EXACT>(x);
        else if (p.potential == POT_QUARTIC) e = potential<POT_QUARTIC, ARITH_EXACT>(x);
        else e = potential<POT_DOUBLE_WELL, ARITH_EXACT>(x);
        vals[0] += e;
#pragma unroll
        for (int k = 0; k < kMaxMoves; ++k) {
            if (k < p.n_moves) {
                const double a = (double)p.acc[(size_t)k * p.M + c];
                const double t = p.tot ? (double)p.tot[(size_t)k * p.M + c] : (double)p.steps_done;
                vals[1 + k] += a / t;
            }
        }
        vals[kMaxOut - 1] += 1.0;
    }
    // count is exported right after the per-move sums: move it to slot 1 + n_moves
    double cnt = vals[kMaxOut - 1];
#pragma unroll
    for (int k = 0; k < kMaxOut; ++k)
        if (k == 1 + p.n_moves) vals[k] = cnt;
    block_reduce_and_finish<kMaxOut>(vals, 2 + p.n_moves, p.partials, p.ticket, p.sums, false);
}

// Per-move totals of the counters (what a single-ensemble host Move would hold): out[k] = Σ_c acc, out[nm+k] = Σ_c tot
__global__ void __launch_bounds__(kBlock) counter_sum_kernel(const uint32_t *acc, const uint32_t *tot, int64_t M,
                                                             int n_moves, int64_t steps_done,
                                                             unsigned long long *out)
{
    for (int k = 0; k < n_moves; ++k) {
        unsigned long long a = 0, t = 0;
        for (int64_t c = (int64_t)blockIdx.x * kBlock + threadIdx.x; c < M; c += (int64_t)gridDim.x * kBlock) {
            a += acc[(size_t)k * M + c];
            t += tot ? tot[(size_t)k * M + c] : (unsigned long long)steps_done;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o);
            t += __shfl_xor_sync(0xffffffffu, t, o);
        }
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(out + k, a);           // integer atomics: order-independent, deterministic
            atomicAdd(out + n_moves + k, t);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// K3: PGMC estimator, ALL learnable moves in one launch (the reference's outer loop, estimator.jl:112, runs inside the
// kernel: one launch and one tail per estimator pass instead of n_learn).  Per learnable move and chain: q_batch x
// pgmc_estimate (gradients.jl:93-109) with the analytic ∂σ log q; sums of (j, ∇j, ∇logq_forward, g, n) are
// block-reduced and ADDED to gd[l][5] by the last block (gradients_data[k] += gd, estimator.jl:130).  Every thread
// visits the same chains for every move, so the EXACT variant's perform/undo drift of x carries from move to move
// exactly as in the reference's sequential loop.  REPLAY reads z[n_learn][q_batch][M] instead of the estimator stream.
// ---------------------------------------------------------------------------------------------------------
struct PgmcParams {
    double *x;
    const double *betas;
    double beta;
    int64_t M;
    int q_batch;
    int n_learn;
    int64_t q0;           // estimator samples already drawn per chain (draw index base of the first learnable move)
    uint64_t sid0;
    double sigma[kMaxMoves];     // of the learnable moves, in order
    double lognorm[kMaxMoves];
    int learn_id[kMaxMoves];     // pool index of each learnable move
    const DevTheta *theta;       // non-null: σ lives on the device
    const double *z;      // replay only
    double *partials;     // [n_learn][gridDim.x][5]
    unsigned int *ticket; // [n_learn]
    double *gd;           // [n_learn][5] accumulators
    const m64::MathTables *tables;
};

template <int POT, int ARITH>
__device__ __forceinline__ void pgmc_sample(double &x, double &e, double beta, double sigma, double lognorm,
                                            double z, double &sj, double &sdj, double &sgf, double &sg,
                                            m64::Tab tb)
{
    if constexpr (ARITH == ARITH_EXACT) {
        double delta = __dadd_rn(0.0, __dmul_rn(sigma, z));                                    // gradients.jl:119
        double s2 = __dmul_rn(sigma, sigma);
        // ∂σ log q = δ²/σ³ − 1/σ, evaluated as (δ·δ)/((σ·σ)·σ) − 1/σ (oracle: ao_dlogq_dsigma)
        double gf = __dsub_rn(__ddiv_rn(__dmul_rn(delta, delta), __dmul_rn(s2, sigma)), __ddiv_rn(1.0, sigma));
        double lqf = __dsub_rn(__ddiv_rn(-__dmul_rn(delta, delta), __dmul_rn(2.0, s2)), lognorm);
        double e1 = e;
        x = __dadd_rn(x, delta);                                                               // :98
        e = potential<POT, ARITH_EXACT>(x);
        double dlogp = __dsub_rn(__dmul_rn(-e, beta), __dmul_rn(-e1, beta));                   // :99
        double r = __dmul_rn(delta, delta);                                                    // :100
        delta = -delta;                                                                        // :101
        double gb = gf, lqb = lqf;                                                             // :102 (even in δ)
        x = __dadd_rn(x, delta);                                                               // :103 undo (drifts)
        e = potential<POT, ARITH_EXACT>(x);
        double ex = exp(__dsub_rn(__dadd_rn(dlogp, lqb), lqf));                                // :104
        double alpha = (ex > 1.0) ? 1.0 : ex;
        double j = __dmul_rn(r, alpha);                                                        // :105
        double dj = __dmul_rn(j, (alpha == 1.0) ? gf : gb);                                    // :106
        sj += j; sdj += dj; sgf += gf; sg += __dmul_rn(gf, gf);                                // :107, :68-76
    } else {
        // FAST accumulates the σ-free quantities; pgmc_kernel applies the powers of σ once per thread:
        //   j = δ²α = σ²·(z²α),  ∂σ log q = (z² − 1)/σ,  ∇j = j·∂σ log q = σ·(z²α)(z² − 1),  g = (z² − 1)²/σ²
        (void)lognorm;
        const double z2 = z * z;
        const double w = fma(z, z, -1.0);
        const double xn = fma(sigma, z, x);
        const double en = potential<POT, ARITH_FAST>(xn);
        const double alpha = m64::exp_nonpos(beta * (e - en), tb);   // = min(1, exp(·))
        const double ja = z2 * alpha;
        sj += ja; sdj = fma(ja, w, sdj); sgf += w; sg = fma(w, w, sg);
    }
}

template <int POT, int ARITH, bool REPLAY>
__global__ void __launch_bounds__(kBlock, kPgmcMinBlocks) pgmc_kernel(const PgmcParams p)
{
    __shared__ m64::MathTables s_T;
    load_tables(&s_T, p.tables);
    __syncthreads();
    const m64::Tab tb = shared_tab(&s_T);
#pragma unroll 1
    for (int l = 0; l < p.n_learn; ++l) {
        const double sigma = p.theta ? p.theta->sigma[p.learn_id[l]] : p.sigma[l];
        const double lognorm = p.theta ? p.theta->lognorm[p.learn_id[l]] : p.lognorm[l];
        const int64_t q0 = p.q0 + (int64_t)l * p.q_batch, qend = q0 + p.q_batch;
        double sj = 0.0, sdj = 0.0, sgf = 0.0, sg = 0.0, sn = 0.0;
        for (int64_t c = (int64_t)blockIdx.x * kBlock + threadIdx.x; c < p.M; c += (int64_t)gridDim.x * kBlock) {
            double x = p.x[c];
            double e = potential<POT, ARITH>(x);
            const double beta = p.betas ? p.betas[c] : p.beta;
            if constexpr (REPLAY) {
                const double *zl = p.z + (size_t)l * p.q_batch * p.M;
                for (int b = 0; b < p.q_batch; ++b)
                    pgmc_sample<POT, ARITH>(x, e, beta, sigma, lognorm, __ldcs(zl + (size_t)b * p.M + c), sj, sdj, sgf, sg, tb);
            } else {
                const uint64_t sid = p.sid0 + (uint64_t)c;
                const PhiloxChain<kTagEstimator, 0> ph(sid);
                // samples [q0, qend) of this chain's estimator stream, two per Box-Muller pair; only the first / last
                // pair of a move can be split (q < 2^33, host check)
                auto pair = [&](uint32_t pr, bool do0, bool do1) {
                    const U64Pair blk = ph.block(pr);
                    double z0, z1;
                    m64::box_muller_u64(u64_of(blk.a_lo, blk.a_hi), u64_of(blk.b_lo, blk.b_hi), tb, z0, z1);
                    if (do0) pgmc_sample<POT, ARITH>(x, e, beta, sigma, lognorm, z0, sj, sdj, sgf, sg, tb);
                    if (do1) pgmc_sample<POT, ARITH>(x, e, beta, sigma, lognorm, z1, sj, sdj, sgf, sg, tb);
                };
                const bool lead = (q0 & 1) != 0, trail = (qend & 1) != 0;
                uint32_t pr = (uint32_t)(q0 >> 1);
                const uint32_t pr_end = (uint32_t)(qend >> 1);      // first pair that is not complete
                if (lead) { pair(pr, false, true); ++pr; }
#pragma unroll 1
                for (; pr < pr_end; ++pr) pair(pr, true, true);
                if (trail) pair(pr, true, false);
            }
            sn += (double)p.q_batch;
            if constexpr (ARITH == ARITH_EXACT) p.x[c] = x;  // perform/undo rounding drift is part of the reference
        }
        if constexpr (ARITH == ARITH_FAST) {   // the powers of σ factored out of pgmc_sample
            const double s1 = sigma, i1 = 1.0 / sigma;
            sj *= s1 * s1; sdj *= s1; sgf *= i1; sg *= i1 * i1;
        }
        double vals[5] = {sj, sdj, sgf, sg, sn};
        __syncthreads();                       // the reduction's shared scratch is reused from move to move
        block_reduce_and_finish<5>(vals, 5, p.partials + (size_t)l * gridDim.x * 5, p.ticket + l, p.gd + 5 * l, true);
    }
}

// ---------------------------------------------------------------------------------------------------------
// PolicyGradientUpdate on the device (update.jl:50-57 + learning.jl): thread l averages the accumulated GradientData of
// learnable move l (gradients.jl:83-85), applies its optimiser's learning_step! -- the six rules restated operation by
// operation as oracle/arianna_oracle.c:ao_learning_step, IEEE sqrt / division, nothing contracted -- writes σ and the
// constants derived from it to the device-resident parameter block, and zeroes the accumulator (update.jl:55).
// ---------------------------------------------------------------------------------------------------------
enum { OPT_STATIC = 0, OPT_VPG = 1, OPT_BLPG = 2, OPT_BLAPG = 3, OPT_NPG = 4, OPT_ANPG = 5, OPT_BLANPG = 6 };
struct UpdateParams {
    int n_learn;
    int learn_id[kMaxMoves];
    int kind[kMaxMoves];
    double p1[kMaxMoves];   // η (VPG, BLPG, NPG) or δ (BLAPG, ANPG, BLANPG)
    double p2[kMaxMoves];   // ϵid
};

__global__ void pgmc_update_kernel(DevTheta *th, double *gd, const UpdateParams u)
{
    const int l = threadIdx.x;
    if (l >= u.n_learn) return;
    const int k = u.learn_id[l];
    const double n = gd[5 * l + 4];
    const double j = __ddiv_rn(gd[5 * l], n), dj = __ddiv_rn(gd[5 * l + 1], n), glq = __ddiv_rn(gd[5 * l + 2], n),
                 g = __ddiv_rn(gd[5 * l + 3], n);
    const double theta = th->sigma[k], p1 = u.p1[l], p2 = u.p2[l];
    double out = theta;
    switch (u.kind[l]) {
    case OPT_VPG: out = __dadd_rn(theta, __dmul_rn(p1, dj)); break;                                        // learning.jl:32-34
    case OPT_BLPG: out = __dadd_rn(theta, __dmul_rn(p1, __dsub_rn(dj, __dmul_rn(j, glq)))); break;         // :50-52
    case OPT_BLAPG: {                                                                                      // :76-79
        const double eta = __dsqrt_rn(__ddiv_rn(__dmul_rn(2.0, p1), __dadd_rn(__dmul_rn(dj, dj), p2)));
        out = __dadd_rn(theta, __dmul_rn(eta, __dsub_rn(dj, __dmul_rn(j, glq))));
        break;
    }
    case OPT_NPG: {                                                                                        // :103-105
        const double Finv = __ddiv_rn(1.0, __dadd_rn(g, __dmul_rn(p2, 1.0)));
        out = __dadd_rn(theta, __dmul_rn(__dmul_rn(p1, Finv), dj));
        break;
    }
    case OPT_ANPG: {                                                                                       // :130-134
        const double Finv = __ddiv_rn(1.0, __dadd_rn(g, __dmul_rn(p2, 1.0)));
        const double eta = __dsqrt_rn(__ddiv_rn(__dmul_rn(2.0, p1), __dmul_rn(dj, __dmul_rn(Finv, dj))));
        out = __dadd_rn(theta, __dmul_rn(__dmul_rn(eta, Finv), dj));
        break;
    }
    case OPT_BLANPG: {                                                                                     // :159-164
        const double Finv = __ddiv_rn(1.0, __dadd_rn(g, __dmul_rn(p2, 1.0)));
        const double bj = __dsub_rn(dj, __dmul_rn(j, glq));
        const double eta = __dsqrt_rn(__ddiv_rn(__dmul_rn(2.0, p1), __dmul_rn(bj, __dmul_rn(Finv, bj))));
        out = __dadd_rn(theta, __dmul_rn(__dmul_rn(eta, Finv), bj));
        break;
    }
    default: break;                                                                                        // Static
    }
    th->sigma[k] = out;
    const double s2 = __dmul_rn(out, out), d = __dmul_rn(2.0, s2);
    th->lognorm[k] = __ddiv_rn(log(__dmul_rn(6.283185307179586, s2)), 2.0);      // particle_1d.jl:53
    th->inv2s2[k] = (d >= 0x1p-300 && d <= 0x1p300) ? __ddiv_rn(1.0, d) : 0.0;
    if (!(out > 0.0) || isinf(out)) atomicOr(&th->bad, 1);
    for (int i = 0; i < 5; ++i) gd[5 * l + i] = 0.0;
}

// K5: synthetic initial condition x0 = 4u − 2 (MC_harmonic_oscillator.jl:13) from stream tag 0.
__global__ void __launch_bounds__(kBlock) init_kernel(double *x, int64_t M, uint64_t sid0)
{
    for (int64_t c = (int64_t)blockIdx.x * kBlock + threadIdx.x; c < M; c += (int64_t)gridDim.x * kBlock) {
        const U64Pair b = philox_block<kTagInit>(sid0 + (uint64_t)c, 0, 0);
        x[c] = __dsub_rn(__dmul_rn(4.0, u53(b.a_lo, b.a_hi)), 2.0);
    }
}

__global__ void __launch_bounds__(kBlock) energy_kernel(const double *x, double *e, int64_t M, int pot)
{
    for (int64_t c = (int64_t)blockIdx.x * kBlock + threadIdx.x; c < M; c += (int64_t)gridDim.x * kBlock) {
        const double v = x[c];
        if (pot == POT_HARMONIC) e[c] = potential<POT_HARMONIC, ARITH_EXACT>(v);
        else if (pot == POT_QUARTIC) e[c] = potential<POT_QUARTIC, ARITH_EXACT>(v);
        else e[c] = potential<POT_DOUBLE_WELL, ARITH_EXACT>(v);
    }
}

// Diagnostic: evaluates the device math layer (csrc/math64.cuh) on arrays so the tests can compare the DEVICE code
// paths (MUFU.RSQ64H seed, MUFU.EX2 filter) with long-double references.  kind: 0 exp_nonpos(x) | 1 neg2log_u53(k) |
// 2 sqrt_pos(x) | 3 sincos_turn53(k) -> out[2i], out[2i+1] | 4 box_muller_u64(a, b) -> out[2i], out[2i+1] |
// 5 accept test (x = a, prefix word = b, refinement word = c) -> out[2i] = filtered, out[2i+1] = reference decision |
// 6 / 7 Philox block of (sid = b, p = c[, sub = a]) through PhiloxChain / philox_block -> out[4i .. 4i+3] = the 4 words
// 10 / 11 accept test of the headline sweep (a = x·log2e, 11- / 12-bit prefix as addend bits) -> like 5 / 8
__global__ void __launch_bounds__(kBlock) debug_math_kernel(int kind, const double *a, const uint64_t *b,
                                                            const uint64_t *cc, double *out, int64_t n,
                                                            const m64::MathTables *tables)
{
    __shared__ m64::MathTables s_T;
    load_tables(&s_T, tables);
    __syncthreads();
    const m64::Tab tb = shared_tab(&s_T);
    for (int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x; i < n; i += (int64_t)gridDim.x * kBlock) {
        if (kind == 0) out[i] = m64::exp_nonpos(a[i], tb);
        else if (kind == 1) out[i] = m64::neg2log_u53(b[i], tb);
        else if (kind == 2) out[i] = m64::sqrt_pos(a[i]);
        else if (kind == 3) m64::sincos_turn53_tab((uint32_t)(b[i] >> 32), (uint32_t)b[i], tb, out[2 * i], out[2 * i + 1]);
        else if (kind == 4) m64::box_muller_u64(b[i], cc[i], tb, out[2 * i], out[2 * i + 1]);
        else if (kind == 9) out[i] = m64::neg2log_k52((uint32_t)(b[i] >> 32), (uint32_t)b[i], tb);
        else if (kind == 6 || kind == 7) {
            // Philox4x32-10 block (sid = b, p = c): 6 = per-chain hoisted form (sub 0), 7 = general form, sub = a
            U64Pair r;
            if (kind == 6) r = PhiloxChain<kTagMetropolis, 0>(b[i]).block((uint32_t)cc[i]);
            else r = philox_block<kTagMetropolis>(b[i], cc[i], (uint32_t)a[i]);
            out[4 * i] = (double)r.a_lo; out[4 * i + 1] = (double)r.a_hi;
            out[4 * i + 2] = (double)r.b_lo; out[4 * i + 3] = (double)r.b_hi;
        } else if (kind == 10 || kind == 11) {
            // the headline sweep's form of the accept test: argument in binary-log units (a = y = x·log2e), prefix as
            // the filter's pre-assembled addend bits; reference = the FP64 decision on x = RN(y·ln2)
            const uint64_t r = cc[i];
            const uint32_t magic = floor_magic_reg();
            const double xr = a[i] * 0x1.62e42fefa39efp-1;
            if (kind == 10) {
                const uint32_t fm = m64::exp_prefix_bits<11>((uint32_t)b[i], magic);
                auto exact_u = [&]() { return m64::u53_prefix_refine<11>(fm & 0x7ffu, (uint32_t)r, (uint32_t)(r >> 32)); };
                out[2 * i] = m64::exp_accept_prefix<11, true>(a[i], fm, exact_u, tb) ? 1.0 : 0.0;
                out[2 * i + 1] = m64::exp_accept_ref(xr, exact_u(), tb) ? 1.0 : 0.0;
            } else {
                const uint32_t fm = m64::exp_prefix_bits<12>((uint32_t)b[i], magic);
                auto exact_u = [&]() { return m64::u53_prefix_refine<12>(fm & 0xfffu, (uint32_t)r, (uint32_t)(r >> 32)); };
                out[2 * i] = m64::exp_accept_prefix<12, true>(a[i], fm, exact_u, tb) ? 1.0 : 0.0;
                out[2 * i + 1] = m64::exp_accept_ref(xr, exact_u(), tb) ? 1.0 : 0.0;
            }
        } else {
            const uint64_t r = cc[i];
            if (kind == 5) {
                const uint32_t f = (uint32_t)b[i] & 0x7ffu;
                auto exact_u = [&]() { return m64::u53_prefix_refine<11>(f, (uint32_t)r, (uint32_t)(r >> 32)); };
                out[2 * i] = m64::exp_accept_prefix<11>(a[i], f, exact_u, tb) ? 1.0 : 0.0;
                out[2 * i + 1] = m64::exp_accept_ref(a[i], exact_u(), tb) ? 1.0 : 0.0;
            } else {
                const uint32_t f = (uint32_t)b[i] & 0xfffu;
                auto exact_u = [&]() { return m64::u53_prefix_refine<12>(f, (uint32_t)r, (uint32_t)(r >> 32)); };
                out[2 * i] = m64::exp_accept_prefix<12>(a[i], f, exact_u, tb) ? 1.0 : 0.0;
                out[2 * i + 1] = m64::exp_accept_ref(a[i], exact_u(), tb) ? 1.0 : 0.0;
            }
        }
    }
}

// FP64 pipe peak: 8 independent DFMA chains per thread, no memory traffic.
__global__ void __launch_bounds__(kBlock) dfma_peak_kernel(double *out, int iters, double a, double b)
{
    double v0 = threadIdx.x, v1 = v0 + 1, v2 = v0 + 2, v3 = v0 + 3, v4 = v0 + 4, v5 = v0 + 5, v6 = v0 + 6, v7 = v0 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            v0 = fma(v0, a, b); v1 = fma(v1, a, b); v2 = fma(v2, a, b); v3 = fma(v3, a, b);
            v4 = fma(v4, a, b); v5 = fma(v5, a, b); v6 = fma(v6, a, b); v7 = fma(v7, a, b);
        }
    }
    out[(size_t)blockIdx.x * kBlock + threadIdx.x] = ((v0 + v1) + (v2 + v3)) + ((v4 + v5) + (v6 + v7));
}

}  // namespace arianna

#include "kernels_multi.cuh"
#include "kernels_replay.cuh"
#include "kernels_f32.cuh"
