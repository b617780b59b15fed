// kernels_histogram.cuh -- on-device histograms and moments of x or e, per ensemble and per group (sm_100a).
//
// Global chain g = chain_offset + c belongs to group g % G.  Each accumulate adds one sample of every local chain:
//   v = x or potential(x)      (F64: EXACT binary64; F32: Float64(x) or Float64(potential_f32(x)), the widened get_state_f32)
//   t = RN(RN(v − lo) · inv_w) (__dsub_rn, __dmul_rn: never contracted), inv_w = RN(n_bins / (hi − lo)) from the host
//   cell = nan if t is NaN, underflow if t < 0, overflow if t >= n_bins, else floor(t)
// into the int64 counts [G][n_bins + 3] = [n_bins regular][underflow][overflow][nan] and the binary64 moments
// [G][3] = (n, Σv, Σv²) over the finite v.  t < 0 <=> floor(t) < 0 and t >= n_bins <=> floor(t) >= n_bins (n_bins is an
// integer), so the comparisons are the bin rule itself; ±inf reach under- or overflow through them.  DESIGN.md §4 "K9".
#pragma once
#include "kernels.cuh"   // (and kernels_f32.cuh: potential_f32)

namespace arianna {

constexpr int kHistMaxCells = 16384;      // G·(n_bins + 3) u32 cells: 64 KB of shared memory per CTA
constexpr int kHistBlock = 512;
constexpr int kHistMinBlocks = 2;         // 64 registers: no spills with kHistUnroll loads in flight (40 at 3 blocks spill)
constexpr int kHistUnroll = 8;            // loads in flight per thread: 64 B (F64) / 32 B (F32)
constexpr int kHistPosition = -1;         // SRC of histogram_kernel: the position; 0..2: the energy of that potential

struct HistogramParams {
    const void *x;                        // double[M] (F64 handles) or float[M] (F32 handles)
    int64_t M;
    int g0;                               // chain_offset % G: the group of local chain 0
    int G;
    int n_bins;
    double lo, inv_w;
    unsigned long long *counts;           // [G][n_bins + 3], accumulated over calls
    double *partials;                     // [gridDim.x][G][3] (n, Σv, Σv²) of this call
};

template <typename T, int SRC>
__device__ __forceinline__ double hist_value(T x)
{
    if constexpr (SRC == kHistPosition) {
        return (double)x;
    } else if constexpr (sizeof(T) == 8) {
        return potential<SRC, ARITH_EXACT>(x);
    } else {
        return (double)potential_f32<SRC>(x);
    }
}

// Grid-stride over the chains with a stride that is a multiple of G: every thread stays in ONE group, so its moments
// are three registers and its cells one row of the per-CTA histogram, while a warp still reads 32 consecutive chains.
// Contention: a thread counts runs of equal cells among its own chains in two registers (the cell, the run length) and
// adds a run to the shared u32 cell only when the cell changes, and once at the end.  A narrow distribution (every chain
// in one bin after set_state(zeros)) then costs one shared atomic per thread and call, for any G, and a distribution
// over a few bins one atomic per change; a broad one one atomic per chain, as without runs.  There are no warp
// collectives: lanes never wait for each other.  At the end the CTA flushes its non-zero cells with 64-bit global
// atomics (integer addition: the counts are exact and do not depend on the order), starting at a CTA-dependent
// cell so that CTAs finishing together do not queue on the same addresses, and writes its moment partials, summed in a
// fixed order (a tree over the threads of each group).
template <typename T, int SRC>
__global__ void __launch_bounds__(kHistBlock, kHistMinBlocks) histogram_kernel(const HistogramParams p)
{
    extern __shared__ unsigned int s_hist[];          // [G][n_bins + 3]
    __shared__ double s_v[kHistBlock];
    const int cells = p.n_bins + 3;
    const int n_cells = p.G * cells;
    for (int i = threadIdx.x; i < n_cells; i += kHistBlock) s_hist[i] = 0u;
    __syncthreads();

    const T *__restrict__ x = static_cast<const T *>(p.x);
    const int64_t T_all = (int64_t)gridDim.x * kHistBlock;
    const int64_t stride = T_all / p.G * p.G;        // >= G: the host launches at least kHistBlock >= kMaxLadder threads
    const int64_t tid = (int64_t)blockIdx.x * kHistBlock + threadIdx.x;
    const bool live = tid < stride;
    const int grp = (int)((p.g0 + tid) % p.G);
    const int row = grp * cells;                     // this thread's row of the shared histogram
    const double nb = (double)p.n_bins;
    unsigned int n = 0;
    double s1 = 0.0, s2 = 0.0;
    int run = -1;                                    // the current run of equal cells: its cell and its length
    unsigned int run_n = 0;

    auto bin = [&](double v) {
        const double t = __dmul_rn(__dsub_rn(v, p.lo), p.inv_w);
        return t != t ? p.n_bins + 2 : (t < 0.0 ? p.n_bins : (t >= nb ? p.n_bins + 1 : (int)t));
    };
    auto add = [&](double v) {
        const int cell = row + bin(v);
        if (cell != run) {
            if (run_n) atomicAdd(&s_hist[run], run_n);
            run = cell;
            run_n = 0;
        }
        ++run_n;
        if (isfinite(v)) {
            ++n;
            s1 = __dadd_rn(s1, v);
            s2 = __dadd_rn(s2, __dmul_rn(v, v));
        }
    };

    if (live) {
        int64_t c = tid;
        for (; c + (int64_t)(kHistUnroll - 1) * stride < p.M; c += kHistUnroll * stride) {
            T v[kHistUnroll];
#pragma unroll
            for (int u = 0; u < kHistUnroll; ++u) v[u] = x[c + u * stride];
#pragma unroll
            for (int u = 0; u < kHistUnroll; ++u) add(hist_value<T, SRC>(v[u]));
        }
        for (; c < p.M; c += stride) add(hist_value<T, SRC>(x[c]));
        if (run_n) atomicAdd(&s_hist[run], run_n);
    }
    __syncthreads();

    // flush: every thread owns distinct cells; start at a CTA-dependent cell (spreads the same-address atomics)
    const int rot = (int)(((int64_t)blockIdx.x * 997) % n_cells);
    for (int i = threadIdx.x; i < n_cells; i += kHistBlock) {
        int j = i + rot;
        if (j >= n_cells) j -= n_cells;
        const unsigned int cnt = s_hist[j];
        if (cnt) atomicAdd(p.counts + j, (unsigned long long)cnt);
    }

    // moment partials: thread t's group is (base + t) % G, base = (g0 + blockIdx.x·kHistBlock) % G; the threads of one
    // group are t0 + j·G (t0 = t % G, j = t / G), reduced by a tree over j, so s_v[t0] ends with the group's sum
    const int base = (int)((p.g0 + (int64_t)blockIdx.x * kHistBlock) % p.G);
    double *out = p.partials + (size_t)blockIdx.x * p.G * 3;
    const int j = threadIdx.x / p.G;
    for (int q = 0; q < 3; ++q) {
        s_v[threadIdx.x] = !live ? 0.0 : (q == 0 ? (double)n : (q == 1 ? s1 : s2));
        for (int s = 1; s * p.G < kHistBlock; s *= 2) {
            __syncthreads();
            if ((j & (2 * s - 1)) == 0 && threadIdx.x + s * p.G < kHistBlock) s_v[threadIdx.x] += s_v[threadIdx.x + s * p.G];
        }
        __syncthreads();
        if (threadIdx.x < p.G) out[(size_t)((base + threadIdx.x) % p.G) * 3 + q] = s_v[threadIdx.x];
        __syncthreads();
    }
}

// Fold: CTA g adds the per-CTA partials of group g, in a fixed order, to the accumulated moments (n, Σv, Σv²).
__global__ void __launch_bounds__(kBlock) histogram_fold_kernel(const double *partials, int n_ctas, int G, double *moments)
{
    __shared__ double s_w[kWarpsPerBlock];
    const int g = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int q = 0; q < 3; ++q) {
        double v = 0.0;
        for (int b = threadIdx.x; b < n_ctas; b += kBlock) v += partials[((size_t)b * G + g) * 3 + q];
        v = warp_sum(v);
        __syncthreads();
        if (lane == 0) s_w[warp] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
#pragma unroll
            for (int k = 0; k < kWarpsPerBlock; ++k) t += s_w[k];
            moments[(size_t)g * 3 + q] += t;
        }
    }
}

}  // namespace arianna
