// kernels_exchange.cuh -- replica exchange (parallel tempering) across per-chain β ladders (sm_100a).
//
// A ladder is L consecutive chains by global index; global chain g is rung g % L of ladder g / L (the host only accepts
// shards that start and end on a ladder boundary, so local index % L is the rung too).  Round R pairs the rungs
// (r, r + 1) with r ≡ R (mod 2) in every ladder (deterministic even/odd scheme) and swaps the two positions iff
//   min(1, exp(Δ)) > u,   Δ = (β_g − β_{g+1})·(e_g − e_{g+1}),   e = potential<POT, EXACT>(x)
// with u = u53 of the first word of philox_block<kTagExchange>(seed + g, R, 0) for the lower chain g.  Only x moves:
// β, the Move counters and the chain's Metropolis stream stay with the slot (the temperature).  DESIGN.md §4 "Replica exchange".
#pragma once
#include "kernels.cuh"

namespace arianna {

constexpr int kMaxLadder = 256;

// per-chain β = ladder[g % L] (arianna_set_ladder; the shard starts on a ladder boundary)
__global__ void __launch_bounds__(kBlock) ladder_betas_kernel(double *betas, const double *ladder, int L, int64_t M)
{
    for (int64_t c = (int64_t)blockIdx.x * kBlock + threadIdx.x; c < M; c += (int64_t)gridDim.x * kBlock)
        betas[c] = ladder[c % L];
}

struct ExchangeParams {
    double *__restrict__ x;
    const double *__restrict__ betas;   // nullptr -> every chain has `beta` (Δ = 0: every active pair swaps)
    double beta;
    int64_t n_ladders;                  // local ladders
    int L;
    int pairs;                          // active pairs per ladder this round: (L − (R & 1)) / 2
    int64_t R;                          // round index (the Philox counter)
    uint64_t sid0;                      // seed + chain_offset
    const m64::MathTables *tables;
    unsigned long long *accepted;       // [L − 1] swaps per rung pair, accumulated over rounds
};

// One thread per active pair, grid-stride with a stride that is a multiple of `pairs`: every thread keeps the SAME pair
// slot j (rung r = (R & 1) + 2j) in all its iterations, so its accepted count is one register.  Counts are combined per
// rung pair by a warp reduction over the lanes that share j, then in shared memory, then one integer atomic per CTA and
// pair (order-independent: the counters are deterministic).  HBM traffic per round: x and β of every chain (16 B) and x
// of the swapped chains (8 B each); the Philox block costs ~20 wide multiplies per pair and hides under the loads.
template <int POT>
__global__ void __launch_bounds__(kBlock) exchange_kernel(const ExchangeParams p)
{
    __shared__ unsigned int s_cnt[kMaxLadder];
    __shared__ double s_exp2[m64::kExpTab];          // the only table exp_core reads (2^(j/32))
    for (int i = threadIdx.x; i < kMaxLadder; i += kBlock) s_cnt[i] = 0u;
    for (int i = threadIdx.x; i < m64::kExpTab; i += kBlock) s_exp2[i] = p.tables->exp2_j[i];
    __syncthreads();
    // m64::Tab addresses the whole MathTables layout: point it so that exp2_j lands on s_exp2
    const m64::Tab tb = shared_tab(reinterpret_cast<const char *>(s_exp2) - m64::kOffExp2);

    const int64_t n_pairs = p.n_ladders * p.pairs;
    const int64_t T = (int64_t)gridDim.x * kBlock;
    const int64_t stride = T / p.pairs * p.pairs;    // >= pairs: the host launches at least `pairs` threads
    const int64_t tid = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    const int j = (int)(tid % p.pairs);
    const int r = (int)(p.R & 1) + 2 * j;
    unsigned int cnt = 0;
    if (tid < stride) {
        for (int64_t i = tid; i < n_pairs; i += stride) {
            const int64_t g = (i / p.pairs) * p.L + r;   // local index of the lower chain
            const double x0 = p.x[g], x1 = p.x[g + 1];
            const double b0 = p.betas ? p.betas[g] : p.beta, b1 = p.betas ? p.betas[g + 1] : p.beta;
            const double e0 = potential<POT, ARITH_EXACT>(x0), e1 = potential<POT, ARITH_EXACT>(x1);
            const double delta = __dmul_rn(__dsub_rn(b0, b1), __dsub_rn(e0, e1));
            const U64Pair w = philox_block<kTagExchange>(p.sid0 + (uint64_t)g, (uint64_t)p.R, 0);
            const double u = u53(w.a_lo, w.a_hi);
            float ulo, uhi;
            m64::ucell_from_double(u, ulo, uhi);
            // min(1, exp(Δ)) > u, strict, NaN rejects (metropolis.jl:183-185 semantics), decided as the FP64 exp would
            if (m64::exp_accept(delta, ulo, uhi, [&]() { return u; }, tb)) {
                p.x[g] = x1;
                p.x[g + 1] = x0;
                ++cnt;
            }
        }
    }
    // lanes holding the same pair slot: one warp sum, then the group leader adds it to the CTA's slot
    const unsigned grp = __match_any_sync(0xffffffffu, tid < stride ? r : -1);
    const unsigned sum = __reduce_add_sync(grp, cnt);
    if (tid < stride && sum && (threadIdx.x & 31) == __ffs(grp) - 1) atomicAdd(&s_cnt[r], sum);
    __syncthreads();
    for (int k = threadIdx.x; k < p.L - 1; k += kBlock)
        if (s_cnt[k]) atomicAdd(p.accepted + k, (unsigned long long)s_cnt[k]);
}

// Per-rung callback sums: partials[cta][L][1 + n_moves] = (Σ e, Σ_c acc_ck / tot_ck per move) over the chains of each
// rung that this CTA visited.  The grid-stride step is a multiple of L, so every thread stays on ONE rung (tid % L) and a
// warp still reads 32 consecutive chains of every array (coalesced for any L).  The CTA's threads of one rung are then
// summed in thread order through shared memory: the reduction order is a function of (grid, L) only.
struct LadderReduceParams {
    const double *x;
    const uint32_t *acc;
    const uint32_t *tot;   // nullptr -> steps_done
    int64_t M;             // local chains (multiple of L)
    int64_t pitch;         // row pitch of the [n_moves][pitch] counter arrays
    int64_t steps_done;
    int n_moves;
    int potential;
    int L;
    double *partials;      // [gridDim.x][L][1 + n_moves]
};

// NM = the largest pool the instantiation serves (1: single-move pools keep 2 accumulators instead of 17)
// (__maxnreg__: left to itself ptxas caps the 17-accumulator instantiation at 64 registers and spills)
template <int NM>
__global__ void __maxnreg__(NM == 1 ? 64 : 96) ladder_reduce_kernel(const LadderReduceParams p)
{
    __shared__ double s_v[kBlock];
    double vals[1 + NM];
#pragma unroll
    for (int i = 0; i <= NM; ++i) vals[i] = 0.0;
    const int64_t T = (int64_t)gridDim.x * kBlock;
    const int64_t stride = T / p.L * p.L;
    const int64_t tid = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (tid < stride) {
        for (int64_t c = tid; c < p.M; c += stride) {
            const double x = p.x[c];
            double e;
            if (p.potential == POT_HARMONIC) e = potential<POT_HARMONIC, ARITH_EXACT>(x);
            else if (p.potential == POT_QUARTIC) e = potential<POT_QUARTIC, ARITH_EXACT>(x);
            else e = potential<POT_DOUBLE_WELL, ARITH_EXACT>(x);
            vals[0] += e;
#pragma unroll
            for (int k = 0; k < NM; ++k) {
                if (k < p.n_moves) {
                    const double a = (double)p.acc[(size_t)k * p.pitch + c];
                    const double t = p.tot ? (double)p.tot[(size_t)k * p.pitch + c] : (double)p.steps_done;
                    vals[1 + k] += a / t;
                }
            }
        }
    }
    // thread t of this CTA is on rung (cta_base + t) % L; rung r's first thread is t0 = (r − cta_base) mod L
    const int base = (int)(((int64_t)blockIdx.x * kBlock) % p.L);
    double *out = p.partials + (size_t)blockIdx.x * p.L * (1 + p.n_moves);
#pragma unroll
    for (int q = 0; q <= NM; ++q) {
        if (q <= p.n_moves) {
            __syncthreads();
            s_v[threadIdx.x] = tid < stride ? vals[q] : 0.0;
            __syncthreads();
            for (int r = threadIdx.x; r < p.L; r += kBlock) {
                double s = 0.0;
                for (int t = (r - base + p.L) % p.L; t < kBlock; t += p.L) s += s_v[t];
                out[(size_t)r * (1 + p.n_moves) + q] = s;
            }
        }
    }
}

// Fold: CTA r sums the per-CTA partials of rung r in a fixed order and writes the record
// out[r] = (Σ e, Σ acc/tot per move, chain count of the rung).
__global__ void __launch_bounds__(kBlock) ladder_fold_kernel(const double *partials, int n_ctas, int L, int n_moves,
                                                             double count, double *out)
{
    __shared__ double s_w[kWarpsPerBlock];
    const int r = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int w = 1 + n_moves;
    for (int q = 0; q < w; ++q) {
        double v = 0.0;
        for (int b = threadIdx.x; b < n_ctas; b += kBlock) v += partials[((size_t)b * L + r) * w + q];
        v = warp_sum(v);
        __syncthreads();
        if (lane == 0) s_w[warp] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
#pragma unroll
            for (int k = 0; k < kWarpsPerBlock; ++k) t += s_w[k];
            out[(size_t)r * (2 + n_moves) + q] = t;
        }
    }
    if (threadIdx.x == 0) out[(size_t)r * (2 + n_moves) + 1 + n_moves] = count;
}

}  // namespace arianna
