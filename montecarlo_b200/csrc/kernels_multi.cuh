// kernels_multi.cuh -- K1m: the fused sweep for MULTI-MOVE pools (included at the end of kernels.cuh).
//
// mc_sweep! with Categorical(weights) (src/metropolis.jl:203-212), native Philox, with an optional series of store
// intervals whose records carry callback_acceptance as the reference defines it: one entry PER MOVE, the mean over
// chains of accepted_calls/total_calls (metropolis.jl:319-321).
//
//  * Move pick.  u_cat(t) = w·2^-32 with w the (t & 3)-th 32-bit word of block (t >> 2, sub 2): ONE extra Philox block
//    per FOUR steps (stream layout v4).  The reference's scan `cp = p[1]; while cp <= u && i < n: cp += p[i += 1]` [EXT
//    Distributions] has cp_j non-decreasing, so k = #{j < n-1 : cp_j <= u} = #{j : T_j <= w} with the integer thresholds
//    T_j = ceil(cp_j·2^32) (host, cp_j summed in binary64 exactly as the scan does).  A 4096-entry byte table indexed by
//    the top 12 bits of w answers directly (entry = k) unless the bucket contains thresholds: ONE threshold T_j (entry
//    0x80 | j) costs a compare, k = j + (w >= T_j); several (entry 0xFF: weights below 2^-12) take the full count.  One
//    shift + one LDS.U8 instead of a data-dependent chain of DADD/DSETP that diverged within the warp.
//  * Counters.  tot/acc of every (move, chain) live in shared memory as [move][tot|acc][thread] u32 and are bumped with
//    one shared-memory reduction each (ATOMS, no read-modify-write sequence); the two addresses differ by a constant.
//    With two buffers the counters of the thread's NEXT chain are fetched by cp.async (LDGSTS) while the current chain
//    runs its steps: at K = 10 the 16 n_moves bytes of counters per chain are the kernel's HBM traffic.
//  * Records.  At a store point every lane computes potential(x) and acc_k/tot_k (0/0 = NaN poisons the sum exactly
//    like the reference's mean), the warp reduces them with shuffles and lane 0 adds them to the warp's accumulator
//    row [store][1 + n_moves] in shared memory (fixed order: deterministic for a given grid); the CTA writes one
//    partial per store and series_fold_multi_kernel sums the partials.  Lanes past the end of the ensemble run as
//    zero-weight dummies so that the shuffles always see a full warp.
#pragma once

namespace arianna {

constexpr int kMultiMinBlocks = 4;  // resident CTAs per SM; the host sizes shared memory (buffers, intervals) to keep them
constexpr int kCatBuckets = 4096;   // top 12 bits of the 32-bit categorical word

struct MultiParams {
    double *x;
    uint32_t *acc;          // [n_moves][pitch]
    uint32_t *tot;          // [n_moves][pitch]
    const double *betas;
    double beta;
    int64_t M;              // chains of this launch (a slice of the handle's ensemble)
    int64_t pitch;          // row pitch of the counter arrays (chains of the whole handle)
    int64_t t0;             // MC steps already done by every chain
    uint64_t sid0;
    const m64::MathTables *tables;
    const uint8_t *cat_table;               // [kCatBuckets]: k | 0x80 + j (one threshold T_j inside) | 0xFF (several)
    uint32_t cat_thr[kMaxMoves];            // T_j = min(ceil(cp_j 2^32), 2^32 - 1), j < n_moves - 1
    int cat_n;                              // thresholds below 2^32 (the others can never be reached by a 32-bit word)
    PoolParams pool;
    const DevTheta *theta;          // non-null: σ (and the constants derived from it) live on the device
    int n_int;                      // intervals of this launch (>= 1)
    int record;                     // 1: a callback record after every interval
    int even;                       // every interval is a positive even number of steps starting on an even step
    int dbuf;                       // 1: two counter buffers in shared memory, the NEXT chain's counters are prefetched
    int K[kMaxSeries + 1];
    double *partials;               // [gridDim.x][n_int][1 + n_moves]
};

__device__ __forceinline__ void red_shared_add(uint32_t a, uint32_t v)
{
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
// global -> shared, 4 bytes, asynchronous (LDGSTS)
__device__ __forceinline__ void cp_async4(uint32_t dst, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// a / t for integer-valued 0 <= a <= t < 2^32 (t = 0: NaN, like 0/0): reciprocal seed + two Newton steps
__device__ __forceinline__ double ratio_fast(double a, double t)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(t));      // ~20 bits; rcp(0) = +inf
    double e = fma(-t, r, 1.0);
    r = fma(r, e, r);                                          // ~40 bits
    e = fma(-t, r, 1.0);
    r = fma(r, e, r);                                          // full precision (1 ulp)
    const double q = a * r;
    return fma(fma(-t, q, a), r, q);                           // one correction step on the quotient
}

// shared-memory footprint of one CTA of the kernel below
__host__ __device__ constexpr size_t multi_smem_bytes(int n_moves, int n_int, int record, int dbuf)
{
    return sizeof(m64::MathTables) + kCatBuckets + (8 + 8 + 8 + 4) * (size_t)kMaxMoves +
           (size_t)n_moves * 8 * kBlock * (dbuf ? 2 : 1) + (record ? (size_t)kWarpsPerBlock * n_int * (1 + n_moves) * 8 : 0);
}

template <int POT, int ARITH, bool BETAS>
__global__ void __launch_bounds__(kBlock, kMultiMinBlocks) sweep_multi_kernel(const MultiParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr uint32_t kTabBytes = (uint32_t)sizeof(m64::MathTables);
    constexpr uint32_t kOffCat = kTabBytes, kOffSigma = kOffCat + kCatBuckets, kOffLognorm = kOffSigma + 8 * kMaxMoves,
                       kOffInv = kOffLognorm + 8 * kMaxMoves, kOffThr = kOffInv + 8 * kMaxMoves, kOffCnt = kOffThr + 4 * kMaxMoves;
    const int nm = p.pool.n_moves, V = 1 + nm;
    const uint32_t cnt_bytes = 8u * kBlock * (uint32_t)nm;            // one counter buffer: [move][tot|acc][thread] u32
    const uint32_t off_rec = kOffCnt + cnt_bytes * (p.dbuf ? 2u : 1u);
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(p.cat_table);
        uint4 *dst = reinterpret_cast<uint4 *>(smem_raw + kOffCat);
        for (int i = threadIdx.x; i < kCatBuckets / 16; i += kBlock) dst[i] = src[i];
        if (threadIdx.x < kMaxMoves) {
            const int i = threadIdx.x;
            reinterpret_cast<double *>(smem_raw + kOffSigma)[i] = p.theta ? p.theta->sigma[i] : p.pool.sigma[i];
            reinterpret_cast<double *>(smem_raw + kOffLognorm)[i] = p.theta ? p.theta->lognorm[i] : p.pool.lognorm[i];
            reinterpret_cast<double *>(smem_raw + kOffInv)[i] = p.theta ? p.theta->inv2s2[i] : p.pool.inv2s2[i];
            reinterpret_cast<uint32_t *>(smem_raw + kOffThr)[threadIdx.x] = p.cat_thr[threadIdx.x];
        }
        if (p.record)
            for (int i = threadIdx.x; i < kWarpsPerBlock * p.n_int * V; i += kBlock)
                reinterpret_cast<double *>(smem_raw + off_rec)[i] = 0.0;
    }
    load_tables(reinterpret_cast<m64::MathTables *>(smem_raw), p.tables);
    __syncthreads();
    const m64::Tab tb = shared_tab(smem_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t a_cat = tb.s + kOffCat, a_sigma = tb.s + kOffSigma, a_lognorm = tb.s + kOffLognorm, a_inv = tb.s + kOffInv, a_thr = tb.s + kOffThr;
    const uint32_t a_rec = tb.s + off_rec + 8u * (uint32_t)(warp * p.n_int * V);
    const uint32_t buf_flip = p.dbuf ? cnt_bytes : 0u;
    const size_t pitch_b = (size_t)p.pitch * 4;
    const uint32_t magic = floor_magic_reg();
    const int64_t stride = (int64_t)gridDim.x * kBlock;
    uint32_t steps_launch = 0;                            // (hoisted by hand: the compiler re-summed K[] per chain)
    for (int i = 0; i < p.n_int; ++i) steps_launch += (uint32_t)p.K[i];
    const uint32_t pr_first = (uint32_t)p.t0 >> 1, pr_last = ((uint32_t)p.t0 + steps_launch) >> 1;

    // counters of chain cc -> the counter buffer at shared address `dst`, asynchronously; pointer stepping keeps the
    // 64-bit address arithmetic to one add per row (indexing [k * pitch + c] cost eight instructions per counter)
    auto fetch_counters = [&](uint32_t dst, int64_t cc) {
        if (cc < p.M) {
            const char *pt = reinterpret_cast<const char *>(p.tot + cc), *pa = reinterpret_cast<const char *>(p.acc + cc);
            for (int k = 0; k < nm; ++k, pt += pitch_b, pa += pitch_b, dst += 8u * kBlock) {
                cp_async4(dst, pt);
                cp_async4(dst + 4u * kBlock, pa);
            }
        }
        cp_async_commit();
    };

    int64_t c = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    uint32_t a_cnt = tb.s + kOffCnt + 4u * threadIdx.x;   // + move·8·kBlock: tot; + 4·kBlock more: acc
    const uint32_t a_both = 2u * a_cnt + buf_flip;        // the other buffer is at a_both - a_cnt
    double x_next = c < p.M ? p.x[c] : 0.0;
    if (p.dbuf) fetch_counters(a_cnt, c);
    // the loop condition is uniform across the warp (its first lane's chain); lanes past the end are dummies
    for (; c - lane < p.M; c += stride) {
        const bool live = c < p.M;
        double x = x_next;
        if (c + stride < p.M) x_next = p.x[c + stride];
        if (p.dbuf) {
            cp_async_wait_all();                          // this chain's counters have landed (own data only: no barrier)
            fetch_counters(a_both - a_cnt, c + stride);   // the next chain's, into the other buffer
        } else {
            fetch_counters(a_cnt, c);
            cp_async_wait_all();
        }
        double e = potential<POT, ARITH>(x);
        const double beta_nat = BETAS ? ((p.betas && live) ? p.betas[c] : p.beta) : p.beta;
        // FAST: the accept argument is formed in binary-log units (CellM, kernels.cuh), β·log2e·(e − e')
        const double beta = ARITH == ARITH_FAST ? beta_nat * 1.4426950408889634 : beta_nat;
        const uint64_t sid = p.sid0 + (uint64_t)c;
        const PhiloxChain<kTagMetropolis, 0> ph(sid);
        const PhiloxChain<kTagMetropolis, 2> ph_cat(sid);
        U64Pair cat{};                   // the four categorical words of quad cat_q
        uint32_t cat_q = 0xffffffffu;    // (t < 2^32, so no quad has this index)

        // move index of the categorical word w
        auto pick = [&](uint32_t w) -> uint32_t {
            uint32_t k = lds_u8(a_cat + (w >> 20));
            if (k & 0x80u) {             // the bucket holds thresholds
                if (k != 0xffu) {        // exactly one, T_j: j moves lie below the bucket
                    const uint32_t j = k & 0x7fu;
                    k = j + (w >= lds_u32(a_thr + 4u * j) ? 1u : 0u);
                } else {                 // several: count the reachable thresholds at or below w
                    k = 0;
                    for (int j = 0; j < p.cat_n; ++j) k += (w >= lds_u32(a_thr + 4u * j)) ? 1u : 0u;
                }
            }
            return k;
        };
        auto one_step = [&](uint32_t w, double z, auto cell, auto exact_u) {
            const uint32_t k = pick(w);
            const double sigma = lds_f64(a_sigma + 8u * k);
            const double lognorm = ARITH == ARITH_EXACT ? lds_f64(a_lognorm + 8u * k) : 0.0;
            const double inv = ARITH == ARITH_EXACT ? lds_f64(a_inv + 8u * k) : 0.0;
            const uint32_t a = mc_step<POT, ARITH>(x, e, beta, sigma, lognorm, inv, z, cell, exact_u, tb) ? 1u : 0u;
            const uint32_t ak = a_cnt + 8u * kBlock * k;
            red_shared_add(ak, 1u);                      // total_calls += 1          (metropolis.jl:209)
            red_shared_add(ak + 4u * kBlock, a);         // accepted_calls += mc_step! (:208)
        };
        // the two steps of pair pr (DO0 / DO1 compile-time)
        auto do_pair = [&](uint32_t pr, auto do0, auto do1) {
            const U64Pair b0 = ph.block(pr);
            double z0, z1;
            m64::box_muller_u64(u64_of(b0.a_lo, b0.a_hi), u64_of(b0.b_lo, b0.b_hi), tb, z0, z1);
            if ((pr >> 1) != cat_q) {    // uniform across the warp: every chain is at the same step
                cat_q = pr >> 1;
                cat = ph_cat.block(cat_q);
            }
            const bool hi = (pr & 1u) != 0;              // steps 4q+2, 4q+3 take the B words
            if constexpr (decltype(do0)::value) {
                const uint32_t f0 = m64::exp_prefix_bits<12>(b0.a_lo, magic);     // prefix | the filter's magic bits
                auto exact_u = [&]() {
                    const U64Pair r = philox_block<kTagMetropolis>(sid, (uint64_t)pr, 1);
                    return m64::u53_prefix_refine<12>(f0 & 0xfffu, r.a_lo, r.a_hi);
                };
                one_step(hi ? cat.b_lo : cat.a_lo, z0, CellM<12>{f0}, exact_u);
            }
            if constexpr (decltype(do1)::value) {
                const uint32_t f1 = m64::exp_prefix_bits<11>(b0.b_lo, magic);
                auto exact_u = [&]() {
                    const U64Pair r = philox_block<kTagMetropolis>(sid, (uint64_t)pr, 1);
                    return m64::u53_prefix_refine<11>(f1 & 0x7ffu, r.b_lo, r.b_hi);
                };
                one_step(hi ? cat.b_hi : cat.a_hi, z1, CellM<11>{f1}, exact_u);
            }
        };
        using T_ = std::true_type;
        using F_ = std::false_type;
        auto run_steps = [&](uint32_t ta, uint32_t te) {       // MC steps [ta, te)
            if (te <= ta) return;
            uint32_t pr = ta >> 1;
            if (ta & 1u) { do_pair(pr, F_{}, T_{}); ++pr; }
            const uint32_t pr_end = te >> 1;
#pragma unroll 1
            for (; pr < pr_end; ++pr) do_pair(pr, T_{}, T_{});
            if (te & 1u) do_pair(pr, T_{}, F_{});
        };
        // the callback record of store s: Σe and Σ_c acc_ck/tot_ck for every move, reduced over the warp
        // (acc/tot through a Newton-refined reciprocal: MUFU.RCP64H + 4 DFMA + 1 DMUL instead of the ~25 instructions
        // of an IEEE division with its slow-path check; relative error < 2^-51, the records are compared at 1e-12)
        auto store_point = [&](int s) {
            const uint32_t row = a_rec + 8u * (uint32_t)(s * V);
            double v = warp_sum(live ? potential<POT, ARITH>(x) : 0.0);
            if (lane == 0) sts_f64(row, lds_f64(row) + v);
            for (int k = 0; k < nm; ++k) {
                const double a = (double)lds_u32(a_cnt + 8u * kBlock * k + 4u * kBlock);
                const double t = (double)lds_u32(a_cnt + 8u * kBlock * k);
                v = warp_sum(live ? ratio_fast(a, t) : 0.0);     // 0/0 = NaN while a chain never tried move k
                if (lane == 0) sts_f64(row + 8u * (1 + k), lds_f64(row + 8u * (1 + k)) + v);
            }
        };

        uint32_t ta = (uint32_t)p.t0;
        if (p.even) {
            // whole pairs only: ONE flat loop over the pairs of all intervals, a countdown marks the store points
            int s = 0;
            int left = p.K[0] >> 1;
#pragma unroll 1
            for (uint32_t pr = pr_first; pr < pr_last; ++pr) {
                do_pair(pr, T_{}, T_{});
                if (--left == 0) {
                    if (p.record) store_point(s);
                    left = p.K[++s] >> 1;
                }
            }
        } else {
#pragma unroll 1
            for (int s = 0; s < p.n_int; ++s) {
                const uint32_t te = ta + (uint32_t)p.K[s];
                run_steps(ta, te);
                if (p.record) store_point(s);
                ta = te;
            }
        }

        if (live) {
            p.x[c] = x;
            char *pt = reinterpret_cast<char *>(p.tot + c), *pa = reinterpret_cast<char *>(p.acc + c);
            uint32_t src = a_cnt;
            for (int k = 0; k < nm; ++k, pt += pitch_b, pa += pitch_b, src += 8u * kBlock) {
                *reinterpret_cast<uint32_t *>(pt) = lds_u32(src);
                *reinterpret_cast<uint32_t *>(pa) = lds_u32(src + 4u * kBlock);
            }
        }
        a_cnt = a_both - a_cnt;
    }
    cp_async_wait_all();
    if (p.record) {
        __syncthreads();
        const double *rec = reinterpret_cast<const double *>(smem_raw + off_rec);
        const int n = p.n_int * V;
        for (int i = threadIdx.x; i < n; i += kBlock) {
            double t = 0.0;
#pragma unroll
            for (int w = 0; w < kWarpsPerBlock; ++w) t += rec[w * n + i];
            p.partials[(size_t)blockIdx.x * n + i] = t;
        }
    }
}

// Fold of the multi-move records: CTA s sums the per-CTA partials of store s in a fixed order,
//   out[s] = [Σ_c e_c(t_s), Σ_c acc_ck/tot_ck (k < n_moves), M]
__global__ void __launch_bounds__(kBlock) series_fold_multi_kernel(const double *partials, int n_ctas, int n_int,
                                                                   int n_moves, int64_t M, double *out, double *sums,
                                                                   int accumulate)
{
    __shared__ double s_w[kWarpsPerBlock];
    const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, V = 1 + n_moves, stride = 2 + n_moves;
    for (int v = 0; v < V; ++v) {
        double t = 0.0;
        for (int b = threadIdx.x; b < n_ctas; b += kBlock) t += partials[((size_t)b * n_int + s) * V + v];
        t = warp_sum(t);
        __syncthreads();
        if (lane == 0) s_w[warp] = t;
        __syncthreads();
        if (threadIdx.x == 0) {
            double r = 0.0;
#pragma unroll
            for (int w = 0; w < kWarpsPerBlock; ++w) r += s_w[w];
            if (accumulate) r += out[(size_t)stride * s + v];
            out[(size_t)stride * s + v] = r;
            if (s == n_int - 1 && sums) sums[v] = r;
        }
    }
    if (threadIdx.x == 0) {
        double r = (double)M;
        if (accumulate) r += out[(size_t)stride * s + V];
        out[(size_t)stride * s + V] = r;
        if (s == n_int - 1 && sums) sums[V] = r;
    }
}

}  // namespace arianna
