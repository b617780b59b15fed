// rng.cuh -- in-register generators of the sweep kernels (sm_100a).
//
//  * Philox4x32-10 (Salmon et al., SC'11) counter-based generator: zero bytes of RNG state in HBM, the stream of
//    chain c is a pure function of (seed + global chain index, draw index), so results are invariant to the
//    launch chunking (K) and to the multi-GPU sharding.  Stream layout: DESIGN.md "RNG stream layout".
//  * xoshiro256++ + 256-layer ziggurat: the generator FAMILY of the reference (Random.Xoshiro, randn [EXT]);
//    32 B of state per chain in HBM, uploaded by the host (arianna_set_rng_state).
#pragma once
#include <cstdint>

namespace arianna {

constexpr uint32_t kPhiloxM0 = 0xD2511F53u;
constexpr uint32_t kPhiloxM1 = 0xCD9E8D57u;
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u;
constexpr uint32_t kPhiloxW1 = 0xBB67AE85u;
constexpr uint32_t kKey1 = 0x41524941u;  // 'ARIA'

enum : uint32_t { kTagInit = 0, kTagMetropolis = 1, kTagEstimator = 2, kTagExchange = 4 };

struct U64Pair {
    uint32_t a_lo, a_hi, b_lo, b_hi;  // A = out[0] | out[1] << 32,  B = out[2] | out[3] << 32
};

// One Philox4x32-10 round on (c0, c1, c2, c3) with round keys (k0, k1).
__device__ __forceinline__ void philox_round(uint32_t &c0, uint32_t &c1, uint32_t &c2, uint32_t &c3, uint32_t k0,
                                             uint32_t k1)
{
    const uint32_t hi0 = __umulhi(kPhiloxM0, c0), lo0 = kPhiloxM0 * c0;
    const uint32_t hi1 = __umulhi(kPhiloxM1, c2), lo1 = kPhiloxM1 * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
}

// Counter layout (v2, identical in oracle/arianna_oracle.c:philox_block):
//   ctr = (sid_lo, p_lo, sid_hi, sub | (p_hi << 8)),  key = (TAG, 'ARIA')
// sid = seed + global chain index, p = block index of the stream (Metropolis: step pair t >> 1; estimator: sample
// pair q >> 1), sub = which block of the pair (0 main, 1 accept-uniform refinement, 2 categorical uniforms).
// The VARYING word p sits in c1, a word that the first round only XORs: with (c0, c2, c3) fixed per chain, one of
// the two 32x32->64 multiplies of each of the first three rounds depends on the chain alone (PhiloxChain below).

// One Philox4x32-10 block, general form.  TAG is a compile-time constant so the ten round keys fold into immediates.
template <uint32_t TAG>
__device__ __forceinline__ U64Pair philox_block(uint64_t sid, uint64_t p, uint32_t sub)
{
    uint32_t c0 = (uint32_t)sid, c1 = (uint32_t)p, c2 = (uint32_t)(sid >> 32), c3 = sub | ((uint32_t)(p >> 32) << 8);
#pragma unroll
    for (int r = 0; r < 10; ++r) philox_round(c0, c1, c2, c3, TAG + (uint32_t)r * kPhiloxW0, kKey1 + (uint32_t)r * kPhiloxW1);
    return U64Pair{c0, c1, c2, c3};
}

// The same function for ONE chain and a fixed sub-block, p < 2^32: the chain-only halves of rounds 0-2 are computed
// once per chain (4 wide multiplies) and every block then costs 16 wide multiplies instead of 20.  On B200 an
// IMAD.WIDE holds the issue port for ~4.5 cycles (profiles/microbench), so these are the most expensive instructions
// of the sweep.  Bit-identical to philox_block<TAG>(sid, p, SUB) (tests/test_gpu_math.py::test_device_philox_kat).
template <uint32_t TAG, uint32_t SUB>
struct PhiloxChain {
    uint32_t X, L0, B2, Q, ql;
    __device__ __forceinline__ explicit PhiloxChain(uint64_t sid)
    {
        constexpr uint32_t k00 = TAG, k10 = kKey1, k01 = TAG + kPhiloxW0, k11 = kKey1 + kPhiloxW1,
                           k02 = TAG + 2u * kPhiloxW0, k12 = kKey1 + 2u * kPhiloxW1;
        const uint32_t s0 = (uint32_t)sid, s1 = (uint32_t)(sid >> 32);
        const uint32_t h0 = __umulhi(kPhiloxM0, s0), l0 = kPhiloxM0 * s0;     // round 0, chain-only
        const uint32_t h1 = __umulhi(kPhiloxM1, s1), l1 = kPhiloxM1 * s1;
        X = h1 ^ k00;                                                         // c0 after round 0 = X ^ p
        const uint32_t C2 = h0 ^ SUB ^ k10;                                   // c2 after round 0
        const uint32_t gh = __umulhi(kPhiloxM1, C2), gl = kPhiloxM1 * C2;     // round 1, chain-only half
        const uint32_t A = gh ^ l1 ^ k01;                                     // c0 after round 1
        L0 = l0 ^ k11;                                                        // c2 after round 1 = hi(M0 c0) ^ L0
        const uint32_t qh = __umulhi(kPhiloxM0, A);                           // round 2, chain-only half
        ql = kPhiloxM0 * A;                                                   // c3 after round 2
        B2 = gl ^ k02;                                                        // c0 after round 2 = hi(M1 c2) ^ B2
        Q = qh ^ k12;                                                         // c2 after round 2 = Q ^ lo(M0 c0 of round 1)
    }
    __device__ __forceinline__ U64Pair block(uint32_t p) const
    {
        const uint32_t a = X ^ p;                                                   // round 0
        const uint32_t ah = __umulhi(kPhiloxM0, a), al = kPhiloxM0 * a;             // round 1
        const uint32_t b = ah ^ L0;
        const uint32_t bh = __umulhi(kPhiloxM1, b), bl = kPhiloxM1 * b;             // round 2
        uint32_t c0 = bh ^ B2, c1 = bl, c2 = Q ^ al, c3 = ql;
#pragma unroll
        for (int r = 3; r < 10; ++r) philox_round(c0, c1, c2, c3, TAG + (uint32_t)r * kPhiloxW0, kKey1 + (uint32_t)r * kPhiloxW1);
        return U64Pair{c0, c1, c2, c3};
    }
};

// u53(w) = (w >> 11) * 2^-53 in [0,1), EXACTLY, without an int->fp64 conversion instruction:
//   k = w >> 11 = k_hi * 2^32 + k_lo  (k_hi: 21 bits)
//   dh = 2^31 + k_hi * 2^-21   (exponent 0x41E, mantissa low word = k_hi)
//   dl = 2^-1 + k_lo * 2^-53   (exponent 0x3FE, mantissa low word = k_lo)
//   (dh - (2^31 + 2^-1)) + dl  -- both additions are exact.
__device__ __forceinline__ double u53_from_k(uint32_t k_hi, uint32_t k_lo)
{
    double dh = __hiloint2double(0x41E00000, (int)k_hi);
    double dl = __hiloint2double(0x3FE00000, (int)k_lo);
    return __dadd_rn(__dadd_rn(dh, -2147483648.5), dl);
}

__device__ __forceinline__ double u53(uint32_t lo, uint32_t hi)
{
    return u53_from_k(hi >> 11, (hi << 21) | (lo >> 11));
}

// ((w >> 11) | 1) * 2^-53 in (0,1): the Box-Muller radius uniform on the odd lattice (log never sees 0 or 1).
__device__ __forceinline__ double u53_open0(uint32_t lo, uint32_t hi)
{
    return u53_from_k(hi >> 11, ((hi << 21) | (lo >> 11)) | 1u);
}

// ---------------------------------------------------------------------------------------------------------
// xoshiro256++ (Blackman & Vigna).  State (1,2,3,4) -> first output 41943041.
// ---------------------------------------------------------------------------------------------------------
struct Xoshiro {
    uint64_t s0, s1, s2, s3;
    __device__ __forceinline__ uint64_t next()
    {
        uint64_t sum = s0 + s3;
        uint64_t r = ((sum << 23) | (sum >> 41)) + s0;
        uint64_t t = s1 << 17;
        s2 ^= s0;
        s3 ^= s1;
        s1 ^= s2;
        s0 ^= s3;
        s2 ^= t;
        s3 = (s3 << 45) | (s3 >> 19);
        return r;
    }
    // rand(rng, Float64) [EXT]: (next >> 11) * 2^-53
    __device__ __forceinline__ double rand()
    {
        uint64_t w = next();
        return u53((uint32_t)w, (uint32_t)(w >> 32));
    }
};

struct ZigTables {
    const uint64_t *ki;  // [256]
    const double *wi;    // [256]
    const double *fi;    // [256]
};

constexpr double kZigR = 3.6541528853610088;
constexpr double kZigInvR = 0.27366123732975828;

// randn(rng) [EXT]: 256-layer ziggurat on 52 random bits; tables live in shared memory.
__device__ __forceinline__ double xoshiro_randn(Xoshiro &g, const ZigTables &T)
{
    for (;;) {
        uint64_t r = g.next() >> 12;
        int64_t rabs = (int64_t)(r >> 1);
        int idx = (int)(rabs & 0xFF);
        double x = __dmul_rn((double)((r & 1) ? -rabs : rabs), T.wi[idx]);
        if ((uint64_t)rabs < T.ki[idx]) return x;
        if (idx == 0) {
            for (;;) {
                double xx = __dmul_rn(-kZigInvR, log(g.rand()));
                double yy = -log(g.rand());
                if (__dadd_rn(yy, yy) > __dmul_rn(xx, xx))
                    return ((rabs >> 8) & 1) ? __dsub_rn(-kZigR, xx) : __dadd_rn(kZigR, xx);
            }
        } else {
            double lhs = __dadd_rn(__dmul_rn(__dsub_rn(T.fi[idx - 1], T.fi[idx]), g.rand()), T.fi[idx]);
            if (lhs < exp(__dmul_rn(__dmul_rn(-0.5, x), x))) return x;
        }
    }
}

}  // namespace arianna
