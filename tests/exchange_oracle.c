/*
 * exchange_oracle.c -- CPU reference of the engine's replica exchange (arianna_replica_exchange, arianna_ladder_sums;
 * DESIGN.md §4 "Replica exchange").  Test infrastructure: compiled by tests/exchange_oracle.py, never by the product.
 *
 * A ladder is L consecutive chains by global index; chain g is rung g % L.  Round R pairs rungs (r, r+1) with
 * r == R (mod 2); the pair with lower chain g swaps x (and e) iff
 *   min(1, exp(D)) > u,   D = (b_g - b_{g+1}) * (e_g - e_{g+1}),   e = potential(x)
 * with u = (A >> 11) * 2^-53, A the first word of Philox4x32-10 with key (4, 'ARIA') and counter
 * (sid_lo, R_lo, sid_hi, R_hi << 8), sid = seed + g (the stream layout of DESIGN.md "RNG stream layout", tag 4).
 * Strict >, NaN rejects (metropolis.jl:183-185).  exp is libm's.
 *
 * Build: gcc -O2 -ffp-contract=off -fPIC -shared -- one IEEE-754 binary64 operation per statement.
 */
#include <math.h>
#include <stdint.h>

#define XO_API __attribute__((visibility("default")))

static void philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
    uint32_t k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* the exchange uniform of the pair whose lower chain has stream id sid, in round R */
XO_API double xo_exchange_uniform(uint64_t sid, uint64_t R)
{
    uint32_t ctr[4] = {(uint32_t)sid, (uint32_t)R, (uint32_t)(sid >> 32), (uint32_t)(R >> 32) << 8};
    uint32_t key[2] = {4u, 0x41524941u};
    uint32_t o[4];
    philox4x32_10(ctr, key, o);
    uint64_t A = (uint64_t)o[0] | ((uint64_t)o[1] << 32);
    return (double)(A >> 11) * 0x1.0p-53;
}

/* potential ids of include/arianna_cuda.h */
static double potential(int pot, double x)
{
    switch (pot) {
    default:
    case 0: return x * x;
    case 1: { double x2 = x * x; return x2 * x2; }
    case 2: { double w = x * x - 1.0; return w * w; }
    }
}

/* One round over x, e, betas: [M] local chains starting at global chain chain_offset (both multiples of L).
 * accepted: [L-1] swaps per rung pair, ADDED to. */
XO_API void xo_exchange_round(int64_t M, int L, int64_t seed, int64_t chain_offset, int64_t R, int pot, double *x,
                              double *e, const double *betas, int64_t *accepted)
{
    for (int64_t base = 0; base < M; base += L) {
        for (int r = (int)(R & 1); r + 1 < L; r += 2) {
            int64_t g = base + r;
            double e0 = potential(pot, x[g]), e1 = potential(pot, x[g + 1]);
            double d = (betas[g] - betas[g + 1]) * (e0 - e1);
            double ex = exp(d);
            double a = (ex > 1.0) ? 1.0 : ex;             /* min(1, .); NaN propagates */
            if (a > xo_exchange_uniform((uint64_t)(seed + chain_offset + g), (uint64_t)R)) {
                double t = x[g]; x[g] = x[g + 1]; x[g + 1] = t;
                e[g] = e1; e[g + 1] = e0;
                accepted[r] += 1;
            }
        }
    }
}

/* Per-rung callback sums: out[r][2 + n_moves] = (sum e, sum_c acc_ck/tot_ck per move, count) over the chains of rung
 * r (local index % L == r), sequential sums.  acc / tot: [n_moves][M]. */
XO_API void xo_ladder_sums(int64_t M, int L, int n_moves, const double *e, const int64_t *acc, const int64_t *tot,
                           double *out)
{
    int w = 2 + n_moves;
    for (int r = 0; r < L; ++r) {
        double se = 0.0, cnt = 0.0;
        for (int64_t c = r; c < M; c += L) { se = se + e[c]; cnt = cnt + 1.0; }
        out[r * w] = se;
        for (int k = 0; k < n_moves; ++k) {
            double s = 0.0;
            for (int64_t c = r; c < M; c += L)
                s = s + (double)acc[(int64_t)k * M + c] / (double)tot[(int64_t)k * M + c];
            out[r * w + 1 + k] = s;
        }
        out[r * w + 1 + n_moves] = cnt;
    }
}
