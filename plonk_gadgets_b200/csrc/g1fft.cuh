// g1fft.cuh -- inverse DFT over G1: the Lagrange-basis form of an SRS from its monomial powers alone,
//     lagrange[i] = L_i(tau) G = (1/n) sum_j w^(-ij) powers_of_g[j],   i < n,
// for a user who holds only powers_of_g = [tau^j] G from a trusted setup (pg_srs_lagrange needs tau itself).  The "scalars" of
// this transform are points and every butterfly multiplies one of them by a 255-bit twiddle:
//   1. k_simple<G1FftIngestBody>  affine powers -> XYZZ, times 1/n, stored in bit-reversed order (n x 192 bytes of scratch);
//   2. k_simple<G1FftStageBody>   log n radix-2 decimation-in-time stages, one thread per butterfly, in place;
//   3. k_simple<G1BatchAffineBody> (msm.cuh) back to affine, written to the caller's buffer.
// The 1/n runs as its own multiplication of every input point (n multiplications: at 2^25 about 9 % on top of the
// (n/2) log n - (n - 1) twiddle multiplications of the stages), with the same schedule as the twiddles.
// Twiddles come from the forward table of ntt.cuh (tw[e] = w^e, e <= n/2): w^(-e) = -w^(n/2 - e), and negating a point is free.
// A butterfly whose twiddle is 1 (j = 0 below: all of the first stage, n - 1 in all) multiplies nothing.
#pragma once
#include "msm.cuh"
#include "ntt.cuh"

namespace pg {

PG_HD G1X g1x_neg(const G1X& p) { G1X r = p; r.y = fp_neg(p.y); return r; }

// k * p for a canonical k < 2^256 by a fixed window schedule: a table of 0..15 * p (1 doubling, 13 additions), then the top 4-bit
// digit, then 63 times (4 doublings, one addition of a table entry; digit 0 adds the table's infinity).  The sequence of group
// operations does not depend on k, so lanes with different twiddles run in step, unlike g1x_mul_limbs, which branches on every bit
// and stays the reference.  Fp multiplications (squarings included; g1x_dbl 9, g1x_add 14): 9 + 13*14 + 63*(4*9 + 14) = 3341.
// The table is indexed by the digit, so it lives in local memory (16 x 192 bytes per thread) by design.
constexpr uint32_t G1FFT_MUL_FP_MULS = 9 + 13 * 14 + 63 * (4 * 9 + 14);
PG_HD G1X g1x_mul_fixed(const G1X& p, const Fr& k) {
    G1X tab[16];
    tab[0] = g1x_inf(); tab[1] = p; tab[2] = g1x_dbl(p);
#pragma unroll 1
    for (int d = 3; d < 16; d++) tab[d] = g1x_add(tab[d - 1], p);
    G1X acc = tab[k.v[7] >> 28];
#pragma unroll 1
    for (int w = 62; w >= 0; w--) {
#pragma unroll 1
        for (int b = 0; b < 4; b++) acc = g1x_dbl(acc);
        acc = g1x_add(acc, tab[(k.v[w >> 3] >> (4 * (w & 7))) & 15u]);
    }
    return acc;
}

// data[bitrev(i)] = scale * powers[i], XYZZ; scale is canonical (1/n)
struct G1FftIngestBody {
    struct Args { const uint4* powers; uint4* data; uint64_t n; uint32_t log_n; Fr scale; };
    PG_HD static void run(const Args& a, uint64_t i) {
        g1x_store(a.data, bitrev64(i, a.log_n), g1x_mul_fixed(g1x_from_affine(g1_affine_load(a.powers, i)), a.scale));
    }
};

// Stage s (half-block m = 2^s, B = n / 2m blocks) of the inverse transform, butterfly t < n/2: j = t / B, block k = t % B, elements
// e0 = 2mk + j and e0 + m, twiddle w^(-jB).  Lanes of a warp share j (and the twiddle) while B >= 32 -- the early stages; in the
// late ones their twiddles differ and the fixed schedule of g1x_mul_fixed keeps them in step.
struct G1FftStageBody {
    struct Args { uint4* data; const uint4* tw; uint64_t n; /* butterflies: 2^(log_n - 1) */ uint32_t log_n, s; };
    PG_HD static void run(const Args& a, uint64_t t) {
        const uint32_t lb = a.log_n - 1u - a.s;
        const uint64_t j = t >> lb, k = t & ((1ull << lb) - 1ull);
        const uint64_t e0 = (k << (a.s + 1u)) + j, e1 = e0 + (1ull << a.s);
        G1X v = g1x_load(a.data, e1);
        if (j) v = g1x_neg(g1x_mul_fixed(v, fr_from_mont(aos_load(a.tw, a.n - (j << lb)))));   // w^(-jB) v = -(w^(n/2 - jB) v)
        const G1X u = g1x_load(a.data, e0);                   // loaded after the multiplication: not live across it
        g1x_store(a.data, e0, g1x_add(u, v));
        g1x_store(a.data, e1, g1x_add(u, g1x_neg(v)));
    }
};

}  // namespace pg
