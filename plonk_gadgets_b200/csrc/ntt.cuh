// ntt.cuh -- number-theoretic transform over the BLS12-381 scalar field on dusk-plonk's evaluation domain
// (SURVEY.md section 8f item 2, first half: the step right after the gadget hot path inside `Prover::prove`:
// wire columns -> zero-padded scalar vectors -> `domain.ifft` -> coefficients of w_l, w_r, w_o, w_4).
//
// Semantics ([DEP] dusk-plonk 0.8 src/fft/domain.rs, reached from /root/reference/tests/range_gadgets_tests.rs:90-91):
//   fft :  A_k = sum_j a_j w^(jk),   w = ROOT_OF_UNITY^(2^(32 - log_n)),  ROOT_OF_UNITY = 7^((q-1)/2^32)
//   ifft:  the same with w^-1, every element multiplied by n^-1.
// Both are natural order in, natural order out.  The DFT of a vector is unique and Fr elements are kept fully reduced, so any
// correct schedule yields the same limbs as the reference's serial radix-2 loop; the schedule here is chosen for the B200:
//
//   1. the bit-reversal permutation (and the n^-1 scaling of the inverse transform) is folded into the loads of the first
//      pass, which writes to a scratch vector; the last pass writes back to the caller's buffer (transforms of up to 2^11
//      points are one block and run in place);
//   2. k_ntt_pass, ceil((log_n - 11) / 8) + 1 launches: a block owns a tile of 2^s x C elements (s butterfly stages; C >= 8
//      neighbouring sub-transforms so that every global access of a warp covers whole 256-byte runs), keeps it in shared
//      memory (64 KiB, 128-bit accesses), and runs the s stages there two at a time: a thread holds four elements in
//      registers and does the four decimation-in-time butterflies (1 Montgomery multiplication, 1 add, 1 sub each) of a
//      stage pair between two barriers.  The vector crosses HBM once per pass (3 passes at 2^26) while the
//      log_n/2 multiplications per element stay on the multiplier pipe: the transform is IMAD-bound like the gate check.
//   Twiddles w^i (i <= n/2) come from a table built once per domain size by k_simple<NttTwiddleBody>.  The inverse transform
//   reads the same table backwards, w^-i = -w^(n/2 - i), and never negates: with t' = x1 * w^(n/2 - i) = -(x1 * w^-i) the
//   butterfly's outputs are x0 - t' and x0 + t' -- the forward butterfly with its two results exchanged (entry n/2 = -1 serves
//   i = 0).  A pass touches about as many table bytes as data bytes, mostly out of L2.
#pragma once
#include "layout.h"

namespace pg {

constexpr uint32_t NTT_TWO_ADICITY = 32;
constexpr uint32_t NTT_MAX_LOG_TILE = 11;     // 2048 elements = 64 KiB of shared memory per block
constexpr int NTT_THREADS = 256;

// 7^((q-1)/2^32) in Montgomery form (dusk-bls12_381 ROOT_OF_UNITY; recomputed by tests/test_oracle_fft.py)
PG_HD Fr fr_root_of_unity() { Fr r = {{0x5f0e466au, 0xb9b58d8cu, 0x1819d7ecu, 0x5b1b4c80u, 0x52a31e64u, 0x0af53ae3u, 0x19e9b27bu, 0x5bf3addau}}; return r; }

PG_HD uint64_t bitrev64(uint64_t x, uint32_t bits) {
#if defined(__CUDA_ARCH__)
    return bits ? __brevll(x) >> (64 - bits) : 0;
#else
    uint64_t r = 0;
    for (uint32_t i = 0; i < bits; i++) { r = (r << 1) | (x & 1); x >>= 1; }
    return r;
#endif
}

// ---- twiddle table: tw[i] = w^i, i <= n/2 (n_entries = n/2 + 1; the last one is -1); 16 consecutive entries per call -----
struct NttTwiddleBody {
    struct Args { uint4* tw; uint64_t n_entries; uint64_t n; /* calls */ uint32_t log_n; Fr pw2[NTT_TWO_ADICITY]; /* w^(2^b) */ };
    PG_HD static void run(const Args& a, uint64_t j) {
        const uint64_t i0 = j * 16;
        Fr x = fr_one();
        for (uint32_t b = 4; b < a.log_n; b++)
            if ((i0 >> b) & 1) x = fr_mul(x, a.pw2[b]);
        for (uint32_t r = 0; r < 16 && i0 + r < a.n_entries; r++) { aos_store(a.tw, i0 + r, x); x = fr_mul(x, a.pw2[0]); }
    }
};

// w^j for any j < n from that table: w^(j + n/2) = -w^j.  log_n == 0 (one point, no table): 1.
PG_HD Fr domain_pow(const uint4* tw, uint32_t log_n, uint64_t j) {
    if (!log_n) return fr_one();
    const uint64_t h = 1ull << (log_n - 1u);
    return j <= h ? aos_load(tw, j) : fr_neg(aos_load(tw, j - h));
}

// zero-fill of the padding rows [n0, n) of a column
struct NttZeroBody {
    struct Args { uint4* data; uint64_t n0; uint64_t n; };
    PG_HD static void run(const Args& a, uint64_t i) { aos_store(a.data, a.n0 + i, fr_zero()); }
};

// ---- one pass = s consecutive butterfly stages [t0, t0 + s) ------------------------------------------------------------
// Index of an element: (g_hi, v, g_lo) with g_lo < 2^t0 and v < 2^s; the pass couples elements that differ in v only.
// Tile `blk` holds the C = 2^log_c values g = blk*C + c of the combined index g = (g_hi, g_lo), all v: tile element
// e = v*C + c.  With t0 >= log_c the C elements of a v share g_hi and are neighbours in memory.
// A pass reads its tile from `src` and writes it to `dst` (the same buffer for the passes in the middle).  The first pass
// of a transform (t0 == 0) can gather its input through the bit-reversal permutation (bitrev != 0) and multiply it by
// `factor` (scale != 0: the n^-1 of the inverse transform): no separate permutation pass.  Such a pass must not run in place
// unless it is a single block.
// shift != 0 (forward transforms only: EvaluationDomain::coset_fft): the first pass also multiplies source element m by h^m, read
// from a two-level table, shift_tab[m & (2^shift_log_lo - 1)] * shift_tab[2^shift_log_lo + (m >> shift_log_lo)] (pow_table_host);
// such a pass runs as k_ntt_coset_pass so that k_ntt_pass is compiled without it.
struct NttPassArgs { const uint4* src; uint4* dst; const uint4* tw; uint32_t log_n, t0, s, log_c; int inverse; int bitrev; int scale; Fr factor;
                     int shift; uint32_t shift_log_lo; const uint4* shift_tab; };

// h^m for m < 2^log_n from a two-level table of h: [h^0 .. h^(L-1)] then [h^0, h^L, h^(2L) ..], L = 2^log_lo
PG_HD Fr pow_table_at(const uint4* tab, uint32_t log_lo, uint64_t m) {
    return fr_mul(aos_load(tab, m & ((1ull << log_lo) - 1ull)), aos_load(tab, (1ull << log_lo) + (m >> log_lo)));
}
PG_HD uint32_t pow_table_log_lo(uint32_t log_n) { return (log_n + 1) / 2; }
PG_HD uint64_t pow_table_entries(uint32_t log_n) { const uint32_t lo = pow_table_log_lo(log_n); return (1ull << lo) + (1ull << (log_n - lo)); }
// the table of h for exponents below 2^log_n (host code; a few thousand multiplications)
inline void pow_table_host(Fr h, uint32_t log_n, Fr* out) {
    const uint32_t lo = pow_table_log_lo(log_n);
    const uint64_t L = 1ull << lo, H = 1ull << (log_n - lo);
    Fr x = fr_one();
    for (uint64_t i = 0; i < L; i++) { out[i] = x; x = fr_mul(x, h); }     // x = h^L afterwards
    Fr y = fr_one();
    for (uint64_t i = 0; i < H; i++) { out[L + i] = y; y = fr_mul(y, x); }
}

PG_HD uint64_t ntt_index(const NttPassArgs& a, uint64_t blk, uint32_t e) {
    const uint32_t c = e & ((1u << a.log_c) - 1u), v = e >> a.log_c;
    const uint64_t g = (blk << a.log_c) | c;
    const uint64_t g_lo = g & ((1ull << a.t0) - 1ull), g_hi = g >> a.t0;
    return (g_hi << (a.t0 + a.s)) | ((uint64_t)v << a.t0) | g_lo;
}
// butterfly b (< 2^(s-1) * C) of step u (stage t0 + u): tile elements e0 < e1 and the twiddle exponent
PG_HD void ntt_butterfly(const NttPassArgs& a, uint64_t blk, uint32_t u, uint32_t b, uint32_t& e0, uint32_t& e1, uint64_t& tw_index) {
    const uint32_t c = b & ((1u << a.log_c) - 1u), bf = b >> a.log_c;
    const uint32_t low = bf & ((1u << u) - 1u);
    const uint32_t v0 = ((bf >> u) << (u + 1)) | low;
    e0 = (v0 << a.log_c) | c;
    e1 = e0 + (1u << (u + a.log_c));
    const uint64_t g = (blk << a.log_c) | c;
    const uint64_t pos = ((uint64_t)low << a.t0) | (g & ((1ull << a.t0) - 1ull));     // index inside the half block of size m = 2^(t0+u)
    tw_index = pos << (a.log_n - 1u - (a.t0 + u));                                    // pos * n / (2m)  < n/2
}
// forward: w^i.  Inverse: w^(n/2 - i) = -w^-i -- the caller exchanges the butterfly's two results instead of negating
PG_HD Fr ntt_twiddle(const NttPassArgs& a, uint64_t tw_index) {
    return aos_load(a.tw, a.inverse ? (1ull << (a.log_n - 1u)) - tw_index : tw_index);
}

#if defined(__CUDACC__)
// Shared-memory tile: two planes of 16-byte half scalars, [lo half of every element][hi half of every element]; a warp that
// touches consecutive elements makes conflict-free 128-bit accesses.
__device__ __forceinline__ Fr tile_load(const uint4* tile, uint32_t E, uint32_t e) {
    const uint4 lo = tile[e], hi = tile[E + e];
    Fr r = {{lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w}};
    return r;
}
__device__ __forceinline__ void tile_store(uint4* tile, uint32_t E, uint32_t e, const Fr& x) {
    tile[e] = make_uint4(x.v[0], x.v[1], x.v[2], x.v[3]);
    tile[E + e] = make_uint4(x.v[4], x.v[5], x.v[6], x.v[7]);
}
// 32-bit index arithmetic throughout: element indices are < 2^32 (log_n <= 32), only the final byte address is 64-bit.
__device__ __forceinline__ uint32_t ntt_index32(const NttPassArgs& a, uint32_t blk, uint32_t e) {
    const uint32_t c = e & ((1u << a.log_c) - 1u), v = e >> a.log_c;
    const uint32_t g = (blk << a.log_c) | c;
    const uint32_t g_lo = a.t0 ? g & (0xffffffffu >> (32u - a.t0)) : 0u, g_hi = a.t0 < 32u ? g >> a.t0 : 0u;
    const uint32_t sh = a.t0 + a.s;
    return (sh < 32u ? g_hi << sh : 0u) | (v << a.t0) | g_lo;
}
template <bool INV>
__device__ __forceinline__ Fr ntt_twiddle32(const NttPassArgs& a, uint32_t ti) {
    return aos_load(a.tw, INV ? (1u << (a.log_n - 1u)) - ti : ti);
}
// x0, x1 <- x0 + w x1, x0 - w x1 with t = x1 * (table entry): the inverse transform's entry is -w, so its results are exchanged
template <bool INV>
__device__ __forceinline__ void ntt_bfly(Fr& x0, Fr& x1, const Fr& t) {
    const Fr s = fr_add(x0, t), d = fr_sub(x0, t);
    x0 = INV ? d : s; x1 = INV ? s : d;
}

// Two butterfly stages per trip through shared memory: a thread takes the four elements that differ in bits u and u+1 of v,
// runs stage t0+u on the pairs (0,1), (2,3) -- they share one twiddle -- and stage t0+u+1 on (0,2), (1,3), whose twiddle
// exponents differ by n/4.  An odd stage count ends with one radix-2 step.
// stages t0+u and t0+u+1 on the tile (FIRST: t0 = u = 0, see k_ntt_pass)
template <bool INV, bool FIRST>
__device__ __forceinline__ void ntt_stage_pair(const NttPassArgs& a, uint4* s_tile, uint32_t E, uint32_t blk, uint32_t u, const QRegs& q) {
    const uint32_t c_mask = (1u << a.log_c) - 1u, lo_mask = a.t0 ? 0xffffffffu >> (32u - a.t0) : 0u;
    const uint32_t sh = a.log_n - 1u - (a.t0 + u);                // stage t0+u: exponent = pos << sh
#pragma unroll 1
    for (uint32_t r = threadIdx.x; r < E / 4; r += NTT_THREADS) {
        const uint32_t c = r & c_mask, bf = r >> a.log_c;
        const uint32_t low = bf & ((1u << u) - 1u);
        const uint32_t v0 = ((bf >> u) << (u + 2)) | low;
        const uint32_t e0 = (v0 << a.log_c) | c, d = 1u << (u + a.log_c);
        const uint32_t pos = (low << a.t0) | (((blk << a.log_c) | c) & lo_mask);
        const uint32_t ti = pos << sh;
        Fr x0 = tile_load(s_tile, E, e0), x1 = tile_load(s_tile, E, e0 + d);
        Fr x2 = tile_load(s_tile, E, e0 + 2 * d), x3 = tile_load(s_tile, E, e0 + 3 * d);
        if (FIRST) {                                              // ti == 0
            ntt_bfly<false>(x0, x1, x1);
            ntt_bfly<false>(x2, x3, x3);
            ntt_bfly<false>(x0, x2, x2);
        } else {
            const Fr w = ntt_twiddle32<INV>(a, ti);
            const Fr t1 = fr_mul_eo(x1, w, q), t3 = fr_mul_eo(x3, w, q);
            ntt_bfly<INV>(x0, x1, t1);
            ntt_bfly<INV>(x2, x3, t3);
            const Fr wa = ntt_twiddle32<INV>(a, ti >> 1);
            const Fr t2 = fr_mul_eo(x2, wa, q);
            ntt_bfly<INV>(x0, x2, t2);
        }
        const Fr wb = ntt_twiddle32<INV>(a, (ti >> 1) + (1u << (a.log_n - 2u)));
        const Fr t3 = fr_mul_eo(x3, wb, q);
        ntt_bfly<INV>(x1, x3, t3);
        tile_store(s_tile, E, e0, x0); tile_store(s_tile, E, e0 + d, x1);
        tile_store(s_tile, E, e0 + 2 * d, x2); tile_store(s_tile, E, e0 + 3 * d, x3);
    }
}
template <bool INV, bool SHIFT>
__device__ __forceinline__ void ntt_pass_body(const NttPassArgs& a, uint4* s_tile, uint32_t* s_q) {
    const uint32_t log_e = a.s + a.log_c, E = 1u << log_e;
    const uint32_t blk = blockIdx.x;
    if (threadIdx.x < 8) s_q[threadIdx.x] = c_q[threadIdx.x];
    for (uint32_t e = threadIdx.x; e < E; e += NTT_THREADS)
    {
        const uint32_t idx = ntt_index32(a, blk, e);
        const uint32_t m = a.bitrev ? (a.log_n ? __brev(idx) >> (32u - a.log_n) : 0u) : idx;
        Fr x = aos_load(a.src, m);
        if (a.scale) x = fr_mul_eo(x, a.factor);
        if (SHIFT) x = fr_mul_eo(x, pow_table_at(a.shift_tab, a.shift_log_lo, m));
        tile_store(s_tile, E, e, x);
    }
    __syncthreads();
    QRegs q;
#pragma unroll
    for (int k = 0; k < 8; k++) q.v[k] = s_q[k];
    const uint32_t c_mask = (1u << a.log_c) - 1u, lo_mask = a.t0 ? 0xffffffffu >> (32u - a.t0) : 0u;
    uint32_t u = 0;
    // The first two stages of a transform (t0 = 0, u = 0) have the twiddles w^0 = 1 (stage 0, and the pairs (0,2) of stage 1) and
    // w^(n/4) (the pairs (1,3)): one multiplication per group of four instead of four.
    if (a.t0 == 0 && a.s >= 2) { ntt_stage_pair<INV, true>(a, s_tile, E, blk, 0, q); __syncthreads(); u = 2; }
    for (; u + 2 <= a.s; u += 2) { ntt_stage_pair<INV, false>(a, s_tile, E, blk, u, q); __syncthreads(); }
    if (u < a.s) {                                                // last single stage
        const uint32_t sh = a.log_n - 1u - (a.t0 + u);
#pragma unroll 1
        for (uint32_t b = threadIdx.x; b < E / 2; b += NTT_THREADS) {
            const uint32_t c = b & c_mask, bf = b >> a.log_c;
            const uint32_t low = bf & ((1u << u) - 1u);
            const uint32_t v0 = ((bf >> u) << (u + 1)) | low;
            const uint32_t e0 = (v0 << a.log_c) | c, e1 = e0 + (1u << (u + a.log_c));
            const uint32_t pos = (low << a.t0) | (((blk << a.log_c) | c) & lo_mask);
            const Fr w = ntt_twiddle32<INV>(a, pos << sh);
            Fr x0 = tile_load(s_tile, E, e0), x1 = tile_load(s_tile, E, e1);
            const Fr t = fr_mul_eo(x1, w, q);
            ntt_bfly<INV>(x0, x1, t);
            tile_store(s_tile, E, e0, x0); tile_store(s_tile, E, e1, x1);
        }
        __syncthreads();
    }
    for (uint32_t e = threadIdx.x; e < E; e += NTT_THREADS)
        aos_store(a.dst, ntt_index32(a, blk, e), tile_load(s_tile, E, e));
}
template <bool INV>
__global__ void __launch_bounds__(NTT_THREADS, 3) k_ntt_pass(const NttPassArgs a) {
    extern __shared__ __align__(16) uint4 s_tile[];               // [2 halves][E]
    __shared__ uint32_t s_q[8];
    ntt_pass_body<INV, false>(a, s_tile, s_q);
}
// the first pass of a coset transform (shift != 0); the other passes of that transform are ordinary k_ntt_pass launches
__global__ void __launch_bounds__(NTT_THREADS, 3) k_ntt_coset_pass(const NttPassArgs a) {
    extern __shared__ __align__(16) uint4 s_tile[];
    __shared__ uint32_t s_q[8];
    ntt_pass_body<false, true>(a, s_tile, s_q);
}
#endif

// the same tile schedule on the host (tests/emu backend and documentation of the kernel's data flow)
inline void ntt_pass_host(const NttPassArgs& a, uint64_t n_blocks) {
    const uint32_t E = 1u << (a.s + a.log_c);
    Fr* tile = new Fr[E];
    for (uint64_t blk = 0; blk < n_blocks; blk++) {
        for (uint32_t e = 0; e < E; e++) {
            const uint64_t idx = ntt_index(a, blk, e);
            const uint64_t m = a.bitrev ? bitrev64(idx, a.log_n) : idx;
            tile[e] = aos_load(a.src, m);
            if (a.scale) tile[e] = fr_mul(tile[e], a.factor);
            if (a.shift) tile[e] = fr_mul(tile[e], pow_table_at(a.shift_tab, a.shift_log_lo, m));
        }
        for (uint32_t u = 0; u < a.s; u++)
            for (uint32_t b = 0; b < E / 2; b++) {
                uint32_t e0, e1; uint64_t ti;
                ntt_butterfly(a, blk, u, b, e0, e1, ti);
                const Fr t = fr_mul(tile[e1], ntt_twiddle(a, ti));
                const Fr x0 = tile[e0];
                if (a.inverse) { tile[e0] = fr_sub(x0, t); tile[e1] = fr_add(x0, t); }
                else { tile[e0] = fr_add(x0, t); tile[e1] = fr_sub(x0, t); }
            }
        for (uint32_t e = 0; e < E; e++) aos_store(a.dst, ntt_index(a, blk, e), tile[e]);
    }
    delete[] tile;
}

// pass plan: the first pass runs on contiguous tiles (C = 1) and takes up to 11 stages, the others at most 8 stages with C >= 8
struct NttPlan { uint32_t n_pass; uint32_t t0[8], s[8], log_c[8]; };
inline NttPlan ntt_plan(uint32_t log_n) {
    NttPlan p; p.n_pass = 0;
    uint32_t t0 = 0;
    while (t0 < log_n) {
        uint32_t s, log_c;
        if (t0 == 0) { s = log_n < NTT_MAX_LOG_TILE ? log_n : NTT_MAX_LOG_TILE; log_c = 0; }
        else {
            const uint32_t rem = log_n - t0, more = (rem + 7) / 8;
            s = (rem + more - 1) / more;
            log_c = NTT_MAX_LOG_TILE - s;
            if (log_c > log_n - s) log_c = log_n - s;
        }
        p.t0[p.n_pass] = t0; p.s[p.n_pass] = s; p.log_c[p.n_pass] = log_c; p.n_pass++;
        t0 += s;
    }
    return p;
}

}  // namespace pg
