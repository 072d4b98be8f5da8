// scan.cuh -- device-wide exclusive prefix product over Fr: out[0] = 1, out[i] = a[0] * ... * a[i-1], plus the product of all
// n elements.  This is the grand product of the permutation argument (dusk-plonk 0.8 compute_fast_permutation_poly: z_0 = 1,
// z_{i+1} = z_i * num_i / den_i), computed over the ratios num_i / den_i.
//
// Three phases over tiles of SCAN_TILE = 1024 consecutive elements:
//   1. k_fr_scan_reduce: the product of every tile (coalesced loads, xor-butterfly over warp shuffles, 8 warp totals in shared memory);
//   2. the exclusive scan of the tile totals -- by one block of k_fr_scan_apply when they fit one tile, else by the same three
//      phases one level up (2^25 elements: 32768 totals -> 32 -> one block);
//   3. k_fr_scan_apply: the tile is staged in shared memory (coalesced), every thread multiplies its 4 consecutive elements
//      serially, the 256 thread products are scanned with shfl_up inside each warp and across the 8 warp totals in shared memory,
//      and every thread walks its elements again from (tile prefix x thread prefix), writing the exclusive products.
// The elements are read twice and written once.  Montgomery multiplication is exact, so the result is bit-identical to the serial
// product for every tiling.  In place (out == in) is allowed: a block reads its whole tile before it writes any of it.
#pragma once
#include "layout.h"

namespace pg {

constexpr int SCAN_THREADS = 256, SCAN_E = 4;
constexpr uint64_t SCAN_TILE = (uint64_t)SCAN_THREADS * SCAN_E;
// scalars of scratch the multi-level scan of n elements needs: the tile totals of every level above the first
inline uint64_t fr_scan_scratch(uint64_t n) {
    uint64_t s = 0;
    while (n > SCAN_TILE) { n = (n + SCAN_TILE - 1) / SCAN_TILE; s += n; }
    return s;
}

// the definition, as one unit of work: out[i] = a[0]*..*a[i-1], *total = the product of all n.  The engine runs it only on a backend
// without a device-wide scan (the test-only loop backend); CudaBackend::run_fr_scan computes the same with the kernels below.
struct FrScanSerialBody {
    struct Args { const uint4* in; uint4* out; uint64_t n; uint4* total; };
    PG_HD static void run(const Args& a, uint64_t) {
        Fr acc = fr_one();
        for (uint64_t i = 0; i < a.n; i++) { const Fr v = aos_load(a.in, i); aos_store(a.out, i, acc); acc = fr_mul(acc, v); }
        aos_store(a.total, 0, acc);
    }
};

// ---- Ruffini division: the exclusive suffix of the linear recurrence s_i = f_i + p * s_(i+1), s_n = 0, with a constant multiplier p:
//   out[i] = s_(i+1) = sum_(k>i) f_k p^(k-i-1)   (i < n),   *rem = s_0 = f(p).
// out[0 .. n-1) is the quotient of f(X) by (X - p) (dusk-plonk Polynomial::ruffini: q_(n-2) = f_(n-1), q_(i-1) = f_i + p q_i) and
// out[n-1] = 0.  Same three phases over tiles of SCAN_TILE elements as the prefix product:
//   1. k_fr_ruffini_reduce: L_b = sum_(j<TILE) f_(bT+j) p^j per tile (Horner in p^256 over a thread's strided elements, times p^t);
//   2. the tile values satisfy S_b = L_b + p^T S_(b+1), the same recurrence with multiplier p^T: one level up, recursively, gives
//      every tile its carry S_(b+1) and the top level's remainder S_0 = f(p);
//   3. k_fr_ruffini_apply: the tile is staged in shared memory, every thread runs Horner over its 4 consecutive elements, the
//      256 thread values are suffix-scanned (shfl_down in a warp with multipliers p^(4d), then across the 8 warps with p^(128d)), the
//      tile's carry enters with p^(T - offset), and every thread walks its elements down again writing s_(i+1).
// A thread's carry in is its top element's offset in the tile: the powers p^k, k <= SCAN_TILE, come from one table per level (RUF_TAB
// entries; level l + 1 holds the powers of p^(T^(l+1))).  Exact arithmetic: bit-identical to the serial loop for every n and tiling.
// In place (out == in) is allowed: a block writes only its own tile, after it has read all of it.
constexpr uint64_t RUF_TAB = SCAN_TILE + 1;
inline uint32_t fr_ruffini_levels(uint64_t n) {
    uint32_t l = 1;
    while (n > SCAN_TILE) { n = (n + SCAN_TILE - 1) / SCAN_TILE; l++; }
    return l;
}

// the definition, as one unit of work; the engine runs it only on a backend without run_fr_ruffini (the test-only loop backend)
struct FrRuffiniSerialBody {
    struct Args { const uint4* in; uint4* out; uint64_t n; Fr p; uint4* rem; };
    PG_HD static void run(const Args& a, uint64_t) {
        Fr acc = fr_zero();
        for (uint64_t i = a.n; i-- > 0;) { const Fr f = aos_load(a.in, i); aos_store(a.out, i, acc); acc = fr_add(f, fr_mul(a.p, acc)); }
        aos_store(a.rem, 0, acc);
    }
};

#if defined(__CUDACC__)
__device__ __forceinline__ Fr shfl_down_fr(const Fr& a, int d) {
    Fr r;
#pragma unroll
    for (int k = 0; k < 8; k++) r.v[k] = __shfl_down_sync(0xffffffffu, a.v[k], d);
    return r;
}
__device__ __forceinline__ Fr shfl_up_fr(const Fr& a, int d) {
    Fr r;
#pragma unroll
    for (int k = 0; k < 8; k++) r.v[k] = __shfl_up_sync(0xffffffffu, a.v[k], d);
    return r;
}
__device__ __forceinline__ Fr shfl_xor_prod(const Fr& a, int mask) {
    Fr r;
#pragma unroll
    for (int k = 0; k < 8; k++) r.v[k] = __shfl_xor_sync(0xffffffffu, a.v[k], mask);
    return fr_mul(a, r);
}
// shared-memory tile: two planes of 16-byte halves, one padding entry every 8 elements, so that a quarter warp reading the
// consecutive elements 4t .. 4t+3 of eight threads hits eight different banks
__device__ __forceinline__ uint32_t scan_slot(uint32_t e) { return e + (e >> 3); }
constexpr uint32_t SCAN_SLOTS = (uint32_t)SCAN_TILE + (uint32_t)SCAN_TILE / 8;

// Exclusive scan of one Fr per thread over the block; *total = product of all SCAN_THREADS values.  Every thread must call.
__device__ __forceinline__ Fr block_exclusive_product(const Fr& x, Fr* s_warp /* 8 */, Fr* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Fr incl = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const Fr y = shfl_up_fr(incl, d); if (lane >= d) incl = fr_mul(incl, y); }
    Fr excl = shfl_up_fr(incl, 1);
    if (lane == 0) excl = fr_one();
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        constexpr int W = SCAN_THREADS / 32;
        Fr h = lane < W ? s_warp[lane] : fr_one();
#pragma unroll
        for (int d = 1; d < W; d <<= 1) { const Fr y = shfl_up_fr(h, d); if (lane >= d) h = fr_mul(h, y); }
        Fr he = shfl_up_fr(h, 1);
        if (lane == 0) he = fr_one();
        __syncwarp();
        if (lane < W) s_warp[lane] = he;
        if (lane == W - 1) s_warp[W] = h;
    }
    __syncthreads();
    *total = s_warp[SCAN_THREADS / 32];
    return fr_mul(s_warp[warp], excl);
}

// phase 1: totals[b] = product of tile b
__global__ void __launch_bounds__(SCAN_THREADS) k_fr_scan_reduce(const uint4* in, uint64_t n, uint4* totals) {
    __shared__ Fr s_warp[SCAN_THREADS / 32];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE;
    Fr p = fr_one();
#pragma unroll
    for (int e = 0; e < SCAN_E; e++) {
        const uint64_t i = base + (uint64_t)e * SCAN_THREADS + threadIdx.x;
        if (i < n) p = fr_mul(p, aos_load(in, i));
    }
#pragma unroll
    for (int m = 1; m < 32; m <<= 1) p = shfl_xor_prod(p, m);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = p;
    __syncthreads();
    if (threadIdx.x == 0) {
        Fr t = s_warp[0];
        for (int w = 1; w < SCAN_THREADS / 32; w++) t = fr_mul(t, s_warp[w]);
        aos_store(totals, blockIdx.x, t);
    }
}

// phase 3 (and phase 2 when one block holds all tile totals): out[i] = prefix[tile] * (exclusive product inside the tile);
// prefix == nullptr: 1.  total != nullptr (single-block launch): the product of all n elements.
__global__ void __launch_bounds__(SCAN_THREADS) k_fr_scan_apply(const uint4* in, uint4* out, uint64_t n, const uint4* prefix, uint4* total) {
    __shared__ __align__(16) uint4 s_lo[SCAN_SLOTS], s_hi[SCAN_SLOTS];
    __shared__ Fr s_warp[SCAN_THREADS / 32 + 1];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE;
    const Fr one = fr_one();
#pragma unroll
    for (int e = 0; e < SCAN_E; e++) {                                    // coalesced: element base + e*256 + t
        const uint32_t j = (uint32_t)e * SCAN_THREADS + threadIdx.x;
        const Fr v = base + j < n ? aos_load(in, base + j) : one;
        s_lo[scan_slot(j)] = make_uint4(v.v[0], v.v[1], v.v[2], v.v[3]);
        s_hi[scan_slot(j)] = make_uint4(v.v[4], v.v[5], v.v[6], v.v[7]);
    }
    __syncthreads();
    auto at = [&](uint32_t j) { const uint4 lo = s_lo[scan_slot(j)], hi = s_hi[scan_slot(j)]; Fr r = {{lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w}}; return r; };
    const uint32_t j0 = threadIdx.x * SCAN_E;                             // this thread's consecutive elements
    Fr mine = at(j0);
#pragma unroll
    for (int e = 1; e < SCAN_E; e++) mine = fr_mul(mine, at(j0 + e));
    Fr tile_total;
    Fr run = block_exclusive_product(mine, s_warp, &tile_total);
    if (prefix) run = fr_mul(aos_load(prefix, blockIdx.x), run);
    Fr v[SCAN_E];
#pragma unroll
    for (int e = 0; e < SCAN_E; e++) v[e] = at(j0 + e);
    __syncthreads();                                                      // every thread has read its elements
#pragma unroll
    for (int e = 0; e < SCAN_E; e++) {
        s_lo[scan_slot(j0 + e)] = make_uint4(run.v[0], run.v[1], run.v[2], run.v[3]);
        s_hi[scan_slot(j0 + e)] = make_uint4(run.v[4], run.v[5], run.v[6], run.v[7]);
        run = fr_mul(run, v[e]);
    }
    if (total && threadIdx.x == SCAN_THREADS - 1) aos_store(total, 0, run);
    __syncthreads();
#pragma unroll
    for (int e = 0; e < SCAN_E; e++) {
        const uint32_t j = (uint32_t)e * SCAN_THREADS + threadIdx.x;
        if (base + j < n) aos_store(out, base + j, at(j));
    }
}

// Ruffini phase 1: totals[b] = sum_(j<TILE) f_(bT+j) p^j; pw = this level's table p^0 .. p^TILE
__global__ void __launch_bounds__(SCAN_THREADS) k_fr_ruffini_reduce(const uint4* in, uint64_t n, const uint4* pw, uint4* totals) {
    __shared__ Fr s_warp[SCAN_THREADS / 32];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE;
    const Fr step = aos_load(pw, SCAN_THREADS);                           // p^256: the distance between a thread's elements
    Fr acc = fr_zero();
#pragma unroll
    for (int e = SCAN_E - 1; e >= 0; e--) {                               // coalesced: element base + e*256 + t
        const uint64_t i = base + (uint64_t)e * SCAN_THREADS + threadIdx.x;
        acc = fr_mul(acc, step);
        if (i < n) acc = fr_add(acc, aos_load(in, i));
    }
    acc = fr_mul(acc, aos_load(pw, threadIdx.x));
#pragma unroll
    for (int m = 1; m < 32; m <<= 1) {
        Fr r;
#pragma unroll
        for (int k = 0; k < 8; k++) r.v[k] = __shfl_xor_sync(0xffffffffu, acc.v[k], m);
        acc = fr_add(acc, r);
    }
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        Fr t = s_warp[0];
        for (int w = 1; w < SCAN_THREADS / 32; w++) t = fr_add(t, s_warp[w]);
        aos_store(totals, blockIdx.x, t);
    }
}

// Ruffini phase 3 (and phase 2 when one block holds all tile values): out[i] = s_(i+1) inside the tile, with the tile's carry
// s_(bT+T) from carry[b] (nullptr: 0, the top of the vector).  rem != nullptr (single-block launch): s_0.
__global__ void __launch_bounds__(SCAN_THREADS) k_fr_ruffini_apply(const uint4* in, uint4* out, uint64_t n, const uint4* pw, const uint4* carry,
                                                                   uint4* rem) {
    __shared__ __align__(16) uint4 s_lo[SCAN_SLOTS], s_hi[SCAN_SLOTS];
    __shared__ Fr s_warp[SCAN_THREADS / 32];
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE;
    const Fr zero = fr_zero();
#pragma unroll
    for (int e = 0; e < SCAN_E; e++) {                                    // coalesced: element base + e*256 + t
        const uint32_t j = (uint32_t)e * SCAN_THREADS + threadIdx.x;
        const Fr v = base + j < n ? aos_load(in, base + j) : zero;
        s_lo[scan_slot(j)] = make_uint4(v.v[0], v.v[1], v.v[2], v.v[3]);
        s_hi[scan_slot(j)] = make_uint4(v.v[4], v.v[5], v.v[6], v.v[7]);
    }
    __syncthreads();
    auto at = [&](uint32_t j) { const uint4 lo = s_lo[scan_slot(j)], hi = s_hi[scan_slot(j)]; Fr r = {{lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w}}; return r; };
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t j0 = threadIdx.x * SCAN_E;                             // this thread's consecutive elements
    const Fr p = aos_load(pw, 1);
    Fr v[SCAN_E];
#pragma unroll
    for (int e = 0; e < SCAN_E; e++) v[e] = at(j0 + e);
    Fr h = v[SCAN_E - 1];                                                 // sum_e f_(j0+e) p^e
#pragma unroll
    for (int e = SCAN_E - 2; e >= 0; e--) h = fr_add(v[e], fr_mul(p, h));
    // suffix inside the warp: incl_t = sum_(t' >= t) h_t' p^(4(t'-t))
    Fr incl = h;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const Fr y = shfl_down_fr(incl, d);
        if (lane + d < 32) incl = fr_add(incl, fr_mul(aos_load(pw, SCAN_E * d), y));
    }
    Fr ex = shfl_down_fr(incl, 1);                                        // threads above this one in the warp
    if (lane == 31) ex = zero;
    if (lane == 0) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {                                                      // across the warps (multiplier p^128 per warp), then the carry
        constexpr int W = SCAN_THREADS / 32;
        Fr x = lane < W ? s_warp[lane] : zero;
#pragma unroll
        for (int d = 1; d < W; d <<= 1) {
            const Fr y = shfl_down_fr(x, d);
            if (lane + d < W) x = fr_add(x, fr_mul(aos_load(pw, 32 * SCAN_E * d), y));
        }
        Fr xe = shfl_down_fr(x, 1);                                       // warps above this one: s at the warp's top, without the carry
        if (lane == W - 1) xe = zero;
        if (carry && lane < W) xe = fr_add(xe, fr_mul(aos_load(pw, 32 * SCAN_E * (W - 1 - lane)), aos_load(carry, blockIdx.x)));
        __syncwarp();
        if (lane < W) s_warp[lane] = xe;
    }
    __syncthreads();
    Fr run = fr_add(ex, fr_mul(aos_load(pw, SCAN_E * (31 - lane)), s_warp[warp]));   // s_(j0+4)
    __syncthreads();                                                      // every thread has read its elements
#pragma unroll
    for (int e = SCAN_E - 1; e >= 0; e--) {
        s_lo[scan_slot(j0 + e)] = make_uint4(run.v[0], run.v[1], run.v[2], run.v[3]);
        s_hi[scan_slot(j0 + e)] = make_uint4(run.v[4], run.v[5], run.v[6], run.v[7]);
        run = fr_add(v[e], fr_mul(p, run));
    }
    if (rem && threadIdx.x == 0) aos_store(rem, 0, run);
    __syncthreads();
#pragma unroll
    for (int e = 0; e < SCAN_E; e++) {
        const uint32_t j = (uint32_t)e * SCAN_THREADS + threadIdx.x;
        if (base + j < n) aos_store(out, base + j, at(j));
    }
}
#endif

}  // namespace pg
