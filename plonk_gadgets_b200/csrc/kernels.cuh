// kernels.cuh -- sm_100a kernels: thin __global__ wrappers around the per-instance bodies (bodies.cuh), the block-wide
// Montgomery batch inversion, the gate-check kernel and the integer-multiply roofline micro-benchmarks.
#pragma once
#include <cuda_runtime.h>
#include <type_traits>
#include "bodies.cuh"
#include "scan.cuh"

namespace pg {

constexpr int BLOCK = 256;            // threads per block of the per-instance kernels (8 warps)
constexpr int NWARPS = BLOCK / 32;

// ---------------------------------------------------------------------------------------------------- simple wrapper
template <class Body>
__global__ void __launch_bounds__(BLOCK) k_simple(const typename Body::Args a) {
    const uint64_t i = (uint64_t)blockIdx.x * BLOCK + threadIdx.x;
    if (i < a.n) Body::run(a, i);
}

// the same with an explicit launch shape (register budget) for bodies that need one: T threads, at least MINB blocks per SM
template <class Body, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) k_simple_shaped(const typename Body::Args a) {
    const uint64_t i = (uint64_t)blockIdx.x * T + threadIdx.x;
    if (i < a.n) Body::run(a, i);
}

// ---------------------------------------------------------------------------------------------------- batch inversion
__device__ __forceinline__ Fr shfl_xor_fr(const Fr& a, int mask) {
    Fr r;
#pragma unroll
    for (int k = 0; k < 8; k++) r.v[k] = __shfl_xor_sync(0xffffffffu, a.v[k], mask);
    return r;
}

// Inverse of one NON-ZERO field element per thread, for a whole thread block, with ONE inversion per block.
// Products are combined with an xor-butterfly over warp shuffles (each lane keeps the sibling product of every level),
// warp totals are staged in shared memory and combined by warp 0 with the same butterfly; the inverse of the block product
// is pushed back down the two butterflies with one multiplication per level.  Every thread of the block must call.
__device__ __forceinline__ Fr block_invert_nonzero(const Fr& p, Fr* smem /* NWARPS entries */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Fr g = p, sib[5];
#pragma unroll
    for (int l = 0; l < 5; l++) { sib[l] = shfl_xor_fr(g, 1 << l); g = fr_mul(g, sib[l]); }      // up-sweep inside the warp
    if (lane == 0) smem[warp] = g;
    __syncthreads();
    if (warp == 0) {
        Fr h = lane < NWARPS ? smem[lane] : fr_one(), hs[3];
#pragma unroll
        for (int l = 0; l < 3; l++) { hs[l] = shfl_xor_fr(h, 1 << l); h = fr_mul(h, hs[l]); }    // NWARPS == 8 -> 3 levels
        Fr ih = lane < NWARPS ? fr_inv_binary(h) : h;                                            // the block's only inversion (the NWARPS lanes hold the same h)
#pragma unroll
        for (int l = 2; l >= 0; l--) ih = fr_mul(ih, hs[l]);                                     // inverse of smem[lane]
        if (lane < NWARPS) smem[lane] = ih;
    }
    __syncthreads();
    Fr ig = smem[warp];                                                                          // inverse of the warp total
#pragma unroll
    for (int l = 4; l >= 0; l--) ig = fr_mul(ig, sib[l]);                                        // inverse of this thread's p
    return ig;
}
static_assert(NWARPS == 8, "block_invert_nonzero's cross-warp butterfly is written for 8 warps");

// Montgomery's trick over table slots, zero-aware:  out_slot[j][i] = in_slot[j][i]^-1, or 0 where the input is 0
// (== BlsScalar::invert().unwrap_or(zero), /root/reference/src/scalar.rs:122; is_non_zero flags the zeros separately).
// The n_pairs x n elements are flattened; a block owns a tile of BLOCK*INV_E consecutive elements and thread t walks the
// elements tile + e*BLOCK + t (every step is a coalesced 128-bit access).
//   pass 1: running product of the thread's elements (zeros patched to 1), each prefix parked in the OUTPUT slot;
//   block : one inversion for the product of all BLOCK*INV_E elements (block_invert_nonzero; binary Euclid, fr_inv_binary);
//   pass 2: walk back -- inverse_e = inv(prefix_e) * prefix_{e-1}, inv(prefix_{e-1}) = inv(prefix_e) * x_e.
// 3 multiplications per element, no per-element state in registers, one inversion per BLOCK*E elements.  E (elements per
// thread) is chosen per launch so that the whole grid is resident at once (one wave, one inversion per block: the launcher
// divides the elements over sm_count x MIN_BLOCKS blocks), with a floor of 8 for small batches.
// Both walks are software-pipelined (the next element's loads are issued before the current multiplication), and the flat index
// is split into (pair, instance) by at most n_pairs - 1 subtractions instead of a 64-bit division.
struct InvCursor {
    uint32_t in_slot, out_slot; uint64_t i; bool valid;
    __device__ __forceinline__ InvCursor(const BatchInvArgs& a, uint64_t idx, uint64_t total) {
        valid = idx < total;
        uint32_t j = 0; i = valid ? idx : 0;
        while (i >= a.n && j + 1 < a.n_pairs) { i -= a.n; j++; }
        in_slot = a.in_slot[j]; out_slot = a.out_slot[j];
    }
};
// Hook (bodies.cuh) fuses a gadget's own element-wise work into the two walks: Hook::pre(h, i) PRODUCES the element to invert
// (and stores it in the input slot, with whatever else the gadget allocates before the inversion) in place of the first
// walk's table load; Hook::post(h, i, x, x^-1) stores what the gadget derives from the inverse.  InvPlain: table to table.
template <class Hook>
__global__ void __launch_bounds__(BLOCK, 2) k_batch_inv(const BatchInvArgs a, const typename Hook::Args h) {
    constexpr bool PLAIN = std::is_same<Hook, InvPlain>::value;
    __shared__ Fr smem[NWARPS];
    const uint64_t total = (uint64_t)a.n_pairs * a.n;
    const int INV_E = (int)a.elems_per_thread;
    const uint64_t first = (uint64_t)blockIdx.x * ((uint64_t)BLOCK * INV_E) + threadIdx.x;
    Fr p = fr_one();
    {
        InvCursor c(a, first, total);
        Fr xn = fr_zero();
        if (c.valid) { if constexpr (PLAIN) xn = tab_load_fr(a.fr, a.stride, c.in_slot, c.i); else xn = Hook::pre(h, c.i); }
#pragma unroll 1
        for (int e = 0; e < INV_E; e++) {
            const Fr x = xn; const InvCursor cur = c;
            if (e + 1 < INV_E) {
                c = InvCursor(a, first + (uint64_t)(e + 1) * BLOCK, total);
                if (c.valid) { if constexpr (PLAIN) xn = tab_load_fr(a.fr, a.stride, c.in_slot, c.i); else xn = Hook::pre(h, c.i); }
            }
            if (cur.valid) {
                if (!fr_is_zero(x)) p = fr_mul(p, x);
                tab_store_fr(a.fr, a.stride, cur.out_slot, cur.i, p);
            }
        }
    }
    Fr ig = block_invert_nonzero(p, smem);                           // inverse of the product of this thread's elements
    {
        InvCursor c(a, first + (uint64_t)(INV_E - 1) * BLOCK, total);
        InvCursor cp(a, first + (uint64_t)(INV_E > 1 ? INV_E - 2 : 0) * BLOCK, total);
        Fr xn = c.valid ? tab_load_fr(a.fr, a.stride, c.in_slot, c.i) : fr_zero();
        Fr pn = (c.valid && INV_E > 1) ? tab_load_fr(a.fr, a.stride, cp.out_slot, cp.i) : fr_one();   // prefix of element e - 1
#pragma unroll 1
        for (int e = INV_E - 1; e >= 0; e--) {
            const Fr x = xn, prev = pn; const InvCursor cur = c;
            if (e > 0) {
                c = cp;                                              // element e - 1 ...
                xn = tab_load_fr(a.fr, a.stride, c.in_slot, c.i);    // (an index past the end is clamped to element 0 by the cursor and not used)
                pn = fr_one();
                if (e > 1) { cp = InvCursor(a, first + (uint64_t)(e - 2) * BLOCK, total); pn = tab_load_fr(a.fr, a.stride, cp.out_slot, cp.i); }   // ... and its prefix
            }
            if (cur.valid) {
                Fr z = fr_zero();
                if (!fr_is_zero(x)) { z = fr_mul(ig, prev); ig = fr_mul(ig, x); }
                tab_store_fr(a.fr, a.stride, cur.out_slot, cur.i, z);
                if constexpr (!PLAIN) Hook::post(h, cur.i, x, z);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------- gate check
struct SmemPool {
    const uint32_t* p;
    const uint32_t* kq = nullptr;              // k*q for k = 0..15, 12 words apart (k_check: the row-end test compares instead of multiplying)
    __device__ __forceinline__ Fr operator()(uint32_t idx) const {
        const uint4 lo = *reinterpret_cast<const uint4*>(p + 8 * idx), hi = *reinterpret_cast<const uint4*>(p + 8 * idx + 4);
        Fr r = {{lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w}};
        return r;
    }
};

// One instance per thread; the row template is walked by all threads in lock step (selector pool in shared memory,
// template rows read with warp-uniform addresses), wire values come from the SoA variable table with coalesced loads.
// Launch shapes of the gate-check kernel: threads per block x minimum blocks per SM (=> register budget, warps per SM).
// pg_cfg.reserved selects one (0 = default); the alternatives are kept for tuning runs (profiles/README.md).
template <int SHAPE> struct CheckShape;
template <> struct CheckShape<0> { static constexpr int BLOCK_T = 128, MIN_BLOCKS = 5; };   // <=102 regs, 20 warps/SM
template <> struct CheckShape<1> { static constexpr int BLOCK_T = 256, MIN_BLOCKS = 2; };   // <=128 regs, 16 warps/SM
template <> struct CheckShape<2> { static constexpr int BLOCK_T = 128, MIN_BLOCKS = 6; };   // <= 85 regs, 24 warps/SM
template <> struct CheckShape<3> { static constexpr int BLOCK_T = 128, MIN_BLOCKS = 7; };   // <= 73 regs, 28 warps/SM
template <> struct CheckShape<4> { static constexpr int BLOCK_T = 128, MIN_BLOCKS = 8; };   // <= 64 regs, 32 warps/SM
constexpr int CHECK_SHAPES = 5;
template <int MODE, int SHAPE>
__global__ void __launch_bounds__(CheckShape<SHAPE>::BLOCK_T, CheckShape<SHAPE>::MIN_BLOCKS) k_check(const CheckArgs a) {
    constexpr int CHECK_BLOCK = CheckShape<SHAPE>::BLOCK_T;
    extern __shared__ __align__(16) uint32_t s_pool[];
    __shared__ uint32_t s_q[8];
    for (uint32_t t = threadIdx.x; t < a.n_pool * 8; t += CHECK_BLOCK) s_pool[t] = a.pool[t];
    if (threadIdx.x < 8) s_q[threadIdx.x] = c_q[threadIdx.x];
    __shared__ __align__(16) uint32_t s_kq[16 * 12];
    if (threadIdx.x < 16) {
        unsigned long long c = 0;
        for (int j = 0; j < 8; j++) { c += (unsigned long long)c_q[j] * threadIdx.x; s_kq[12 * threadIdx.x + j] = (uint32_t)c; c >>= 32; }
        s_kq[12 * threadIdx.x + 8] = (uint32_t)c;
        s_kq[12 * threadIdx.x + 9] = s_kq[12 * threadIdx.x + 10] = s_kq[12 * threadIdx.x + 11] = 0;
    }
    __syncthreads();
    QRegs q;                                   // modulus limbs in vector registers (see QRegs in fr.cuh)
#pragma unroll
    for (int k = 0; k < 8; k++) q.v[k] = s_q[k];
    const uint64_t i = (uint64_t)blockIdx.x * CHECK_BLOCK + threadIdx.x;
    unsigned long long first_bad = ~0ull;
    uint32_t bad = 0;
    if (i < a.n_inst) {
        SmemPool pool = {s_pool, s_kq};
        bad = CheckBody::run<MODE, 65536 / (CHECK_BLOCK * CheckShape<SHAPE>::MIN_BLOCKS) >= 96>(a, pool, q, i, first_bad);   // FOLD: >= 96 registers
    }
    // warp-level reduction, then one atomic per warp that saw a violation
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, first_bad, o);
        first_bad = other < first_bad ? other : first_bad;
    }
    if ((threadIdx.x & 31) == 0 && bad) {
        atomicAdd(a.counters + CNT_UNSAT, (unsigned long long)bad);
        atomicMin(a.counters + CNT_FIRST_BAD, first_bad);
    }
}

// The structure-aware check as a compiled row program (layout.h SpOp, bodies.cuh SparseProgBody); same skeleton as k_check.
// DEPTH: loads in flight per thread inside a chain (register budget: 8 registers per load).
struct SmemQ {
    const uint32_t* p;
    __device__ __forceinline__ QRegs operator()() const { QRegs q;
#pragma unroll
        for (int k = 0; k < 8; k++) q.v[k] = p[k];
        return q; }
};
template <int SHAPE> struct ProgDepth { static constexpr int D = 4; };
template <> struct ProgDepth<0> { static constexpr int D = 3; };     // 102 registers: no spill at all with three loads in flight
template <> struct ProgDepth<3> { static constexpr int D = 2; };
template <> struct ProgDepth<4> { static constexpr int D = 2; };
template <int SHAPE>
__global__ void __launch_bounds__(CheckShape<SHAPE>::BLOCK_T, CheckShape<SHAPE>::MIN_BLOCKS) k_check_prog(const CheckProgArgs args) {
    const CheckArgs& a = args.a; const SparseProg& prog = args.prog;
    constexpr int CHECK_BLOCK = CheckShape<SHAPE>::BLOCK_T;
    extern __shared__ __align__(16) uint32_t s_pool[];
    __shared__ uint32_t s_q[8];
    for (uint32_t t = threadIdx.x; t < a.n_pool * 8; t += CHECK_BLOCK) s_pool[t] = a.pool[t];
    if (threadIdx.x < 8) s_q[threadIdx.x] = c_q[threadIdx.x];
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * CHECK_BLOCK + threadIdx.x;
    unsigned long long first_bad = ~0ull;
    uint32_t bad = 0;
    if (i < a.n_inst) {
        SmemPool pool = {s_pool};
        SmemQ qs = {s_q};
        bad = SparseProgBody::run<ProgDepth<SHAPE>::D>(a, prog, pool, qs, i, first_bad);     // (segments without a program are launched as k_check<1>)
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, first_bad, o);
        first_bad = other < first_bad ? other : first_bad;
    }
    if ((threadIdx.x & 31) == 0 && bad) {
        atomicAdd(a.counters + CNT_UNSAT, (unsigned long long)bad);
        atomicMin(a.counters + CNT_FIRST_BAD, first_bad);
    }
}

// Row-parallel mapping of the same check (thread = one row of one instance) for segments whose instance count cannot fill
// the chip: a single range_check call (n = 1) is then 271 threads instead of one thread walking 271 rows.
template <int MODE>
__global__ void __launch_bounds__(128, 5) k_check_rowpar(const CheckArgs a) {
    extern __shared__ __align__(16) uint32_t s_pool[];
    __shared__ uint32_t s_q[8];
    for (uint32_t t = threadIdx.x; t < a.n_pool * 8; t += 128) s_pool[t] = a.pool[t];
    if (threadIdx.x < 8) s_q[threadIdx.x] = c_q[threadIdx.x];
    __syncthreads();
    QRegs q;
#pragma unroll
    for (int k = 0; k < 8; k++) q.v[k] = s_q[k];
    const uint64_t t = (uint64_t)blockIdx.x * 128 + threadIdx.x;
    unsigned long long first_bad = ~0ull;
    uint32_t bad = 0;
    if (t < a.n_inst * a.n_rows) { SmemPool pool = {s_pool}; bad = CheckBody::run_one<MODE>(a, pool, q, t, first_bad); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, first_bad, o);
        first_bad = other < first_bad ? other : first_bad;
    }
    if ((threadIdx.x & 31) == 0 && bad) {
        atomicAdd(a.counters + CNT_UNSAT, (unsigned long long)bad);
        atomicMin(a.counters + CNT_FIRST_BAD, first_bad);
    }
}

// Segments with rows of the range widget (bodies.cuh GateRowsCheckBody): thread = one row of one instance, lanes = instances.
// MINB: blocks per SM (5 -> 96 registers, 20 warps/SM; 6 -> 80 registers, 24 warps/SM; 7 -> 72 registers, 28 warps/SM).
template <int MINB>
__global__ void __launch_bounds__(128, MINB) k_check_gates(const CheckArgs a) {
    extern __shared__ __align__(16) uint32_t s_pool[];
    __shared__ uint32_t s_q[8];
    for (uint32_t t = threadIdx.x; t < a.n_pool * 8; t += 128) s_pool[t] = a.pool[t];
    if (threadIdx.x < 8) s_q[threadIdx.x] = c_q[threadIdx.x];
    __syncthreads();
    QRegs q;
#pragma unroll
    for (int k = 0; k < 8; k++) q.v[k] = s_q[k];
    const uint64_t t = (uint64_t)blockIdx.x * 128 + threadIdx.x;
    unsigned long long first_bad = ~0ull;
    uint32_t bad = 0;
    if (t < a.n_inst * a.n_rows) { SmemPool pool = {s_pool}; bad = GateRowsCheckBody::run_one(a, pool, q, t, first_bad); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, first_bad, o);
        first_bad = other < first_bad ? other : first_bad;
    }
    if ((threadIdx.x & 31) == 0 && bad) {
        atomicAdd(a.counters + CNT_UNSAT, (unsigned long long)bad);
        atomicMin(a.counters + CNT_FIRST_BAD, first_bad);
    }
}

// The same segments with one thread per instance walking the rows (GateRowsCheckBody::run): large segments.
__global__ void __launch_bounds__(128, 5) k_check_gates_walk(const CheckArgs a) {
    extern __shared__ __align__(16) uint32_t s_pool[];
    __shared__ uint32_t s_q[8];
    for (uint32_t t = threadIdx.x; t < a.n_pool * 8; t += 128) s_pool[t] = a.pool[t];
    if (threadIdx.x < 8) s_q[threadIdx.x] = c_q[threadIdx.x];
    __syncthreads();
    QRegs q;
#pragma unroll
    for (int k = 0; k < 8; k++) q.v[k] = s_q[k];
    const uint64_t i = (uint64_t)blockIdx.x * 128 + threadIdx.x;
    unsigned long long first_bad = ~0ull;
    uint32_t bad = 0;
    if (i < a.n_inst) { SmemPool pool = {s_pool}; bad = GateRowsCheckBody::run(a, pool, q, i, first_bad); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, first_bad, o);
        first_bad = other < first_bad ? other : first_bad;
    }
    if ((threadIdx.x & 31) == 0 && bad) {
        atomicAdd(a.counters + CNT_UNSAT, (unsigned long long)bad);
        atomicMin(a.counters + CNT_FIRST_BAD, first_bad);
    }
}

__global__ void __launch_bounds__(BLOCK) k_check_rows(const CheckRowsBody::Args a) {
    const uint64_t i = (uint64_t)blockIdx.x * BLOCK + threadIdx.x;
    uint32_t bad = i < a.n ? CheckRowsBody::run(a, i) : 0u;
    unsigned long long first_bad = bad ? (unsigned long long)i : ~0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, first_bad, o);
        first_bad = other < first_bad ? other : first_bad;
    }
    if ((threadIdx.x & 31) == 0 && bad) {
        atomicAdd(a.counters + CNT_UNSAT, (unsigned long long)bad);
        atomicMin(a.counters + CNT_FIRST_BAD, first_bad);
    }
}

// ---------------------------------------------------------------------------------------------------- tiled materialisation
// Wire values and selector columns of whole instances in the reference composer's row order (pure HBM streaming).
// A block owns a tile of 32 instances x 32 template rows.
//   wire values: read with lanes = instances (one slot of the SoA table -> 512 contiguous bytes per half), transposed through
//                padded shared memory, written with lanes = rows (the 32 rows of one instance are 1 KiB contiguous in every
//                output column) -- both sides fully coalesced 128-bit accesses;
//   selectors  : instance-independent.  The tile's 32 x 32 B selector values are staged once in shared memory and replicated
//                into the 32 instances' output runs with TMA bulk copies (cp.async.bulk shared -> global, 1 KiB each): no
//                register traffic at all for 5/11 of the bytes written.
constexpr int MT_I = 32, MT_R = 32;                  // instances x rows per tile
constexpr int MT_PITCH = MT_I * 2 + 1;               // uint4 per staged row (+1: conflict-free transposed reads)
__global__ void __launch_bounds__(BLOCK) k_materialize_tiled(const MatTileArgs a) {
    __shared__ __align__(128) uint4 s_val[MT_R * MT_PITCH];          // [row][instance][half]
    __shared__ __align__(128) uint4 s_sel[5][MT_R * 2];              // [selector][row][half]
    const DevSeg& s = a.seg;
    const uint32_t tiles_r = (s.n_rows + MT_R - 1) / MT_R;
    const uint64_t ti = blockIdx.x / tiles_r; const uint32_t tr = blockIdx.x % tiles_r;
    const uint64_t i_lo = a.inst0 + ti * MT_I;                        // first instance of the tile
    const uint32_t r_lo = tr * MT_R;
    const uint32_t n_i = (uint32_t)min((uint64_t)MT_I, a.inst0 + a.n_inst - i_lo), n_r = min((uint32_t)MT_R, s.n_rows - r_lo);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // output column offset of (instance i_lo + ii, row r_lo + rr):
    const uint64_t o_base = a.out_off + (i_lo - a.inst0) * (uint64_t)s.n_rows + r_lo;

    if (a.sel) {                                                      // stage the tile's selector values: 5 x n_r scalars
        for (uint32_t t = threadIdx.x; t < 5 * n_r; t += BLOCK) {
            const uint32_t k = t / n_r, rr = t % n_r;
            const Fr v = pool_load(s.pool, s.rows[r_lo + rr].sel[k]);
            s_sel[k][2 * rr] = make_uint4(v.v[0], v.v[1], v.v[2], v.v[3]); s_sel[k][2 * rr + 1] = make_uint4(v.v[4], v.v[5], v.v[6], v.v[7]);
        }
    }
    for (int w = 0; w < 4; w++) {
        if (a.w_val) {
            __syncthreads();                                          // previous transposed reads of s_val are done
            for (uint32_t rr = warp; rr < n_r; rr += NWARPS) {        // lanes = instances
                if ((uint32_t)lane < n_i) {
                    const Fr v = loc_load(s.tab, s.rows[r_lo + rr].loc[w], i_lo + lane);
                    s_val[rr * MT_PITCH + 2 * lane] = make_uint4(v.v[0], v.v[1], v.v[2], v.v[3]);
                    s_val[rr * MT_PITCH + 2 * lane + 1] = make_uint4(v.v[4], v.v[5], v.v[6], v.v[7]);
                }
            }
            __syncthreads();
            for (uint32_t ii = warp; ii < n_i; ii += NWARPS) {        // lanes = rows: 1 KiB contiguous per instance
                if ((uint32_t)lane < n_r) {
                    const uint4 lo = s_val[lane * MT_PITCH + 2 * ii], hi = s_val[lane * MT_PITCH + 2 * ii + 1];
                    const Fr v = {{lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w}};
                    st256(a.w_val + 2 * ((uint64_t)w * a.stride + o_base + (uint64_t)ii * s.n_rows + lane), v);   // one full sector per lane
                }
            }
        }
    }
    if (a.sel) {
        __syncthreads();                                              // s_sel complete
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // make the generic-proxy smem writes visible to the bulk-copy engine
        // 5 selector columns x n_i instances: one bulk copy of n_r*32 bytes each, issued by distinct threads
        for (uint32_t t = threadIdx.x; t < 5 * n_i; t += BLOCK) {
            const uint32_t k = t / n_i, ii = t % n_i;
            uint4* dst = a.sel + 2 * ((uint64_t)k * a.stride + o_base + (uint64_t)ii * s.n_rows);
            const uint32_t src = (uint32_t)__cvta_generic_to_shared(&s_sel[k][0]);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(n_r * 32u) : "memory");
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");     // smem may be released only after the engine has read it
    }
}

// ---------------------------------------------------------------------------------------------------- pipe micro-benchmarks
// Roofline denominators and instruction-cost evidence, measured on the device the engine runs on.  Every chain feeds its
// own previous result back into a multiplier/adder INPUT, so ptxas can neither hoist, share nor re-associate the
// operations; 8 independent chains per thread and 8 blocks per SM hide the dependent-issue latency.
//   0 IMAD (32-bit lo, accumulate)         acc = acc*b + c
//   1 IMAD.WIDE.U32, no addend              p   = hi(p)*b            (64-bit product only)
//   2 IMAD.WIDE.U32, 64-bit accumulate      acc = lo(acc)*b + acc
//   3 IMAD.HI.U32, accumulate               acc = hi(acc*b) + c
//   4 mad.lo.cc/madc.hi.cc rows             the carry-chain rows of fr_mul (IMAD.WIDE.U32.X): 4 products per row
//   5 IADD3 (3-input add)                   acc = acc + b + c
//   6 Fr Montgomery multiplication          acc = fr_mul(acc, b)     (even/odd carry-chain multiplier)
//   7 Fr Montgomery multiplication          acc = fr_mul_cios(acc, b) (portable 64-bit C)
//   8 Fr addition                           acc = fr_add(acc, b)
//   9 DFMA (fp64 fused multiply-add)        acc = acc*b + c          (the other wide multiplier on the SM, for reference)
//  10 IMAD.WIDE and DFMA interleaved 1:1    do the integer multiplier and the fp64 pipe run concurrently?  (ops = both kinds)
enum { UB_IMAD_LO = 0, UB_WIDE_MUL = 1, UB_WIDE_ACC = 2, UB_IMAD_HI = 3, UB_CARRY_ROWS = 4, UB_IADD3 = 5, UB_FR_MUL = 6, UB_FR_MUL_CIOS = 7, UB_FR_ADD = 8, UB_DFMA = 9, UB_WIDE_DFMA_MIX = 10, UB_MODES = 11 };

template <int MODE>
__global__ void __launch_bounds__(BLOCK) k_ubench(uint32_t* out, uint32_t x, uint32_t y, int iters) {
    const uint32_t tid = blockIdx.x * BLOCK + threadIdx.x;
    uint32_t b = y | 1u, c = x ^ 0x5bd1e995u;
    uint32_t sink = 0;
    if (MODE == UB_IMAD_LO || MODE == UB_IMAD_HI || MODE == UB_IADD3) {
        uint32_t acc[8];
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] = tid * (2 * k + 3) + x;
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int k = 0; k < 8; k++) {
                if (MODE == UB_IMAD_LO) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(acc[k]) : "r"(b), "r"(c));
                if (MODE == UB_IMAD_HI) asm volatile("mad.hi.u32 %0, %0, %1, %2;" : "+r"(acc[k]) : "r"(b), "r"(c));
                if (MODE == UB_IADD3) asm volatile("{ .reg .u32 t; add.u32 t, %0, %1; add.u32 %0, t, %2; }" : "+r"(acc[k]) : "r"(b), "r"(c));
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k++) sink ^= acc[k];
    } else if (MODE == UB_WIDE_MUL || MODE == UB_WIDE_ACC) {
        uint64_t acc[8];
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] = ((uint64_t)(tid * (2 * k + 3) + x) << 32) | (tid + k);
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int k = 0; k < 8; k++) {
                if (MODE == UB_WIDE_MUL) asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %0; mul.wide.u32 %0, hi, %1; }" : "+l"(acc[k]) : "r"(b));
                if (MODE == UB_WIDE_ACC) asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %0; mad.wide.u32 %0, lo, %1, %0; }" : "+l"(acc[k]) : "r"(b));
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k++) sink ^= (uint32_t)acc[k] ^ (uint32_t)(acc[k] >> 32);
    } else if (MODE == UB_WIDE_DFMA_MIX) {
        uint64_t acc[4]; double dacc[4]; const double fb = 1.0 + (double)(b & 0xffu) * 1e-9, fc = (double)(c & 0xffu) * 1e-3;
#pragma unroll
        for (int k = 0; k < 4; k++) { acc[k] = ((uint64_t)(tid * (2 * k + 3) + x) << 32) | (tid + k); dacc[k] = (double)(tid + k); }
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                asm volatile("{ .reg .u32 lo, hi; mov.b64 {lo, hi}, %0; mad.wide.u32 %0, lo, %1, %0; }" : "+l"(acc[k]) : "r"(b));
                asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(dacc[k]) : "d"(fb), "d"(fc));
            }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) sink ^= (uint32_t)acc[k] ^ (uint32_t)(acc[k] >> 32) ^ (uint32_t)__double2ll_rn(dacc[k]);
    } else if (MODE == UB_DFMA) {
        double acc[8]; const double fb = 1.0 + (double)(b & 0xffu) * 1e-9, fc = (double)(c & 0xffu) * 1e-3;
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] = (double)(tid + k);
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int k = 0; k < 8; k++) asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(acc[k]) : "d"(fb), "d"(fc));
        }
#pragma unroll
        for (int k = 0; k < 8; k++) sink ^= (uint32_t)__double2ll_rn(acc[k]);
    } else if (MODE == UB_CARRY_ROWS) {
        uint32_t acc[2][8], top[2] = {0, 0};
#pragma unroll
        for (int k = 0; k < 8; k++) { acc[0][k] = tid * (2 * k + 3) + x; acc[1][k] = tid * (2 * k + 5) + y; }
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int r = 0; r < 2; r++) mad_row(acc[r], top[r], b, c, x, y, acc[r][1]);   // multiplier input depends on the chain
        }
#pragma unroll
        for (int k = 0; k < 8; k++) sink ^= acc[0][k] ^ acc[1][k];
        sink ^= top[0] ^ top[1];
    } else {
        Fr acc[2], m;
#pragma unroll
        for (int k = 0; k < 8; k++) { acc[0].v[k] = (tid * (2 * k + 3) + x) & 0x3fffffffu; acc[1].v[k] = (tid * (2 * k + 5) + y) & 0x3fffffffu; m.v[k] = (b * (k + 7)) & 0x3fffffffu; }
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int r = 0; r < 2; r++) {
                if (MODE == UB_FR_MUL) acc[r] = fr_mul(acc[r], m);
                if (MODE == UB_FR_MUL_CIOS) acc[r] = fr_mul_cios(acc[r], m);
                if (MODE == UB_FR_ADD) acc[r] = fr_add(acc[r], m);
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k++) sink ^= acc[0].v[k] ^ acc[1].v[k];
    }
    out[tid] = sink;
}
// operations per thread per loop iteration in each mode
__host__ __device__ constexpr int ubench_ops_per_iter(int mode) { return mode <= UB_IMAD_HI || mode == UB_IADD3 || mode == UB_DFMA || mode == UB_WIDE_DFMA_MIX ? 8 : (mode == UB_CARRY_ROWS ? 8 : 2); }

}  // namespace pg
