// layout.h -- data layout of the device-resident composer (shared by host logic and kernels).
//
// The reference composer (dusk-plonk StandardComposer) keeps, per row, four `Variable`s and eleven selector scalars, and a
// hash map Variable -> BlsScalar.  For n independent instances of one gadget that is n copies of the same row *structure*:
// only the variable values (and, with per-instance bounds, two q_c entries) differ.  The engine therefore stores a
// SEGMENT per batched call:
//
//   * a row TEMPLATE (rows x {4 wire references, 6 selector pool indices, optional per-instance q_c / PI parameter});
//   * a selector POOL (the distinct Fr constants of the template: 0, 1, -1, 2^i, bounds ...);
//   * the per-instance VARIABLE TABLE in structure-of-arrays form, sized n_alloc instances:
//       fr   [slot][n_alloc]        32 B    -- one 32-byte Montgomery scalar per (slot, instance): a warp reading/writing
//                                             slot s touches 1 KiB of contiguous memory with ONE 256-bit access per thread
//                                             (sm_100 LDG/STG.E.ENL2.256: a whole 32-byte sector per lane);
//       bits [plane][word][n_alloc] u32    -- the 256 bit-variables of one decomposition packed as the canonical
//                                             little-endian 256-bit integer (bit b of the plane = Variable B_b);
//       param[slot][n_alloc]        32 B    -- per-instance selector/public-input values (q_c overrides, PI).
//
// Variable numbering is the reference's: Variable id of local variable j of instance i = base_var + i*n_vars + j;
// row id of local row r = base_row + i*n_rows + r (instances are appended one after another by the sequential loop).
#pragma once
#include <stdint.h>
#include "fr.cuh"

namespace pg {

// ---- value locations ------------------------------------------------------------------------------------------------
// 32-bit code: [31:30] kind, [29:27] table (0 = this segment, 1..4 = operand column e-1), [26:0] payload
enum : uint32_t { LOC_ZERO = 0u, LOC_FR = 1u, LOC_BIT = 2u };
PG_HD uint32_t loc_make(uint32_t kind, uint32_t tab, uint32_t payload) { return (kind << 30) | (tab << 27) | payload; }
PG_HD uint32_t loc_kind(uint32_t l) { return l >> 30; }
PG_HD uint32_t loc_tab(uint32_t l) { return (l >> 27) & 7u; }
PG_HD uint32_t loc_payload(uint32_t l) { return l & 0x07ffffffu; }
PG_HD uint32_t loc_with_tab(uint32_t l, uint32_t tab) { return (l & ~(7u << 27)) | (tab << 27); }

constexpr int MAX_TABS = 5;   // own table + up to 4 operand columns

struct DevTab {
    const uint4* fr;          // pre-offset by the operand's first instance (2 uint4 per scalar)
    const uint32_t* bits;
    uint64_t stride;          // n_alloc of the owning segment
    uint64_t var_base;        // Variable id of (instance 0 of this view, local variable 0)
    uint64_t var_stride;      // n_vars of the owning segment
};

struct DevRow {               // 96 bytes
    uint32_t loc[4];          // where the values of w_l, w_r, w_o, w_4 live
    uint32_t var[4];          // local Variable index inside the owning table's segment (unused for LOC_ZERO)
    uint16_t sel[6];          // pool indices: q_m q_l q_r q_o q_4 q_c
    uint16_t pi_sel;          // pool index of a uniform public input (0 = the constant zero = no PI)
    int16_t qc_param;         // >= 0: q_c is param slot qc_param of the instance (sel[5] ignored)
    int16_t pi_param;         // >= 0: PI is param slot pi_param of the instance
    uint16_t gate;            // GATE_ARITH (q_arith = 1), GATE_RANGE (q_range = 1, q_arith = 0) or GATE_NONE (both 0)
    uint16_t fold;            // entry of the segment's fold table that belongs to q_m (fr_mul_folded's eight constants)
    uint16_t bfold[3];        // blocks of the segment's byte-fold table that belong to q_r, q_o, q_4 (generic mode: k_check_tc)
    uint16_t pad[2];
    // pre-resolved device address of instance 0 of each wire value (FR: the 32-byte scalar; BIT: the 32-bit word holding the
    // bit; ZERO: 0).  The gate-check kernel adds i*32 (or i*4) and never touches the table descriptors: no per-row
    // slot*stride products on the multiplier pipe.
    uint64_t addr[4];
};
static_assert(sizeof(DevRow) == 96, "DevRow must stay 96 bytes");

// Which widget's selector is switched on for a row.  The six gadgets of the reference only emit arithmetic rows; dusk-plonk's native
// range_gate (SURVEY.md 8f.4) emits rows with q_range = 1 (every selector of the arithmetic widget 0) and one closing row with
// neither.  Segments that contain such rows are checked by GateRowsCheckBody (bodies.cuh), all others by the k_check kernels.
enum : uint16_t { GATE_ARITH = 0, GATE_RANGE = 1, GATE_NONE = 2 };

// ---- structure-aware row program (PG_CHECK_SPARSE) ----------------------------------------------------------------------
// The rows of a template compiled, once per segment on the host, into a linear list of term operations (bodies.cuh,
// SparseProgBody): what a structure-aware check has to do and nothing else.  `addr` is the pre-resolved instance-0 address of
// the operand, `stride` its size per instance (32: scalar, 4: word of packed bits, 0: no memory operand).
// Flag SP_ROW_END on an operation: the row is complete after it (test the sum, next row).  SP_TRIVIAL: a row whose folded
// polynomial is identically zero (e.g. b*b - b on a packed bit variable): nothing to evaluate, only the row counter moves.
// SP_CHAIN (+ two SP_CHAIN_AUX words): a run of L rows of the shape  sel_j * bit_j + x_j - x_{j+1} = 0  over consecutive scalar slots
// x_0 .. x_L and consecutive packed bits -- the accumulator rows of a bit decomposition (range.rs:146-152) -- found in the compiled
// program by build_sparse_program and executed as one tight loop: x_{j+1} stays in registers as the next row's x_j (one 32-byte load
// per row), four loads in flight per thread, no per-row program fetch.
//   word 0: addr = x_0 of instance 0, stride 32, sel = first index of the L selectors (a contiguous run of the pool), sh = bit position of bit_0
//   word 1: addr = the 32-bit word holding bit_0 (instance 0), stride 4, sel = L, sh = rows per element (trivially-true rows that precede each chain row + 1)
//   word 2: addr = distance in bytes between consecutive scalar slots (n_alloc * 32; bit words are an eighth of that apart), stride 0
enum : uint8_t { SP_END = 0, SP_ADD_FR, SP_SUB_FR, SP_MASK, SP_BITSEL, SP_MUL_SEL_FR, SP_LOAD_FR, SP_MUL_FR, SP_MULSEL_V, SP_ADD_V, SP_ADD_POOL, SP_TRIVIAL,
                 SP_CHAIN, SP_CHAIN_AUX, SP_ROW_END = 0x80 };
constexpr uint32_t SP_CHAIN_MIN = 4;      // shorter runs stay ordinary operations
struct SpOp { uint64_t addr; uint32_t stride; uint16_t sel; uint8_t op; uint8_t sh; };
static_assert(sizeof(SpOp) == 16, "SpOp must stay 16 bytes");

// reserved pool entries
enum : uint16_t { POOL_ZERO = 0, POOL_ONE = 1, POOL_MINUS_ONE = 2 };

// ---- byte-fold blocks (generic gate check on the tensor cores, kernels.cuh k_check_tc) ----------------------------------------
// For a selector s (Montgomery form) F_k = s * 2^(8k) * R^-1 mod q, k = 0..31, so that for any 256-bit wire w with bytes w_k
//     sum_k w_k * F_k == s*w*R^-1 (mod q)      (the Montgomery product fr_mul_eo(s, w) up to a multiple of q).
// As bytes this is [w_0 .. w_31] x B with B[k][j] = byte j of F_k: a dense 32 x 32 u8 matrix, the B operand of the int8 MMA.  The
// block is stored as the MMA reads it from shared memory: K-major, no swizzle, core matrices of 8 rows (j) x 16 bytes (k).  With
// the core matrices of one 16-byte K chunk stacked along j, element (j, k) sits at (k / 16) * BF_LBO + j * 16 + k % 16.
constexpr uint32_t BF_BYTES = 1024;       // one block
constexpr uint32_t BF_LBO = 512;          // leading-dimension byte offset: from one 16-byte K chunk to the next
constexpr uint32_t BF_SBO = 128;          // stride-dimension byte offset: from rows j..j+7 to rows j+8..j+15
PG_HD uint32_t bf_offset(uint32_t j, uint32_t k) { return (k >> 4) * BF_LBO + j * 16 + (k & 15); }
// the block of selector s (host: template building)
inline void byte_fold_block(uint8_t* blk, const Fr& s) {
    for (uint32_t k = 0; k < 32; k++) {
        Fr p = {{0, 0, 0, 0, 0, 0, 0, 0}};
        p.v[k >> 2] = 1u << (8 * (k & 3));                                  // 2^(8k), a plain value below q
        const Fr f = fr_mul_cios(s, p);                                     // s * 2^(8k) * R^-1 mod q
        for (uint32_t j = 0; j < 32; j++) blk[bf_offset(j, k)] = (uint8_t)(f.v[j >> 2] >> (8 * (j & 3)));
    }
}

// ---- 256-bit accesses -------------------------------------------------------------------------------------------------
// A scalar is exactly one 32-byte DRAM sector.  sm_100 has 256-bit global loads/stores (ld/st.global.v8.b32 ->
// LDG/STG.E.ENL2.256); with two 128-bit accesses per scalar every warp instruction would touch only half of each sector.
// Pointers are kept as uint4* (16-byte units); addresses passed here are 32-byte aligned.
PG_HD Fr ld256(const uint4* p) {
    Fr r;
#if defined(__CUDA_ARCH__)
    asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7]) : "l"(p));
#else
    const uint4 lo = p[0], hi = p[1];
    r.v[0] = lo.x; r.v[1] = lo.y; r.v[2] = lo.z; r.v[3] = lo.w; r.v[4] = hi.x; r.v[5] = hi.y; r.v[6] = hi.z; r.v[7] = hi.w;
#endif
    return r;
}
PG_HD void st256(uint4* p, const Fr& v) {
#if defined(__CUDA_ARCH__)
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"l"(p), "r"(v.v[0]), "r"(v.v[1]), "r"(v.v[2]), "r"(v.v[3]), "r"(v.v[4]), "r"(v.v[5]), "r"(v.v[6]), "r"(v.v[7]) : "memory");
#else
    p[0] = make_uint4(v.v[0], v.v[1], v.v[2], v.v[3]); p[1] = make_uint4(v.v[4], v.v[5], v.v[6], v.v[7]);
#endif
}

// ---- table accessors ------------------------------------------------------------------------------------------------
PG_HD Fr tab_load_fr(const uint4* base, uint64_t stride, uint32_t slot, uint64_t i) { return ld256(base + 2 * ((uint64_t)slot * stride + i)); }
PG_HD void tab_store_fr(uint4* base, uint64_t stride, uint32_t slot, uint64_t i, const Fr& v) { st256(base + 2 * ((uint64_t)slot * stride + i), v); }
PG_HD uint32_t tab_load_bit(const uint32_t* bits, uint64_t stride, uint32_t plane_bit, uint64_t i) {
    const uint32_t plane = plane_bit >> 8, bit = plane_bit & 255u;
    const uint32_t w = (bits + i)[(uint64_t)(plane * 8 + (bit >> 5)) * stride];
    return (w >> (bit & 31u)) & 1u;
}
// value of a located variable for instance i
PG_HD Fr loc_load(const DevTab* tabs, uint32_t loc, uint64_t i) {
    const uint32_t kind = loc_kind(loc);
    if (kind == LOC_ZERO) return fr_zero();
    const DevTab& t = tabs[loc_tab(loc)];
    if (kind == LOC_FR) return tab_load_fr(t.fr, t.stride, loc_payload(loc), i);
    const uint32_t b = tab_load_bit(t.bits, t.stride, loc_payload(loc), i);
    const Fr one = fr_one();
    Fr r;
#pragma unroll
    for (int k = 0; k < 8; k++) r.v[k] = b ? one.v[k] : 0u;
    return r;
}
#if defined(__CUDACC__)
__device__ __align__(32) const uint4 g_zero_fr[2] = {};      // the zero variable's value as a loadable scalar (row_load)
#endif
// the same through the pre-resolved addresses of a DevRow
PG_HD Fr row_load(const DevRow& row, int w, uint64_t i) {
    const uint32_t kind = loc_kind(row.loc[w]);
#if defined(__CUDA_ARCH__)
    // the zero variable's wire is a load too (one 32-byte broadcast out of L1): eight register initialisations per zero wire, half of
    // which ptxas puts on the multiplier pipe, cost the generic check 1.7 ms of 261 (run r05e)
    if (kind != LOC_BIT) return ld256(kind == LOC_FR ? reinterpret_cast<const uint4*>(row.addr[w]) + 2 * i : g_zero_fr);
#endif
    if (kind == LOC_ZERO) return fr_zero();
    if (kind == LOC_FR) return ld256(reinterpret_cast<const uint4*>(row.addr[w]) + 2 * i);
    const uint32_t word = reinterpret_cast<const uint32_t*>(row.addr[w])[i];
    const uint32_t b = (word >> (row.loc[w] & 31u)) & 1u;
    const Fr one = fr_one();
    Fr r;
#pragma unroll
    for (int k = 0; k < 8; k++) r.v[k] = b ? one.v[k] : 0u;
    return r;
}
PG_HD void row_prefetch(uint32_t loc, uint64_t addr, uint64_t i) {
#if defined(__CUDA_ARCH__)
    const uint32_t kind = loc_kind(loc);
    if (kind == LOC_FR) asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const uint4*>(addr) + 2 * i));
    else if (kind == LOC_BIT) asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const uint32_t*>(addr) + i));
#else
    (void)loc; (void)addr; (void)i;
#endif
}
// request the cache lines a later loc_load(tabs, loc, i) will touch (no destination registers)
PG_HD void loc_prefetch(const DevTab* tabs, uint32_t loc, uint64_t i) {
#if defined(__CUDA_ARCH__)
    const uint32_t kind = loc_kind(loc);
    if (kind == LOC_ZERO) return;
    const DevTab& t = tabs[loc_tab(loc)];
    if (kind == LOC_FR) {
        const uint32_t slot = loc_payload(loc);
        asm volatile("prefetch.global.L1 [%0];" ::"l"(t.fr + 2 * ((uint64_t)slot * t.stride + i)));
    } else {
        const uint32_t pb = loc_payload(loc);
        asm volatile("prefetch.global.L1 [%0];" ::"l"((t.bits + i) + (uint64_t)((pb >> 8) * 8 + ((pb & 255u) >> 5)) * t.stride));
    }
#else
    (void)tabs; (void)loc; (void)i;
#endif
}
// AoS scalar (caller memory: BlsScalar[n]) access
PG_HD Fr aos_load(const uint4* p, uint64_t i) { return ld256(p + 2 * i); }
PG_HD void aos_store(uint4* p, uint64_t i, const Fr& v) { st256(p + 2 * i, v); }
PG_HD Fr pool_load(const uint32_t* pool, uint32_t idx) {
    Fr r;
#pragma unroll
    for (int k = 0; k < 8; k++) r.v[k] = pool[8 * idx + k];
    return r;
}

}  // namespace pg
