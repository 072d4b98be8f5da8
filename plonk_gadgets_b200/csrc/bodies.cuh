// bodies.cuh -- per-instance kernel bodies ("one gadget instance per thread").
//
// Every body is a plain __host__ __device__ function of (arguments, instance index).  The CUDA backend (kernels.cuh)
// wraps them in __global__ kernels; the test-only host backend (tests/emu) calls them in a loop so that templates,
// numbering and witness arithmetic can be checked on a machine without a GPU.  Gadgets that need a field inversion are
// split in a Pre body (everything up to the value to invert, written to its table slot), the stand-alone batch-inversion
// kernel over those slots (kernels.cuh: Montgomery's trick, 8 elements per thread, one Fermat inversion per 2048
// elements) and a Post body.
//
// Reference functions restated here (witness arithmetic only; row structure lives in templates.hpp):
//   RangePre/Post   /root/reference/src/range.rs:27-43 (range_check), :82-113 (max_bound), :53-76 (min_bound),
//                   :119-158 (scalar_decomposition_gadget), :161-170 (scalar_to_bits)
//   MaybeEqualFused    /root/reference/src/scalar.rs:105-140   IsNonZeroFused /root/reference/src/scalar.rs:63-97
//   SelectZeroBody  /root/reference/src/scalar.rs:21-27        SelectOneBody  /root/reference/src/scalar.rs:36-59
#pragma once
#include "layout.h"
#include "ntt.cuh"

namespace pg {

// 2^i * R mod q for i in 0..255 (Montgomery form of the q_l selectors / accumulator increments of range.rs:146-152)
#if defined(__CUDACC__)
__constant__ Fr c_pow2[256];
#endif
extern Fr h_pow2[256];
PG_HD const Fr& pow2_entry(uint32_t i) {
#if defined(__CUDA_ARCH__)
    return c_pow2[i];
#else
    return h_pow2[i];
#endif
}

// counters shared by all kernels of a ctx (device memory, 8 x u64)
// words 0..CNT_STICKY-1 are re-initialised before every use (Engine::reset_counters); CNT_BAD_INPUT / CNT_FIRST_BAD_INPUT are
// sticky until the composer is reset: every kernel that ingests caller scalars counts the ones that are not fully reduced (>= q)
// there, and the next call that reads the counters reports PG_ERR_ARG (include/pg_b200.h, "Scalars").
// CNT_FUSED_*: verdict of the rows that were evaluated inside witness generation (PG_F_FUSED_CHECK), added in by pg_check.
enum { CNT_UNSAT = 0, CNT_FIRST_BAD = 1, CNT_MIXED_BITS = 2, CNT_N_ERR = 3, CNT_FIRST_ERR = 4, CNT_STICKY = 5,
       CNT_BAD_INPUT = 5, CNT_FIRST_BAD_INPUT = 6, CNT_FUSED_UNSAT = 7, CNT_FUSED_FIRST = 8, CNT_WORDS = 12 };

// rows [local_base, local_end) of a segment verified inside witness generation, and the index its first row has in the numbering asked for
struct FusedSpan { unsigned long long local_base, local_end, global_base; };

PG_HD void counter_add(unsigned long long* c, unsigned long long v) {
#if defined(__CUDA_ARCH__)
    atomicAdd(c, v);
#else
    *c += v;
#endif
}
PG_HD void counter_min(unsigned long long* c, unsigned long long v) {
#if defined(__CUDA_ARCH__)
    atomicMin(c, v);
#else
    if (v < *c) *c = v;
#endif
}

// ingest check: a caller scalar must be the fully reduced Montgomery form (< q) -- dusk-bls12_381's Scalar always is.  An
// unreduced value would break invariants the kernels rely on (a table value equal to q is "non-zero" with a zero Montgomery
// product; the structure-aware check's 7q headroom), so it is counted here and reported as PG_ERR_ARG by the engine.
PG_HD bool fr_is_reduced(const Fr& a) {
    const uint32_t q[8] = {PG_Q0, PG_Q1, PG_Q2, PG_Q3, PG_Q4, PG_Q5, PG_Q6, PG_Q7};
    uint32_t d[8];
    return fr_sub_limbs(d, a.v, q) != 0;              // a - q borrows  <=>  a < q
}
PG_HD void count_unreduced(unsigned long long* counters, const Fr& a, uint64_t index) {
    if (!fr_is_reduced(a)) { counter_add(counters + CNT_BAD_INPUT, 1ull); counter_min(counters + CNT_FIRST_BAD_INPUT, (unsigned long long)index); }
}

// bit length of a canonical (non-Montgomery) 256-bit integer
PG_HD uint32_t limbs_bitlen(const Fr& c) {
    uint32_t n = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        if (c.v[i]) {
#if defined(__CUDA_ARCH__)
            n = 32u * i + (32u - __clz(c.v[i]));
#else
            n = 32u * i + (32u - (uint32_t)__builtin_clz(c.v[i]));
#endif
        }
    }
    return n;
}
// num_bits_closest_power_of_two(max-1): bits_count(2^bits_count(s) mod q)  -- range.rs:173-189.
// bits_count(s) = max(1, bitlen(s)); for n <= 254, 2^n < q so the result is n + 1; n = 255 cannot happen for s < q
// (q < 2^255), the table value below covers it anyway: bitlen(2^255 mod q) = 252.
PG_HD uint32_t num_bits_from_canonical(const Fr& c) {
    uint32_t n = limbs_bitlen(c);
    if (n < 1) n = 1;
    return n <= 254 ? n + 1 : 252;
}

// ---------------------------------------------------------------------------------------------------- add_input
struct AddInputBody {
    struct Args { const uint4* src; uint4* fr; uint64_t stride; uint64_t n; };
    PG_HD static void run(const Args& a, uint64_t i) { tab_store_fr(a.fr, a.stride, 0, i, aos_load(a.src, i)); }
};

// scalars [i0, i0 + n) of a caller batch (already in device memory) are fully reduced, or counted as bad input
struct ValidateBody {
    struct Args { const uint4* src; uint64_t i0; uint64_t n; unsigned long long* counters; };
    PG_HD static void run(const Args& a, uint64_t i) { count_unreduced(a.counters, aos_load(a.src, a.i0 + i), a.i0 + i); }
};

// ---------------------------------------------------------------------------------------------------- range gadgets
struct DecompSlots { uint32_t v, a0, u, z, y, plane; };   // a0..a0+k are the accumulators A_0..A_k

struct RangeArgs {
    DevTab x_tab; uint32_t x_loc;
    uint4* fr; uint32_t* bits; uint4* param; uint64_t stride;
    uint64_t n; uint32_t k;
    uint64_t i0;                                     // first instance of this launch (chunked launches behind input copies)
    int uniform; Fr m; Fr negmin;                    // uniform bounds: max-1 and -min
    const uint4* max_aos; const uint4* min_aos;      // per-instance bounds
    uint32_t param_m, param_negmin;
    DecompSlots d[2]; uint32_t slot_o;
    unsigned long long* counters;
    uint64_t base_row; uint32_t n_rows;              // FUSED only: global index of the segment's first row, rows per instance
};

// which table slots the batch inversion reads and writes: out[j] = in[j]^-1 (or 0) for every instance
struct BatchInvArgs { uint4* fr; uint64_t stride; uint64_t n; uint32_t n_pairs; uint32_t in_slot[4]; uint32_t out_slot[4]; uint32_t elems_per_thread; };

// FUSED (PG_F_FUSED_CHECK): the kernels that generate a range gadget's witness also evaluate its rows, on the values they hold in
// registers and with the structure-aware arithmetic of the compiled row program (packed bits are boolean by construction; a row
// x + t - y = 0 is tested as fr_sum_equals(x, t, y)), so the table is written once and not read again for the verdict.  Unsatisfied
// rows are added to the sticky CNT_FUSED_* words; pg_check skips such a segment unless one of its Variables was overwritten since.
// Local row numbers of a decomposition that starts (with its V row) at row r0:  V: r0, A_0: r0+1, boolean / accumulate of bit p:
// r0+2+2p / r0+3+2p, u: r0+2k+2, y: r0+2k+3, y*u: r0+2k+4; the second decomposition of range_check starts at 2k+5, y1*y2 is row 4k+10.
struct FusedVerdict {
    uint32_t bad = 0, first = ~0u;
    PG_HD void row(bool holds, uint32_t r) { if (!holds) { bad++; first = first < r ? first : r; } }
    PG_HD void flush(const RangeArgs& a, uint64_t i) const;
    // rows of instance i start at global row `row0`
    PG_HD void flush_at(unsigned long long* counters, unsigned long long row0) const {
        if (!bad) return;
        counter_add(counters + CNT_FUSED_UNSAT, (unsigned long long)bad);
        counter_min(counters + CNT_FUSED_FIRST, row0 + first);
    }
};
// what the scalar gadgets' kernels need to evaluate their own rows (PG_F_FUSED_CHECK): null counters = not fused
struct FusedSite { unsigned long long* counters; unsigned long long base_row; };
template <bool RANGE, bool FUSED = false>
struct RangePre {
    static constexpr int E = RANGE ? 2 : 1;
    typedef RangeArgs Args;

    // scalar_decomposition_gadget up to (and including) u = acc - v
    PG_HD static void decompose(const Args& a, uint64_t i, const DecompSlots& s, const Fr& v, FusedVerdict& fv, uint32_t r0) {
        tab_store_fr(a.fr, a.stride, s.v, i, v);
        const Fr c = fr_from_mont(v);                                          // to_bytes(): canonical integer, range.rs:163
#pragma unroll
        for (int w = 0; w < 8; w++) a.bits[(uint64_t)(s.plane * 8 + w) * a.stride + i] = c.v[w];   // the 256 bit variables
        Fr acc = fr_zero();
        tab_store_fr(a.fr, a.stride, s.a0, i, acc);                            // A_0 = 0, range.rs:138-141
        if (FUSED) fv.row(fr_is_zero(acc), r0 + 1);                            // constrain_to_constant(A_0, 0)
        for (uint32_t p = 0; p < a.k; p++) {                                   // range.rs:143-153
            const uint32_t bit = (c.v[p >> 5] >> (p & 31u)) & 1u;
            const Fr prev = acc;
            if (bit) acc = fr_add(acc, pow2_entry(p));
            tab_store_fr(a.fr, a.stride, s.a0 + 1 + p, i, acc);
            if (FUSED) {                                                       // 2^p * b_p + A_p - A_{p+1} = 0 (the boolean row holds: packed bit)
                Fr t = pow2_entry(p);
#pragma unroll
                for (int j = 0; j < 8; j++) t.v[j] &= 0u - bit;
                fv.row(fr_sum_equals(prev, t, acc), r0 + 3 + 2 * p);
            }
        }
        const Fr u = fr_sub(acc, v);
        tab_store_fr(a.fr, a.stride, s.u, i, u);                               // maybe_equal: u = a - b, scalar.rs:111-121
        if (FUSED) fv.row(fr_sum_equals(v, u, acc), r0 + 2 * a.k + 2);         // A_k - v - u = 0
    }
    PG_HD static void run(const Args& a, uint64_t i_launch) {
        const uint64_t i = a.i0 + i_launch;
        const Fr x = loc_load(&a.x_tab, a.x_loc, i);
        Fr m = a.m, negmin = a.negmin;
        if (!a.uniform) {
            const Fr mx = aos_load(a.max_aos, i);
            count_unreduced(a.counters, mx, i);
            m = fr_sub(mx, fr_one());                                          // max_range - one, range.rs:87
            tab_store_fr(a.param, a.stride, a.param_m, i, m);
            if (num_bits_from_canonical(fr_from_mont(m)) != a.k) counter_add(a.counters + CNT_MIXED_BITS, 1ull);
            if (RANGE) {
                const Fr mn = aos_load(a.min_aos, i);
                count_unreduced(a.counters, mn, i);
                negmin = fr_neg(mn);                                           // q_c = -min_range, range.rs:62
                tab_store_fr(a.param, a.stride, a.param_negmin, i, negmin);
            }
        }
        FusedVerdict fv;
        const Fr v0 = fr_sub(m, x);
        if (FUSED) fv.row(fr_sum_equals(x, v0, m), 0);                         // -x - v + (max - 1) = 0
        decompose(a, i, a.d[0], v0, fv, 0);                                    // b - x, range.rs:93-102
        if (RANGE) {
            const Fr v1 = fr_add(x, negmin);
            if (FUSED) fv.row(fr_sum_equals(x, negmin, v1), 2 * a.k + 5);      // x - v' - min = 0
            decompose(a, i, a.d[E - 1], v1, fv, 2 * a.k + 5);                  // x - a, range.rs:60-69
        }
        if (FUSED) fv.flush(a, i);
    }
};
template <bool RANGE, bool FUSED = false>
struct RangePost {   // after z = u^-1 (or 0) has been written by the batch inversion (scalar.rs:122-123)
    static constexpr int E = RANGE ? 2 : 1;
    typedef RangeArgs Args;
    PG_HD static void run(const Args& a, uint64_t i_launch) {
        const uint64_t i = a.i0 + i_launch;                                    // (chunked launches: see RangePre)
        Fr y[E];
        FusedVerdict fv;
#pragma unroll
        for (int e = 0; e < E; e++) {
            const Fr u = tab_load_fr(a.fr, a.stride, a.d[e].u, i), z = tab_load_fr(a.fr, a.stride, a.d[e].z, i);
            const Fr zu = fr_mul(z, u);
            y[e] = fr_sub(fr_one(), zu);                                       // y = 1 - z*u, scalar.rs:126
            tab_store_fr(a.fr, a.stride, a.d[e].y, i, y[e]);
            if (FUSED) {
                const uint32_t r0 = e ? 2 * a.k + 5 : 0;
                fv.row(fr_sum_equals(y[e], zu, fr_one()), r0 + 2 * a.k + 3);   // -z*u - y + 1 = 0
                fv.row(fr_is_zero(fr_mul(y[e], u)), r0 + 2 * a.k + 4);         // y*u = 0, scalar.rs:129-138
            }
        }
        if (RANGE) {
            const Fr o = fr_mul(y[0], y[E - 1]);
            tab_store_fr(a.fr, a.stride, a.slot_o, i, o);                      // y1*y2, range.rs:42
            if (FUSED) fv.row(fr_eq(fr_mul(y[0], y[E - 1]), o), 4 * a.k + 10);
        }
        if (FUSED) fv.flush(a, i);
    }
};
PG_HD void FusedVerdict::flush(const RangeArgs& a, uint64_t i) const {
    if (!bad) return;
    counter_add(a.counters + CNT_FUSED_UNSAT, (unsigned long long)bad);
    counter_min(a.counters + CNT_FUSED_FIRST, (unsigned long long)(a.base_row + i * (uint64_t)a.n_rows + first));
}

// ---------------------------------------------------------------------------------------------------- maybe_equal
struct MaybeEqualArgs { DevTab a_tab, b_tab; uint32_t a_loc, b_loc; uint4* fr; uint64_t stride; uint64_t n; FusedSite fused; };
// maybe_equal inside the batch inversion's walks (k_batch_inv<MaybeEqualFused>): u is produced where the first walk would
// load it, y where the second walk has just written z.  in_slot = 0 (u), out_slot = 1 (z).  Rows (3 per instance): a - b - u = 0,
// -z*u - y + 1 = 0, y*u = 0.
struct MaybeEqualFused {
    typedef MaybeEqualArgs Args;
    PG_HD static Fr pre(const Args& a, uint64_t i) {
        const Fr va = loc_load(&a.a_tab, a.a_loc, i), vb = loc_load(&a.b_tab, a.b_loc, i);
        const Fr u = fr_sub(va, vb);                                                                                    // scalar.rs:111-121
        tab_store_fr(a.fr, a.stride, 0, i, u);
        if (a.fused.counters) { FusedVerdict fv; fv.row(fr_sum_equals(vb, u, va), 0); fv.flush_at(a.fused.counters, a.fused.base_row + 3 * i); }
        return u;
    }
    PG_HD static void post(const Args& a, uint64_t i, const Fr& u, const Fr& z) {
        const Fr zu = fr_mul(z, u), y = fr_sub(fr_one(), zu);
        tab_store_fr(a.fr, a.stride, 2, i, y);                                                                          // y, scalar.rs:126
        if (a.fused.counters) {
            FusedVerdict fv;
            fv.row(fr_sum_equals(y, zu, fr_one()), 1);
            fv.row(fr_is_zero(fr_mul(y, u)), 2);                                                                        // scalar.rs:129-138
            fv.flush_at(a.fused.counters, a.fused.base_row + 3 * i);
        }
    }
};
struct InvPlain { struct Args {}; };     // the batch inversion without a fused gadget: table slot in, table slot out

// ---------------------------------------------------------------------------------------------------- is_non_zero
struct IsNonZeroFused {   // inside k_batch_inv's walks (in_slot = 0, out_slot = 1); slots: 0 = var_assigned, 1 = inv, 2 = one
    struct Args { const uint4* assigned; uint4* fr; uint64_t stride; uint64_t n; unsigned long long* counters; uint8_t* flags;
                  DevTab var_tab; uint32_t var_loc; FusedSite fused; };      // var_*: the operand column (read by the fused check only)
    PG_HD static Fr pre(const Args& a, uint64_t i) {
        const Fr va = aos_load(a.assigned, i);
        count_unreduced(a.counters, va, i);
        tab_store_fr(a.fr, a.stride, 0, i, va);                                              // var_assigned, scalar.rs:69
        const bool none = fr_is_zero(va);                                                    // invert() is None, scalar.rs:73-80
        if (none) {
            counter_add(a.counters + CNT_N_ERR, 1ull);
            counter_min(a.counters + CNT_FIRST_ERR, (unsigned long long)i);
        }
        if (a.flags) a.flags[i] = none ? 1 : 0;                                              // per-instance Result (pg_is_non_zero_batch_flags)
        tab_store_fr(a.fr, a.stride, 2, i, fr_one());                                        // one, scalar.rs:83
        if (a.fused.counters) {                                                              // var - var_assigned = 0 (the constant-one row holds)
            FusedVerdict fv; fv.row(fr_eq(loc_load(&a.var_tab, a.var_loc, i), va), 0); fv.flush_at(a.fused.counters, a.fused.base_row + 3 * i);
        }
        return va;
    }
    PG_HD static void post(const Args& a, uint64_t i, const Fr&, const Fr& inv) {            // var*inv - 1 = 0, scalar.rs:84-94
        if (!a.fused.counters) return;
        FusedVerdict fv; fv.row(fr_eq(fr_mul(loc_load(&a.var_tab, a.var_loc, i), inv), fr_one()), 2); fv.flush_at(a.fused.counters, a.fused.base_row + 3 * i);
    }
};

// ---------------------------------------------------------------------------------------------------- selections
struct SelectZeroBody {
    struct Args { DevTab x_tab, s_tab; uint32_t x_loc, s_loc; uint4* fr; uint64_t stride; uint64_t n; FusedSite fused; };
    PG_HD static void run(const Args& a, uint64_t i) {
        const Fr x = loc_load(&a.x_tab, a.x_loc, i), s = loc_load(&a.s_tab, a.s_loc, i);
        const Fr r = fr_mul(x, s);                                                            // scalar.rs:26
        tab_store_fr(a.fr, a.stride, 0, i, r);
        if (a.fused.counters) { FusedVerdict fv; fv.row(fr_eq(fr_mul(x, s), r), 0); fv.flush_at(a.fused.counters, a.fused.base_row + i); }   // x*s - r = 0
    }
};
struct SelectOneBody {
    struct Args { DevTab y_tab, s_tab; uint32_t y_loc, s_loc; uint4* fr; uint64_t stride; uint64_t n; FusedSite fused; };
    PG_HD static void run(const Args& a, uint64_t i) {
        const Fr y = loc_load(&a.y_tab, a.y_loc, i), s = loc_load(&a.s_tab, a.s_loc, i), one = fr_one();
        const Fr sy = fr_mul(y, s);                                                           // scalar.rs:43
        const Fr oms = fr_sub(one, s);                                                        // scalar.rs:45-50
        const Fr r = fr_add(sy, oms);                                                         // scalar.rs:53-58
        tab_store_fr(a.fr, a.stride, 0, i, one);                                              // scalar.rs:41
        tab_store_fr(a.fr, a.stride, 1, i, sy);
        tab_store_fr(a.fr, a.stride, 2, i, oms);
        tab_store_fr(a.fr, a.stride, 3, i, r);
        if (a.fused.counters) {                                   // rows: one = 1 (holds), y*s - sy = 0, one - s - oms = 0, sy + oms - r = 0
            FusedVerdict fv;
            fv.row(fr_eq(fr_mul(y, s), sy), 1);
            fv.row(fr_sum_equals(s, oms, one), 2);
            fv.row(fr_sum_equals(sy, oms, r), 3);
            fv.flush_at(a.fused.counters, a.fused.base_row + 4 * i);
        }
    }
};

// ---------------------------------------------------------------------------------------------------- constrain_to_constant
struct ConstrainBody {   // only launched when the constant and/or the public input is per-instance
    struct Args { const uint4* constant; const uint4* pi; uint4* param; uint64_t stride; uint64_t n; int32_t param_qc, param_pi; unsigned long long* counters; };
    PG_HD static void run(const Args& a, uint64_t i) {
        if (a.param_qc >= 0) {
            const Fr c = aos_load(a.constant, i);
            count_unreduced(a.counters, c, i);
            tab_store_fr(a.param, a.stride, (uint32_t)a.param_qc, i, fr_neg(c));                                          // q_c = -constant
        }
        if (a.param_pi >= 0) {
            const Fr p = aos_load(a.pi, i);
            count_unreduced(a.counters, p, i);
            tab_store_fr(a.param, a.stride, (uint32_t)a.param_pi, i, p);
        }
    }
};

// ---------------------------------------------------------------------------------------------------- range_gate
// Witness side of StandardComposer::range_gate [dusk-plonk 0.8, recalled; SURVEY.md 8f.4, /root/reference/src/range.rs:9-12]: the
// num_bits/2 accumulators a_j = 4*a_{j-1} + quad_j over the base-4 digits of the canonical witness, most significant quad first
// (slot j = allocation order).  Bits of the witness above num_bits never enter: then the last accumulator differs from the witness
// and the closing assert_equal row is what fails.
struct RangeGateBody {
    struct Args { DevTab x_tab; uint32_t x_loc; uint4* fr; uint64_t stride; uint64_t n; uint32_t n_acc; };
    PG_HD static void run(const Args& a, uint64_t i) {
        const Fr c = fr_from_mont(loc_load(&a.x_tab, a.x_loc, i));             // to_bytes(): canonical integer
        const Fr one = fr_one(), two = fr_add(one, one), three = fr_add(two, one);   // BlsScalar::from(quad)
        Fr acc = fr_zero();
#pragma unroll
        for (int limb = 7; limb >= 0; limb--) {                                // limbs by static index: the scalar stays in registers
#pragma unroll 1
            for (int sh = 30; sh >= 0; sh -= 2) {
                const uint32_t bit = 32u * (uint32_t)limb + (uint32_t)sh;      // bit_index = (num_quads - i) << 1, most significant quad first
                if (bit >= 2u * a.n_acc) continue;
                const uint32_t quad = (c.v[limb] >> sh) & 3u;                  // q_0 + 2*q_1 (bit is even: both in one limb)
                acc = fr_add(acc, acc); acc = fr_add(acc, acc);                // four * accumulator
                Fr q;
#pragma unroll
                for (int k = 0; k < 8; k++) q.v[k] = quad == 1u ? one.v[k] : quad == 2u ? two.v[k] : quad == 3u ? three.v[k] : 0u;
                acc = fr_add(acc, q);
                tab_store_fr(a.fr, a.stride, a.n_acc - 1u - (bit >> 1), i, acc);
            }
        }
    }
};

// ---------------------------------------------------------------------------------------------------- gate check
// q_arith*(q_m*a*b + q_l*a + q_r*b + q_o*c + q_4*d + PI + q_c) for every row of every instance of one segment.
struct CheckArgs {
    DevTab tab[MAX_TABS];
    const uint4* param; uint64_t param_stride;
    const DevRow* rows; const uint32_t* pool;
    const Fr* fold;                  // fr_fold_constants of every q_m of the template, 8 per entry (DevRow::fold)
    const uint4* bfold;              // byte_fold_block of every q_r / q_o / q_4 of the template, BF_BYTES each (DevRow::bfold; generic mode)
    uint32_t n_rows, n_pool;
    uint64_t n_inst; uint64_t base_row;
    unsigned long long* counters;
    int mode;
};
// structure-aware row program of a segment (PG_CHECK_SPARSE), passed next to CheckArgs: the generic kernel's argument block and
// code stay exactly as they were measured
struct SparseProg { const SpOp* ops; uint32_t n; };
struct CheckProgArgs { CheckArgs a; SparseProg prog; };      // one argument block for k_check_prog

// GENERIC mode evaluates  a*(q_m*b + q_l) + q_r*b + q_o*c + q_4*d + q_c + PI  -- the gate polynomial with the bilinear term
// factored, five multiplications instead of six, still without looking at any selector value: u = q_m*b through the eight
// constants the host folded from q_m (fr_mul_folded: 64 products and two reduction steps, u < q + 2^227, + q_l without reduction),
// then the four remaining products as ONE dot product with a single interleaved reduction (fr_dot_wide): 64+12 + 4*64+48 = 380
// wide multiplier instructions per row instead of 6*(64+64).  The 9-limb result plus q_c and PI is tested for "0 mod q" directly.
// This is the reference the tests compare against and the body of the small-segment, tuning-shape and range-widget kernels; large
// generic segments run k_check_tc (kernels.cuh), which takes q_r*b + q_o*c + q_4*d to the tensor cores.
// SPARSE mode: structure-aware, see sparse_terms.
struct CheckBody {
    typedef CheckArgs Args;
    // gate equation of row `row` for instance i: true iff it holds
    PG_HD static void masked_add(uint32_t (&t)[9], Fr v, uint32_t mask) {      // t += v & mask
#pragma unroll
        for (int j = 0; j < 8; j++) v.v[j] &= mask;
        add9_fr(t, v);
    }
    // 0 or ~0 according to the bit variable behind wire w
    PG_HD static uint32_t wire_bit_mask(const DevRow& row, int w, uint64_t i) {
        const uint32_t word = reinterpret_cast<const uint32_t*>(row.addr[w])[i];
        return 0u - ((word >> (row.loc[w] & 31u)) & 1u);
    }
    PG_HD static Fr wire_fr(const DevRow& row, int w, uint64_t i) { return ld256(reinterpret_cast<const uint4*>(row.addr[w]) + 2 * i); }

    // Structure-aware evaluation: the same polynomial on the same stored values, but a term costs what its structure needs.
    //  * selector is the constant 0, or the wire is the zero variable: nothing (the value is not even loaded);
    //  * the wire is a packed bit variable (its value is 0 or 1 by construction): selector AND mask, no multiplication;
    //  * selector +-1: addition / subtraction;   * otherwise: one Montgomery multiplication.
    // All decisions are taken on the row template, i.e. they are uniform across the warp.  One multiplier site in a rolled loop.
    template <class PoolT>
    PG_HD static void sparse_terms(uint32_t (&t)[9], const DevRow& row, const PoolT& pool, const QRegs& q, uint64_t i) {
#pragma unroll
        for (int k = 0; k < 9; k++) t[k] = 0;
#pragma unroll 1
        for (int k = 0; k < 5; k++) {
            const uint32_t si = row.sel[k];
            const int w = k ? k - 1 : 0;
            const uint32_t kind = loc_kind(row.loc[w]);
            if (si == POOL_ZERO || kind == LOC_ZERO) continue;
            uint32_t mask = ~0u;                 // product of the bit-valued factors
            bool have_v = false; Fr v = fr_zero();  // product of the scalar-valued factors (so far at most one)
            int n_mul = 0; Fr x = fr_zero();
            if (kind == LOC_BIT) mask = wire_bit_mask(row, w, i); else { v = wire_fr(row, w, i); have_v = true; }
            if (k == 0) {                        // bilinear term: times w_r
                const uint32_t kb = loc_kind(row.loc[1]);
                if (kb == LOC_ZERO) continue;
                if (kb == LOC_BIT) mask &= wire_bit_mask(row, 1, i);
                else if (!have_v) { v = wire_fr(row, 1, i); have_v = true; }
                else { x = wire_fr(row, 1, i); n_mul = 1; }
            }
            const bool general = si != POOL_ONE && si != POOL_MINUS_ONE;
            if (!have_v) {                       // bits only: the term is the selector or nothing
                Fr sv = pool(si);
#pragma unroll
                for (int j = 0; j < 8; j++) sv.v[j] &= mask;
                add9_fr(t, sv);
                continue;
            }
            if (general) { if (n_mul == 0) x = pool(si); n_mul++; }
            for (int p = 0; p < n_mul; p++) { v = fr_mul_eo(x, v, q); x = pool(si); }
            if (si == POOL_MINUS_ONE) v = fr_neg(v);
#pragma unroll
            for (int j = 0; j < 8; j++) v.v[j] &= mask;
            add9_fr(t, v);
        }
    }

    // gate equation of row `row` for instance i: true iff it holds.  FOLD: q_m*b through fr_mul_folded (kernels with a budget of at
    // least 96 registers); otherwise through fr_mul_eo -- the fold constants in flight make the kernels of 64..85 registers and the
    // range-widget kernels spill more than they do
    template <int MODE, bool FOLD = true, class PoolT>
    PG_HD static bool row_holds(const Args& a, const DevRow& row, const PoolT& pool, const QRegs& q, uint64_t i) {
        if (MODE != 0) return row_holds_sparse(a, row, pool, q, i);
        Fr w[5];
#pragma unroll
        for (int k = 0; k < 4; k++) w[k + 1] = row_load(row, k, i);
        uint32_t t[9];
        Fr sel[4];
        const Fr qmb = FOLD ? fr_mul_folded(a.fold + 8 * (uint32_t)row.fold, w[2], q) : fr_mul_eo(pool(row.sel[0]), w[2], q);
        sel[0] = fr_add_noreduce(qmb, pool(row.sel[1]));                                     // q_m*b + q_l  (< 2q + 2^227 < 2^256)
#pragma unroll
        for (int k = 1; k < 4; k++) sel[k] = pool(row.sel[k + 1]);                           // q_r q_o q_4
        fr_dot_wide<4>(t, w + 1, sel, q);                                                     // a*u + b*q_r + c*q_o + d*q_4
        add9_fr(t, row.qc_param >= 0 ? tab_load_fr(a.param, a.param_stride, (uint32_t)row.qc_param, i) : pool(row.sel[5]));
        if (row.pi_param >= 0) add9_fr(t, tab_load_fr(a.param, a.param_stride, (uint32_t)row.pi_param, i));
        else if (row.pi_sel != POOL_ZERO) add9_fr(t, pool(row.pi_sel));
        return pool_is_multiple_of_q(pool, t);
    }
    // t == k*q for k = t[0] <= 15: through the pool's table of multiples when it has one (three 128-bit shared-memory loads instead of
    // eight products), else by multiplying
    template <class PoolT>
    PG_HD static bool pool_is_multiple_of_q(const PoolT& pool, const uint32_t* t) {
#if defined(__CUDA_ARCH__)
        if (pool.kq) {
            const uint32_t k = t[0] < 15u ? t[0] : 15u;
            const uint4* e = reinterpret_cast<const uint4*>(pool.kq + 12 * k);
            const uint4 a0 = e[0], a1 = e[1], a2 = e[2];
            uint32_t diff = (a0.x ^ t[0]) | (a0.y ^ t[1]) | (a0.z ^ t[2]) | (a0.w ^ t[3]) | (a1.x ^ t[4]) | (a1.y ^ t[5]) | (a1.z ^ t[6]) | (a1.w ^ t[7]) | (a2.x ^ t[8]);
            return diff == 0;                  // (t[0] > 15 differs from 15*q's low limb 15)
        }
#endif
        (void)pool;
        return limbs9_is_multiple_of_q(t);
    }
    // the same row through the structure-aware term evaluation (small segments; large ones run the compiled program)
    template <class PoolT>
    PG_HD static bool row_holds_sparse(const Args& a, const DevRow& row, const PoolT& pool, const QRegs& q, uint64_t i) {
        uint32_t t[9];
        sparse_terms(t, row, pool, q, i);
        add9_fr(t, row.qc_param >= 0 ? tab_load_fr(a.param, a.param_stride, (uint32_t)row.qc_param, i) : pool(row.sel[5]));
        if (row.pi_param >= 0) add9_fr(t, tab_load_fr(a.param, a.param_stride, (uint32_t)row.pi_param, i));
        else if (row.pi_sel != POOL_ZERO) add9_fr(t, pool(row.pi_sel));
        return limbs9_is_multiple_of_q(t);
    }
    // evaluates all rows of instance i; returns the number of unsatisfied rows, updates first_bad (global row index)
    template <int MODE, bool FOLD = true, class PoolT>
    PG_HD static uint32_t run(const Args& a, const PoolT& pool, const QRegs& q, uint64_t i, unsigned long long& first_bad) {
        uint32_t bad = 0;
        // (No prefetch of the next row's wires: requesting them into L1 one row ahead -- eight more warp-uniform loads of the next
        // template row, four kind tests and four cache-control instructions per row -- was worth 5 % when it came in with run r01g and
        // costs 2.7 % on the leaner row loop of run r05e: 256.2 -> 249.3 ms, run r05n.  Twenty resident warps per SM hide the loads.)
        for (uint32_t r = 0; r < a.n_rows; r++) {
            const DevRow row = a.rows[r];
            if (!row_holds<MODE, FOLD>(a, row, pool, q, i)) {
                bad++;
                const unsigned long long g = a.base_row + i * (uint64_t)a.n_rows + r;
                if (g < first_bad) first_bad = g;
            }
        }
        return bad;
    }
    // one (instance, row) pair per call: the mapping used for segments too small to fill the GPU with one thread per instance
    template <int MODE, class PoolT>
    PG_HD static uint32_t run_one(const Args& a, const PoolT& pool, const QRegs& q, uint64_t t, unsigned long long& first_bad) {
        const uint64_t i = t / a.n_rows; const uint32_t r = (uint32_t)(t - i * a.n_rows);
        bool ok;
        if (MODE == 0) { const DevRow row = a.rows[r]; ok = row_holds<MODE>(a, row, pool, q, i); }
        else ok = row_holds<MODE>(a, a.rows[r], pool, q, i);
        if (ok) return 0u;
        first_bad = a.base_row + t;
        return 1u;
    }
};

// Structure-aware check as a linear program (layout.h, SpOp): the template's rows compiled on the host into the term operations
// a row needs -- nothing is decided per row on the device, operand addresses are known SP_AHEAD operations ahead (prefetch),
// and a range_check row costs a handful of adds: the check becomes bound by instruction issue and HBM, not by the multiplier.
#ifndef PG_SP_AHEAD
#define PG_SP_AHEAD 12
#endif
#ifndef PG_SP_PREFETCH
#define PG_SP_PREFETCH "prefetch.global.L1 [%0];"
#endif
constexpr uint32_t SP_AHEAD = PG_SP_AHEAD;
// one 128-bit load per operation (the 16-byte SpOp, 16-byte aligned in the segment image) instead of one load per field
PG_HD SpOp sp_fetch(const SpOp* ops, uint32_t j) {
#if defined(__CUDA_ARCH__)
    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(ops) + j);
    SpOp o;
    o.addr = (uint64_t)raw.x | ((uint64_t)raw.y << 32); o.stride = raw.z;
    o.sel = (uint16_t)raw.w; o.op = (uint8_t)(raw.w >> 16); o.sh = (uint8_t)(raw.w >> 24);
    return o;
#else
    return ops[j];
#endif
}
// A row's accumulator starts at 7q instead of 0, so that "- x" terms are plain 9-limb subtractions (x < q, at most 7 terms per row:
// five selector terms, q_c, PI) instead of a modular negation and an addition; the row-end test accepts any k*q with k <= 15
// (7 + at most 7 additions = 14).
PG_HD void sp_row_init(uint32_t* t) {
    t[0] = 0x00000007u; t[1] = 0xfffffff9u; t[2] = 0xfff483f8u; t[3] = 0x4a2f7c14u; t[4] = 0x436ce825u;
    t[5] = 0x6694e838u; t[6] = 0x234e6cf9u; t[7] = 0x2b7f9346u; t[8] = 0x00000003u;
}
struct QDefault { PG_HD QRegs operator()() const { return q_regs_default(); } };
struct SparseProgBody {
    // SP_CHAIN (layout.h): L rows  sel_j * bit_j + x_j - x_{j+1} = 0.  DEPTH loads of x in flight; x_{j+1} is the next row's x_j.
    template <int DEPTH, class PoolT>
    PG_HD static void run_chain(const SpOp& c0, const SpOp& c1, const SpOp& c2, const PoolT& pool, uint64_t i,
                                uint32_t& bad, uint32_t& first_local, uint32_t& r) {
        const uint32_t L = c1.sel, rows_per = c1.sh;
        const uint64_t slot_step = c2.addr >> 4, word_step = c2.addr >> 5;   // in uint4 / u32 units (bit words are an eighth of the distance apart)
        const uint4* px = reinterpret_cast<const uint4*>(c0.addr) + 2 * i;
        const uint32_t* pw = reinterpret_cast<const uint32_t*>(c1.addr) + i;
        uint32_t left = 32u - c0.sh;                                 // bits of the current word not yet consumed
        uint32_t word = *pw >> c0.sh, word_next = 0;
        if (L > left) { pw += word_step; word_next = *pw; }
        Fr prev = ld256(px);
        px += slot_step;                                             // -> x_1
        uint32_t sel = c0.sel, rr = r + rows_per - 1u;               // pool index / local row of the element being tested
#pragma unroll 1
        for (uint32_t j = 0; j < L; j += DEPTH) {
            Fr nx[DEPTH];
#pragma unroll
            for (uint32_t u = 0; u < DEPTH; u++) if (j + u < L) nx[u] = ld256(px + u * slot_step);
            px += DEPTH * slot_step;
#pragma unroll
            for (uint32_t u = 0; u < DEPTH; u++) {
                if (j + u >= L) break;
                const uint32_t m = 0u - (word & 1u);
                word >>= 1;
                if (--left == 0) {                                   // next word (loaded one word ahead)
                    word = word_next; left = 32;
                    if (L - (j + u + 1) > 32u) { pw += word_step; word_next = *pw; }
                }
                Fr t = pool(sel);
#pragma unroll
                for (int k = 0; k < 8; k++) t.v[k] &= m;
                if (!fr_sum_equals(u == 0 ? prev : nx[u ? u - 1 : 0], t, nx[u])) {
                    bad++;
                    first_local = first_local < rr ? first_local : rr;
                }
                sel++; rr += rows_per;
            }
            prev = nx[DEPTH - 1];
        }
        r += L * rows_per;
    }

    // QSrc: where the modulus limbs come from at the (rare) multiplier site -- shared memory on the device, so that they are not
    // eight registers held for the whole kernel
    template <int DEPTH, class PoolT, class QSrc>
    PG_HD static uint32_t run(const CheckArgs& a, const SparseProg& prog, const PoolT& pool, const QSrc& qsrc, uint64_t i, unsigned long long& first_bad) {
        uint32_t t[9];
        sp_row_init(t);
        uint32_t mask = ~0u, bad = 0, r = 0, first_local = ~0u;      // first unsatisfied row of this instance (local index)
        Fr v = fr_zero();                                            // product register of the multiplication chain (a handful of operations per instance use it)
#pragma unroll 1
        for (uint32_t j = 0; j < prog.n; j++) {
            const SpOp op = sp_fetch(prog.ops, j);
#if defined(__CUDA_ARCH__)
            if (j + SP_AHEAD < prog.n) {
                const SpOp nx = sp_fetch(prog.ops, j + SP_AHEAD);
                if (nx.addr && nx.stride) asm volatile(PG_SP_PREFETCH ::"l"(nx.addr + i * nx.stride));
            }
#endif
            const uint32_t code = op.op & 0x7fu;
            if (code == SP_CHAIN) {
                const SpOp c1 = sp_fetch(prog.ops, j + 1), c2 = sp_fetch(prog.ops, j + 2);
                run_chain<DEPTH>(op, c1, c2, pool, i, bad, first_local, r);
                j += 2;
                sp_row_init(t); v = fr_zero(); mask = ~0u;          // a chain starts and ends at a row boundary: nothing is carried across it
                continue;
            }
            if (code <= SP_BITSEL) {                                // the operations range rows are made of: no multiplication, `v` untouched
                switch (code) {
                    case SP_ADD_FR: add9_fr(t, ld256(reinterpret_cast<const uint4*>(op.addr) + 2 * i)); break;
                    case SP_SUB_FR: sub9_fr(t, ld256(reinterpret_cast<const uint4*>(op.addr) + 2 * i)); break;
                    case SP_MASK: mask &= 0u - ((reinterpret_cast<const uint32_t*>(op.addr)[i] >> op.sh) & 1u); break;
                    case SP_BITSEL: {
                        const uint32_t m = mask & (0u - ((reinterpret_cast<const uint32_t*>(op.addr)[i] >> op.sh) & 1u));
                        CheckBody::masked_add(t, pool(op.sel), m); mask = ~0u;
                    } break;
                    default: break;                                 // SP_END: nothing to add
                }
            } else {
                Fr x = fr_zero(), y = fr_zero();
                bool mul = false;
                switch (code) {
                    case SP_MUL_SEL_FR: x = pool(op.sel); y = ld256(reinterpret_cast<const uint4*>(op.addr) + 2 * i); mul = true; break;
                    case SP_LOAD_FR: v = ld256(reinterpret_cast<const uint4*>(op.addr) + 2 * i); break;
                    case SP_MUL_FR: x = v; y = ld256(reinterpret_cast<const uint4*>(op.addr) + 2 * i); mul = true; break;
                    case SP_MULSEL_V: x = pool(op.sel); y = v; mul = true; break;
                    case SP_ADD_V: { CheckBody::masked_add(t, op.sh ? fr_neg(v) : v, mask); mask = ~0u; } break;
                    case SP_ADD_POOL: add9_fr(t, pool(op.sel)); break;
                    case SP_TRIVIAL: r += op.stride; break;         // `stride` consecutive rows that hold for every witness
                    default: break;
                }
                if (mul) {                                          // the one multiplier site
                    const Fr p = fr_mul_eo(x, y, qsrc());
                    if (code == SP_MUL_SEL_FR) add9_fr(t, p); else v = p;
                }
            }
            if ((op.op & SP_ROW_END) || op.op == SP_END) {          // the row is complete
                if (!limbs9_is_multiple_of_q(t)) {
                    bad++;
                    first_local = first_local < r ? first_local : r;
                }
                r++; mask = ~0u;
                sp_row_init(t);
            }
        }
        if (bad) {
            const unsigned long long g = a.base_row + i * (uint64_t)a.n_rows + first_local;
            if (g < first_bad) first_bad = g;
        }
        return bad;
    }
};

// D(hi - 4*lo), D(f) = f(f-1)(f-2)(f-3): zero iff hi - 4*lo is a base-4 digit (range widget of dusk-plonk, recalled)
PG_HD Fr range_delta(const Fr& hi, const Fr& lo) {
    Fr l4 = fr_add(lo, lo); l4 = fr_add(l4, l4);
    const Fr f = fr_sub(hi, l4), one = fr_one();
    Fr g = fr_sub(f, one), p = fr_mul(f, g);
    g = fr_sub(g, one); p = fr_mul(p, g);
    g = fr_sub(g, one); return fr_mul(p, g);
}
PG_HD Fr range_quad_sum(const Fr& a, const Fr& b, const Fr& c, const Fr& d, const Fr& d_next) {
    Fr sum = fr_add(range_delta(c, d), range_delta(b, c));
    sum = fr_add(sum, range_delta(a, b));
    return fr_add(sum, range_delta(d_next, a));
}

// caller-supplied materialised rows (column-major AoS scalars).  q_arith / q_range null: the arithmetic widget alone (q_arith = 1);
// otherwise the full  q_arith*(...) + q_range*(sum of the four D terms), d_next = w_4 of row (i+1) mod n.
struct CheckRowsBody {
    struct Args { const uint4* w; const uint4* sel; const uint4* pi; uint64_t n; unsigned long long* counters; const uint4* q_arith; const uint4* q_range; };
    PG_HD static uint32_t run(const Args& a, uint64_t i) {
        if (a.q_arith || a.q_range) return run_ex(a, i);
        Fr w[5], sel[5];
        w[1] = aos_load(a.w, i); w[2] = aos_load(a.w, a.n + i); w[3] = aos_load(a.w, 2 * a.n + i); w[4] = aos_load(a.w, 3 * a.n + i);
        sel[0] = fr_add_noreduce(fr_mul(aos_load(a.sel, i), w[2]), aos_load(a.sel, a.n + i));         // q_m*b + q_l
#pragma unroll
        for (int k = 1; k < 4; k++) sel[k] = aos_load(a.sel, (uint64_t)(k + 1) * a.n + i);             // q_r q_o q_4
        uint32_t t[9];
        fr_dot_wide<4>(t, w + 1, sel);
        add9_fr(t, aos_load(a.sel, 5 * a.n + i));
        if (a.pi) add9_fr(t, aos_load(a.pi, i));
        return limbs9_is_multiple_of_q(t) ? 0u : 1u;
    }
    PG_HD static uint32_t run_ex(const Args& a, uint64_t i) {
        const Fr wa = aos_load(a.w, i), wb = aos_load(a.w, a.n + i), wc = aos_load(a.w, 2 * a.n + i), wd = aos_load(a.w, 3 * a.n + i);
        Fr t = fr_mul(fr_mul(aos_load(a.sel, i), wa), wb);
        t = fr_add(t, fr_mul(aos_load(a.sel, a.n + i), wa)); t = fr_add(t, fr_mul(aos_load(a.sel, 2 * a.n + i), wb));
        t = fr_add(t, fr_mul(aos_load(a.sel, 3 * a.n + i), wc)); t = fr_add(t, fr_mul(aos_load(a.sel, 4 * a.n + i), wd));
        if (a.pi) t = fr_add(t, aos_load(a.pi, i));
        t = fr_add(t, aos_load(a.sel, 5 * a.n + i));
        if (a.q_arith) t = fr_mul(aos_load(a.q_arith, i), t);
        if (a.q_range) {
            const Fr qr = aos_load(a.q_range, i);
            if (!fr_is_zero(qr)) t = fr_add(t, fr_mul(qr, range_quad_sum(wa, wb, wc, wd, aos_load(a.w, 3 * a.n + (i + 1 == a.n ? 0 : i + 1)))));
        }
        return fr_is_zero(t) ? 0u : 1u;
    }
};

// Segments that hold rows of another widget (GATE_RANGE / GATE_NONE, layout.h): one thread per (row, instance), lanes = instances
// (kernels.cuh k_check_gates).
//   arithmetic rows: the generic kernel's row evaluation (CheckBody::row_holds<0>, with q_m*b through fr_mul_eo);
//   range rows     : q_range*(D(c - 4d) + D(b - 4c) + D(a - 4b) + D(d_next - 4a)), D(f) = f(f-1)(f-2)(f-3), with d_next the fourth
//                    wire of the NEXT row [dusk-plonk check_circuit_satisfied / range widget, recalled].  Evaluated as
//                    D(f) = u^2 - 1, u = f(f-3) + 1  (f(f-3) = g, (f-1)(f-2) = g + 2, g(g+2) = (g+1)^2 - 1): four multiplications,
//                    then sum u_k^2 as ONE dot product with a single interleaved reduction, minus 4 -- 4*(64+48) + 4*64+48 = 752
//                    wide multiplier instructions per row instead of 12 full multiplications; the 9-limb sum is tested for
//                    "0 mod q" directly.  (Writing u as the square (f - 3/2)^2 - 5/4 and squaring with 36 products brings a row
//                    to 528 products and is slower: the additions a squaring needs cost more integer-pipe time than the
//                    products save on the multiplier pipe -- profiles/r05a_range_rows_variants.md.)  Inside a template a
//                    range row is never the last one (range_gate closes with a q_range = 0 gate and assert_equal);
//   rows with neither selector hold trivially.
//   PG_CHECK_SPARSE: arithmetic rows through the structure-aware term evaluation, range rows through the digit test (see below).
struct GateRowsCheckBody {
    // the range widget's term of one row: w = d, c, b, a, d_next (each term is D(w[k+1] - 4*w[k]))
    PG_HD static bool range_row_holds(const Fr* w, const QRegs& q, int mode) {
        // Montgomery forms of the small constants (literals: an fr_add chain here would be recomputed by every thread)
        const Fr one = fr_one();
        const Fr two = {{0xfffffffcu, 0x00000003u, 0x00069004u, 0xb1096ff4u, 0xd9789feau, 0x33189fdfu, 0x598a0adfu, 0x304962b3u}};
        const Fr three = {{0xfffffffau, 0x00000005u, 0x0009d806u, 0x098e27eeu, 0xc634efe0u, 0xcca4efcfu, 0x064f104eu, 0x486e140du}};
        const Fr minus_three = {{0x00000007u, 0xfffffff9u, 0xfff483f8u, 0x4a2f7c14u, 0x436ce825u, 0x6694e838u, 0x234e6cf9u, 0x2b7f9346u}};
        const Fr minus_four = {{0x00000009u, 0xfffffff7u, 0xfff13bf6u, 0xf1aac41au, 0x56b0982fu, 0xcd089848u, 0x76896789u, 0x135ae1ecu}};
        Fr f[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {                                           // unrolled: everything stays in registers
            Fr l4 = fr_add(w[k], w[k]); l4 = fr_add(l4, l4);
            f[k] = fr_sub(w[k + 1], l4);
        }
        if (mode != 0) {
            // structure-aware: D(f) = f(f-1)(f-2)(f-3) vanishes iff f is a base-4 digit (a field has no zero divisors), so a row whose
            // four differences all are digits holds and nothing is multiplied; any other row goes through the polynomial below -- the
            // verdict is the same for every witness.  Lanes of a warp share the row, so honest batches never leave the fast path.
            bool digits = true;
#pragma unroll
            for (int k = 0; k < 4; k++) digits = digits && (fr_is_zero(f[k]) || fr_eq(f[k], one) || fr_eq(f[k], two) || fr_eq(f[k], three));
            if (digits) return true;
        }
        // u = f(f-3) + 1.  Neither f - 3 nor u is reduced: the multiplier's SCANNED operand (the second) may be any 256-bit value when
        // the first is below q (the running value stays below 2q; tests/emu), the dot product takes operands below 2q -- an addition
        // without the conditional subtraction each.
        Fr u[4];
#pragma unroll
        for (int k = 0; k < 4; k++) u[k] = fr_add_noreduce(fr_mul_eo(f[k], fr_add_noreduce(f[k], minus_three), q), one);
        uint32_t t[9];
        fr_dot_wide<4>(t, u, u, q);                                             // sum u_k^2 ...
        add9_fr(t, minus_four);                                                 // ... - 4  =  sum D(f_k)
        return limbs9_is_multiple_of_q(t);
    }
    template <class PoolT>
    PG_HD static bool arith_row_holds(const CheckArgs& a, const DevRow& row, const PoolT& pool, const QRegs& q, uint64_t i) {
        return a.mode != 0 ? CheckBody::row_holds_sparse(a, row, pool, q, i) : CheckBody::row_holds<0, false>(a, row, pool, q, i);
    }
    template <class PoolT>
    PG_HD static bool row_ok(const CheckArgs& a, const PoolT& pool, const QRegs& q, uint32_t r, uint64_t i) {
        const DevRow row = a.rows[r];
        if (row.gate == GATE_ARITH) return arith_row_holds(a, row, pool, q, i);
        if (row.gate != GATE_RANGE) return true;
        Fr w[5];
        w[0] = row_load(row, 3, i); w[1] = row_load(row, 2, i); w[2] = row_load(row, 1, i); w[3] = row_load(row, 0, i);
        w[4] = r + 1 < a.n_rows ? row_load(a.rows[r + 1], 3, i) : fr_zero();
        return range_row_holds(w, q, a.mode);
    }
    // one (row, instance) pair per call: segments too small to fill the chip with one thread per instance
    template <class PoolT>
    PG_HD static uint32_t run_one(const CheckArgs& a, const PoolT& pool, const QRegs& q, uint64_t t, unsigned long long& first_bad) {
        const uint32_t r = (uint32_t)(t / a.n_inst); const uint64_t i = t - (uint64_t)r * a.n_inst;
        if (row_ok(a, pool, q, r, i)) return 0u;
        first_bad = a.base_row + i * (uint64_t)a.n_rows + r;
        return 1u;
    }
    // one instance per call, rows walked in order (like CheckBody::run): the fourth wire of the next row -- needed as d_next by a range
    // row -- is loaded once and kept as that row's own d; the next row's other wires are requested while this row is evaluated
    template <class PoolT>
    PG_HD static uint32_t run(const CheckArgs& a, const PoolT& pool, const QRegs& q, uint64_t i, unsigned long long& first_bad) {
        uint32_t bad = 0, first_local = ~0u;
        Fr d_cur = row_load(a.rows[0], 3, i);
        for (uint32_t r = 0; r < a.n_rows; r++) {
            const DevRow row = a.rows[r];
            Fr d_next = fr_zero();
            if (r + 1 < a.n_rows) {
                const DevRow& nr = a.rows[r + 1];
                d_next = row_load(nr, 3, i);
#pragma unroll
                for (int k = 0; k < 3; k++) row_prefetch(nr.loc[k], nr.addr[k], i);   // (no effect either way here: run r05o)
            }
            bool ok = true;
            if (row.gate == GATE_ARITH) ok = arith_row_holds(a, row, pool, q, i);
            else if (row.gate == GATE_RANGE) {
                Fr w[5];
                w[0] = d_cur; w[1] = row_load(row, 2, i); w[2] = row_load(row, 1, i); w[3] = row_load(row, 0, i); w[4] = d_next;
                ok = range_row_holds(w, q, a.mode);
            }
            if (!ok) { bad++; first_local = first_local < r ? first_local : r; }
            d_cur = d_next;
        }
        if (bad) { const unsigned long long g = a.base_row + i * (uint64_t)a.n_rows + first_local; if (g < first_bad) first_bad = g; }
        return bad;
    }
};

// ---------------------------------------------------------------------------------------------------- read-back
struct DevSeg {
    uint64_t base_row, base_var, n_inst;
    uint32_t n_rows, n_vars;
    DevTab tab[MAX_TABS];
    const DevRow* rows; const uint32_t* varloc; const uint32_t* pool;
    const uint4* param; uint64_t param_stride;
};

PG_HD uint32_t seg_find(const DevSeg* segs, uint32_t n_segs, uint64_t id, bool by_row) {
    uint32_t lo = 0, hi = n_segs;                      // last segment whose base <= id and that is not empty
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        const uint64_t base = by_row ? segs[mid].base_row : segs[mid].base_var;
        if (base <= id) lo = mid; else hi = mid;
    }
    return lo;
}

struct ReadVarsBody {
    struct Args { const DevSeg* segs; uint32_t n_segs; uint64_t var0; uint64_t n; uint4* dst; };
    PG_HD static void run(const Args& a, uint64_t t) {
        const uint64_t v = a.var0 + t;
        const DevSeg& s = a.segs[seg_find(a.segs, a.n_segs, v, false)];
        const uint64_t off = v - s.base_var;
        const uint64_t i = off / s.n_vars; const uint32_t j = (uint32_t)(off % s.n_vars);
        aos_store(a.dst, t, loc_load(s.tab, s.varloc[j], i));
    }
};

struct ColReadBody {   // one column (strided variables) -> contiguous scalars
    struct Args { DevTab tab; uint32_t loc; uint4* dst; uint64_t n; };
    PG_HD static void run(const Args& a, uint64_t i) { aos_store(a.dst, i, loc_load(&a.tab, a.loc, i)); }
};

// Expands rows into the reference composer's representation.  Outputs are column-major with `stride` rows per column; this
// launch covers rows [row0, row0 + n) and writes them at column offsets [out_off, out_off + n).  `what` selects the columns:
// the tiled kernel (kernels.cuh, k_materialize_tiled) produces wire values and the five instance-independent selector columns
// for whole instances; this body then only adds w_idx, q_c and PI for those rows, and everything for the ragged ends.
enum : uint32_t { MAT_W_IDX = 1u, MAT_W_VAL = 2u, MAT_SEL5 = 4u, MAT_QC = 8u, MAT_PI = 16u, MAT_ALL = 31u };
struct MaterializeBody {
    struct Args { const DevSeg* segs; uint32_t n_segs; uint32_t what; uint64_t row0; uint64_t n; uint64_t stride; uint64_t out_off;
                  unsigned long long* w_idx; uint4* w_val; uint4* sel; uint4* pi; };
    PG_HD static void run(const Args& a, uint64_t t) {
        const uint64_t g = a.row0 + t, o = a.out_off + t;
        const DevSeg& s = a.segs[seg_find(a.segs, a.n_segs, g, true)];
        const uint64_t off = g - s.base_row;
        const uint64_t i = off / s.n_rows; const uint32_t r = (uint32_t)(off % s.n_rows);
        const DevRow row = s.rows[r];
#pragma unroll
        for (int w = 0; w < 4; w++) {
            const uint32_t loc = row.loc[w];
            if (a.w_idx && (a.what & MAT_W_IDX)) {
                const DevTab& tb = s.tab[loc_tab(loc)];
                a.w_idx[(uint64_t)w * a.stride + o] = loc_kind(loc) == LOC_ZERO ? 0ull : tb.var_base + i * tb.var_stride + row.var[w];
            }
            if (a.w_val && (a.what & MAT_W_VAL)) aos_store(a.w_val, (uint64_t)w * a.stride + o, loc_load(s.tab, loc, i));
        }
        if (a.sel && (a.what & MAT_SEL5)) {
#pragma unroll
            for (int k = 0; k < 5; k++) aos_store(a.sel, (uint64_t)k * a.stride + o, pool_load(s.pool, row.sel[k]));
        }
        if (a.sel && (a.what & MAT_QC))
            aos_store(a.sel, 5ull * a.stride + o, row.qc_param >= 0 ? tab_load_fr(s.param, s.param_stride, (uint32_t)row.qc_param, i)
                                                                   : pool_load(s.pool, row.sel[5]));
        if (a.pi && (a.what & MAT_PI)) aos_store(a.pi, o, row.pi_param >= 0 ? tab_load_fr(s.param, s.param_stride, (uint32_t)row.pi_param, i)
                                                                          : pool_load(s.pool, row.pi_sel));
    }
};
// q_arith and q_range columns of rows [row0, row0 + n): one (R = BlsScalar::one()) or zero per row kind
struct GateSelBody {
    struct Args { const DevSeg* segs; uint32_t n_segs; uint64_t row0; uint64_t n; uint4* q_arith; uint4* q_range; };
    PG_HD static void run(const Args& a, uint64_t t) {
        const uint64_t g = a.row0 + t;
        const DevSeg& s = a.segs[seg_find(a.segs, a.n_segs, g, true)];
        const uint32_t gate = s.rows[(uint32_t)((g - s.base_row) % s.n_rows)].gate;
        if (a.q_arith) aos_store(a.q_arith, t, gate == GATE_ARITH ? fr_one() : fr_zero());
        if (a.q_range) aos_store(a.q_range, t, gate == GATE_RANGE ? fr_one() : fr_zero());
    }
};
// whole instances [inst0, inst0 + n_inst) of ONE segment, written from column offset out_off (row of instance inst0, local row 0)
struct MatTileArgs { DevSeg seg; uint64_t inst0, n_inst; uint64_t stride, out_off; uint4* w_val; uint4* sel; };

// ---------------------------------------------------------------------------------------------------- permutation map
// Copy constraints (SURVEY.md section 8f item 1).  dusk-plonk records, for every row it appends, the four wire positions in
// `perm.variable_map[var]` (add_variables_to_map: Left(n), Right(n), Output(n), Fourth(n) in that order) and later links the
// positions of one Variable into a cycle: sigma(position_k) = position_{k+1 mod len}.  Here the cycle successor of every
// wire position is computed directly from (template x instance) structure: the uses of a variable are its uses inside the
// instance that allocated it (template order), followed by its uses in later calls that took its column as an operand, in
// call order; the zero variable's uses are chained through every instance of every segment.
// Positions are encoded as row*4 + wire (wire: 0 = w_l, 1 = w_r, 2 = w_o, 3 = w_4).
constexpr uint32_t PERM_NONE = 0xffffffffu;
constexpr uint32_t PERM_REF_UNMAPPED = 0x7fffffffu;   // `ref` of a wire position that was never entered in the map: a fixed point of sigma
struct PermCons { uint32_t seg, op; uint64_t inst_off, n; uint32_t next; uint32_t pad; };   // a consumer of a column: segment `seg` binds it as operand `op`
struct PermSeg {
    uint64_t base_row, n_inst; uint32_t n_rows, pad;
    const uint32_t* next_in_inst;    // [n_rows*4]: next use (r*4+w) of the same variable inside the same instance, or PERM_NONE
    const uint32_t* ref;             // [n_rows*4]: 0 = zero variable, 1+j = local variable j, 0x80000000|e = operand e (canonicalised)
    const uint32_t* first_local;     // [n_vars]: first use of local variable j in its own instance, or PERM_NONE
    const uint32_t* cons_head;       // [n_vars]: index+1 into the consumer array of the first consumer of local variable j's column, 0 = none
    uint32_t first_op[4];            // first use of operand e inside an instance of this segment
    uint32_t first_zero;             // first use of the zero variable inside an instance, or PERM_NONE
    uint32_t next_zero_seg;          // next segment (index) with zero-variable uses and instances, or PERM_NONE
    uint32_t op_src_seg[4], op_src_local[4]; uint64_t op_inst_off[4]; uint32_t op_cons_idx[4];   // operand e: source column and this segment's record in its consumer list
};
struct PermBody {
    struct Args { const DevSeg* segs; const PermSeg* psegs; const PermCons* cons; uint32_t n_segs; uint32_t first_zero_seg; uint64_t row0; uint64_t n; unsigned long long* sigma; };

    // first consumer at or after list position `c` (index+1) that covers source instance i: returns its first use as a global position
    PG_HD static bool consumer_first_use(const Args& a, uint32_t c, uint64_t i, unsigned long long* out) {
        while (c) {
            const PermCons& k = a.cons[c - 1];
            if (i >= k.inst_off && i - k.inst_off < k.n) {
                const PermSeg& t = a.psegs[k.seg];
                const uint32_t f = t.first_op[k.op];
                *out = (t.base_row + (i - k.inst_off) * t.n_rows + (f >> 2)) * 4ull + (f & 3u);
                return true;
            }
            c = k.next;
        }
        return false;
    }
    // first use overall of local variable j of instance i of segment s
    PG_HD static unsigned long long variable_first_use(const Args& a, uint32_t s, uint32_t j, uint64_t i) {
        const PermSeg& t = a.psegs[s];
        const uint32_t f = t.first_local[j];
        if (f != PERM_NONE) return (t.base_row + i * t.n_rows + (f >> 2)) * 4ull + (f & 3u);
        unsigned long long out = 0;
        consumer_first_use(a, t.cons_head[j], i, &out);          // a used variable without own uses has a consumer
        return out;
    }
    PG_HD static void run(const Args& a, uint64_t tix) {
        const uint64_t g = a.row0 + tix;
        const uint32_t si = seg_find(a.segs, a.n_segs, g, true);
        const PermSeg& s = a.psegs[si];
        const uint64_t off = g - s.base_row;
        const uint64_t i = off / s.n_rows; const uint32_t r = (uint32_t)(off % s.n_rows);
#pragma unroll
        for (uint32_t w = 0; w < 4; w++) {
            const uint32_t ref = s.ref[r * 4 + w], nxt = s.next_in_inst[r * 4 + w];
            unsigned long long out;
            if (ref == PERM_REF_UNMAPPED) out = g * 4ull + w;
            else if (nxt != PERM_NONE) out = (s.base_row + i * s.n_rows + (nxt >> 2)) * 4ull + (nxt & 3u);
            else if (ref == 0) {                                 // zero variable: next instance, next segment, or wrap to the very first use
                if (i + 1 < s.n_inst) out = (s.base_row + (i + 1) * s.n_rows + (s.first_zero >> 2)) * 4ull + (s.first_zero & 3u);
                else {
                    const uint32_t ns = s.next_zero_seg != PERM_NONE ? s.next_zero_seg : a.first_zero_seg;
                    const PermSeg& t = a.psegs[ns];
                    out = (t.base_row + (t.first_zero >> 2)) * 4ull + (t.first_zero & 3u);
                }
            } else if (ref & 0x80000000u) {                      // operand: later consumers of the same column, else wrap to the variable's first use
                const uint32_t e = ref & 3u;
                const uint64_t i_src = i + s.op_inst_off[e];
                if (!consumer_first_use(a, a.cons[s.op_cons_idx[e]].next, i_src, &out))
                    out = variable_first_use(a, s.op_src_seg[e], s.op_src_local[e], i_src);
            } else {                                             // own variable: consumers of its column, else wrap
                const uint32_t j = ref - 1u;
                if (!consumer_first_use(a, s.cons_head[j], i, &out)) out = variable_first_use(a, si, j, i);
            }
            a.sigma[(uint64_t)w * a.n + tix] = out;
        }
    }
};

// ---------------------------------------------------------------------------------------------------- permutation argument
// [DEP] dusk-plonk 0.8 permutation.rs.  The identity of wire position (i, w) is k_w * w^i, k = (1, K1, K2, K3); sigma maps it
// to the identity of its cycle successor.  Positions: PermBody's encoding row*4 + wire; rows >= n_sig (padding) map to themselves.
PG_HD uint64_t perm_successor(const unsigned long long* sigma, uint64_t n_sig, uint64_t i, uint32_t w) {
    return i < n_sig ? sigma[(uint64_t)w * n_sig + i] : i * 4ull + w;
}
// sigma_w(w^i) = k_{w'} * w^{r'} (compute_permutation_lagrange): out is 4 columns of n evaluations
struct PermSigmaBody {
    struct Args { const unsigned long long* sigma; uint64_t n_sig; uint64_t n; const uint4* tw; uint32_t log_n; Fr k[4]; uint4* out; };
    PG_HD static void run(const Args& a, uint64_t i) {
#pragma unroll
        for (uint32_t w = 0; w < 4; w++) {
            const uint64_t p = perm_successor(a.sigma, a.n_sig, i, w);
            aos_store(a.out, (uint64_t)w * a.n + i, fr_mul(a.k[p & 3u], domain_pow(a.tw, a.log_n, p >> 2)));
        }
    }
};
// The ratios of the grand product (compute_fast_permutation_poly), inside k_batch_inv's two walks (in_slot 0 = den, out_slot 1):
//   num_i = prod_w (v_w(i) + beta*k_w*w^i + gamma),  den_i = prod_w (v_w(i) + beta*sigma_w(w^i) + gamma)
// pre parks num_i in `ratio` and hands den_i to the inversion; post writes ratio_i = num_i * den_i^-1.  A zero den_i (the reference
// panics in invert().unwrap()) is counted in CNT_N_ERR / CNT_FIRST_ERR -- the zero-aware inversion would store 0 silently.
// check (caller-supplied rows): a sigma entry >= 4n or an unreduced wire value is counted in CNT_UNSAT / CNT_FIRST_BAD (and the
// position is read as a fixed point, so no access leaves the twiddle table).
struct PermRatioHook {
    struct Args { const uint4* w; uint64_t n; const unsigned long long* sigma; uint64_t n_sig; const uint4* tw; uint32_t log_n;
                  Fr bk[4]; Fr gamma; uint4* den; uint4* ratio; unsigned long long* counters; int check; };
    PG_HD static Fr pre(const Args& a, uint64_t i) {
        const Fr wi = domain_pow(a.tw, a.log_n, i);
        Fr num = fr_one(), den = fr_one();
        bool bad = false;
#pragma unroll
        for (uint32_t w = 0; w < 4; w++) {
            const Fr v = aos_load(a.w, (uint64_t)w * a.n + i);
            uint64_t p = perm_successor(a.sigma, a.n_sig, i, w);
            if (a.check) {
                if (!fr_is_reduced(v)) bad = true;
                if (p >= 4ull * a.n) { bad = true; p = i * 4ull + w; }
            }
            num = fr_mul(num, fr_add(fr_add(v, fr_mul(a.bk[w], wi)), a.gamma));
            den = fr_mul(den, fr_add(fr_add(v, fr_mul(a.bk[p & 3u], domain_pow(a.tw, a.log_n, p >> 2))), a.gamma));
        }
        if (bad) { counter_add(a.counters + CNT_UNSAT, 1ull); counter_min(a.counters + CNT_FIRST_BAD, (unsigned long long)i); }
        if (fr_is_zero(den)) { counter_add(a.counters + CNT_N_ERR, 1ull); counter_min(a.counters + CNT_FIRST_ERR, (unsigned long long)i); }
        aos_store(a.ratio, i, num);
        tab_store_fr(a.den, a.n, 0, i, den);
        return den;
    }
    PG_HD static void post(const Args& a, uint64_t i, const Fr&, const Fr& den_inv) { aos_store(a.ratio, i, fr_mul(aos_load(a.ratio, i), den_inv)); }
};

// ---------------------------------------------------------------------------------------------------- quotient polynomial
// [DEP] dusk-plonk 0.8 quotient_poly.rs (compute_circuit_satisfiability_equation + compute_permutation_checks), recalled.  The 4N
// coset g*<zeta> is taken as four size-N sub-cosets h_j*H, h_j = g*zeta^j: point k of sub-coset j is x = h_j * w^k, and x*w is point
// k+1 (mod N) of the same sub-coset.  Evaluation vectors, N scalars each, in this order (QV_*); the first QV_COEF are coefficient
// vectors too (Engine::quotient), the last one is alpha^2 * L_1 (coset FFT of the constant coefficient vector alpha^2 / N).
enum : uint32_t { QV_W = 0, QV_Z = 4, QV_S = 5, QV_QM = 9, QV_QL, QV_QR, QV_QO, QV_Q4, QV_QC, QV_QARITH, QV_QRANGE, QV_PI, QV_COEF, QV_L1 = QV_COEF, QV_EV };
PG_HD Fr quot_delta(const Fr& f, const Fr& two, const Fr& three) {       // f(f-1)(f-2)(f-3) = u(u+2), u = f(f-3)
    const Fr u = fr_mul(f, fr_sub(f, three));
    return fr_mul(u, fr_add(u, two));
}
PG_HD Fr quot_times4(const Fr& x) { const Fr y = fr_add(x, x); return fr_add(y, y); }
// t(x) on sub-coset j: (arith + range + perm) / (x^N - 1), 39 Montgomery multiplications per point with the range widget, 26
// without.  has_pi / has_range are decided on the composer's row templates (no PI parameter / no range-widget row: the polynomial
// is zero), never on witness values.
struct QuotientBody {
    struct Args { const uint4* ev; uint64_t n; const uint4* tw; uint32_t log_n; int has_pi, has_range;
                  Fr bkh[4];      /* beta * k_w * h_j */
                  Fr beta, gamma, alpha, rho, kappa, zh_inv, two, three; uint4* out; };
    PG_HD static Fr ld(const Args& a, uint32_t v, uint64_t k) { return aos_load(a.ev, (uint64_t)v * a.n + k); }
    PG_HD static void run(const Args& a, uint64_t k) {
        const uint64_t kn = (k + 1) & (a.n - 1);
        const Fr w_a = ld(a, QV_W, k), w_b = ld(a, QV_W + 1, k), w_c = ld(a, QV_W + 2, k), w_d = ld(a, QV_W + 3, k);
        // arithmetic widget: q_arith * (q_m a b + q_l a + q_r b + q_o c + q_4 d + q_c) + PI
        Fr g = fr_mul(fr_mul(ld(a, QV_QM, k), w_a), w_b);
        g = fr_add(g, fr_mul(ld(a, QV_QL, k), w_a));
        g = fr_add(g, fr_mul(ld(a, QV_QR, k), w_b));
        g = fr_add(g, fr_mul(ld(a, QV_QO, k), w_c));
        g = fr_add(g, fr_mul(ld(a, QV_Q4, k), w_d));
        g = fr_add(g, ld(a, QV_QC, k));
        Fr t = fr_mul(ld(a, QV_QARITH, k), g);
        if (a.has_pi) t = fr_add(t, ld(a, QV_PI, k));
        // range widget: rho * q_range * (D(c-4d) + kappa D(b-4c) + kappa^2 D(a-4b) + kappa^3 D(d(xw)-4a)), Horner in kappa
        if (a.has_range) {
            Fr s = quot_delta(fr_sub(ld(a, QV_W + 3, kn), quot_times4(w_a)), a.two, a.three);
            s = fr_add(fr_mul(s, a.kappa), quot_delta(fr_sub(w_a, quot_times4(w_b)), a.two, a.three));
            s = fr_add(fr_mul(s, a.kappa), quot_delta(fr_sub(w_b, quot_times4(w_c)), a.two, a.three));
            s = fr_add(fr_mul(s, a.kappa), quot_delta(fr_sub(w_c, quot_times4(w_d)), a.two, a.three));
            t = fr_add(t, fr_mul(fr_mul(a.rho, ld(a, QV_QRANGE, k)), s));
        }
        // permutation: alpha (z(x) prod_w (v_w + beta k_w x + gamma) - z(xw) prod_w (v_w + beta sigma_w(x) + gamma)) + alpha^2 L_1(x) (z(x) - 1)
        const Fr wk = domain_pow(a.tw, a.log_n, k);
        const Fr v[4] = {w_a, w_b, w_c, w_d};
        Fr num = fr_add(fr_add(v[0], fr_mul(a.bkh[0], wk)), a.gamma);
        Fr den = fr_add(fr_add(v[0], fr_mul(a.beta, ld(a, QV_S, k))), a.gamma);
#pragma unroll
        for (uint32_t w = 1; w < 4; w++) {
            num = fr_mul(num, fr_add(fr_add(v[w], fr_mul(a.bkh[w], wk)), a.gamma));
            den = fr_mul(den, fr_add(fr_add(v[w], fr_mul(a.beta, ld(a, QV_S + w, k))), a.gamma));
        }
        const Fr z = ld(a, QV_Z, k);
        const Fr p = fr_mul(a.alpha, fr_sub(fr_mul(z, num), fr_mul(ld(a, QV_Z, kn), den)));
        t = fr_add(t, fr_add(p, fr_mul(ld(a, QV_L1, k), fr_sub(z, fr_one()))));
        aos_store(a.out, k, fr_mul(t, a.zh_inv));                                 // / Z_H(x) = x^N - 1, one constant per sub-coset
    }
};
// t's coefficients from the inverse size-N transforms c_j of the four sub-cosets' values (in place, t[j*n + m] = c_j[m]):
//   c_j[m] = zeta^(jm) * sum_r iota^(jr) * t_(m+rN) g^(m+rN),  iota = zeta^N,
// so with e_j = c_j[m] * h_j^-m (h_j^-m = g^-m zeta^-jm, from two-level tables) a 4-point inverse DFT over j gives
// t_(m+rN) = (1/4) g^-rN * sum_j iota^-jr e_j, written to t[r*n + m]: split_tx_poly's t_1 .. t_4 directly.
struct QuotientSplitBody {
    struct Args { uint4* t; uint64_t n; const uint4* inv_tab[4]; uint32_t log_lo; Fr iota_inv; Fr scale[4]; };
    PG_HD static void run(const Args& a, uint64_t m) {
        Fr e[4];
#pragma unroll
        for (uint32_t j = 0; j < 4; j++) e[j] = fr_mul(aos_load(a.t, (uint64_t)j * a.n + m), pow_table_at(a.inv_tab[j], a.log_lo, m));
        const Fr s02 = fr_add(e[0], e[2]), d02 = fr_sub(e[0], e[2]);
        const Fr s13 = fr_add(e[1], e[3]), d13 = fr_mul(a.iota_inv, fr_sub(e[1], e[3]));
        const Fr y[4] = {fr_add(s02, s13), fr_add(d02, d13), fr_sub(s02, s13), fr_sub(d02, d13)};
#pragma unroll
        for (uint32_t r = 0; r < 4; r++) aos_store(a.t, (uint64_t)r * a.n + m, fr_mul(y[r], a.scale[r]));
    }
};
// data[i] = v
struct FillBody {
    struct Args { uint4* data; Fr v; uint64_t n; };
    PG_HD static void run(const Args& a, uint64_t i) { aos_store(a.data, i, a.v); }
};

// ---------------------------------------------------------------------------------------------------- openings (rounds 4 and 5)
// [DEP] dusk-plonk 0.8 Prover::prove (evaluations, linearisation_poly::compute, compute_quotient_opening_poly /
// compute_aggregate_witness), recalled.  Vectors: the QV_PI coefficient vectors of the quotient (wires, z, sigma, selectors; QV_*
// order) and t_1 .. t_4 (OV_T ..).  Pairs (vector, point): every vector at zeta (pair = vector), and w_l, w_r, w_4, z at zeta*w
// (OV_SHIFTED ..).
enum : uint32_t { OV_T = QV_PI, OV_VEC = OV_T + 4, OV_SHIFTED = OV_VEC, OV_PAIRS = OV_SHIFTED + 4 };
PG_HD int open_shift_slot(uint32_t v) { return v == QV_W ? 0 : v == QV_W + 1 ? 1 : v == QV_W + 3 ? 2 : v == QV_Z ? 3 : -1; }
// Evaluation pass, index i = v * s + j (j < s, s | len = N): partial[pair][j] = p^j * sum_k c_v[j + k s] (p^s)^k by Horner over the strided
// coefficients, for p = zeta and, for the shifted vectors, zeta*w.  One Fr multiplication per coefficient and pair.  The t vectors
// are caller input: an unreduced coefficient is counted in CNT_UNSAT / CNT_FIRST_BAD (index r * n + m of t).
struct OpenEvalBody {
    struct Args { const uint4* coef; const uint4* t; uint64_t len, s, n /* OV_VEC * s */; uint32_t log_lo; const uint4* tab[2]; Fr step[2];
                  uint4* partial; unsigned long long* counters; };
    PG_HD static void run(const Args& a, uint64_t i) {
        const uint32_t v = (uint32_t)(i / a.s); const uint64_t j = i % a.s;
        const uint4* c = v < OV_T ? a.coef + 2 * (uint64_t)v * a.len : a.t + 2 * (uint64_t)(v - OV_T) * a.len;
        const int sh = open_shift_slot(v);
        Fr acc = fr_zero(), acc2 = fr_zero();
        for (uint64_t m = a.len - a.s + j;; m -= a.s) {
            const Fr x = aos_load(c, m);
            if (v >= OV_T && !fr_is_reduced(x)) { counter_add(a.counters + CNT_UNSAT, 1ull); counter_min(a.counters + CNT_FIRST_BAD, (unsigned long long)((v - OV_T) * a.len + m)); }
            acc = fr_add(fr_mul(acc, a.step[0]), x);
            if (sh >= 0) acc2 = fr_add(fr_mul(acc2, a.step[1]), x);
            if (m < a.s) break;
        }
        aos_store(a.partial, (uint64_t)v * a.s + j, fr_mul(acc, pow_table_at(a.tab[0], a.log_lo, j)));
        if (sh >= 0) aos_store(a.partial, (uint64_t)(OV_SHIFTED + sh) * a.s + j, fr_mul(acc2, pow_table_at(a.tab[1], a.log_lo, j)));
    }
};
// out[i] = sum_(k < len) in[i * len + k], i < n
struct OpenSumBody {
    struct Args { const uint4* in; uint4* out; uint64_t len, n; };
    PG_HD static void run(const Args& a, uint64_t i) {
        Fr s = fr_zero();
        for (uint64_t k = 0; k < a.len; k++) s = fr_add(s, aos_load(a.in, i * a.len + k));
        aos_store(a.out, i, s);
    }
};
// Combination pass, pointwise over the coefficients m: out = [agg_zeta, agg_zeta_w, r] (3 x n), with the host's weights
//   r          = rw . (q_m, q_l, q_r, q_o, q_4, q_c, q_range, z, sigma_4)
//   agg_zeta   = t_1 + zeta^N t_2 + zeta^2N t_3 + zeta^3N t_4 + v r + v^2 w_l + v^3 w_r + v^4 w_o + v^5 w_4 + v^6 sigma_1 + v^7 sigma_2 + v^8 sigma_3
//   agg_zeta_w = z + v' w_l + v'^2 w_r + v'^3 w_4
// 23 Montgomery multiplications per coefficient.
struct OpenCombineBody {
    struct Args { const uint4* coef; const uint4* t; uint64_t n; Fr rw[9]; Fr zn[3]; Fr v[8]; Fr vs[3]; uint4* out; };
    PG_HD static Fr ld(const Args& a, uint32_t v, uint64_t m) { return aos_load(a.coef, (uint64_t)v * a.n + m); }
    PG_HD static void run(const Args& a, uint64_t m) {
        Fr r = fr_mul(a.rw[0], ld(a, QV_QM, m));
#pragma unroll
        for (int k = 1; k < 6; k++) r = fr_add(r, fr_mul(a.rw[k], ld(a, QV_QM + k, m)));      // q_l q_r q_o q_4 q_c
        r = fr_add(r, fr_mul(a.rw[6], ld(a, QV_QRANGE, m)));
        r = fr_add(r, fr_mul(a.rw[7], ld(a, QV_Z, m)));
        r = fr_add(r, fr_mul(a.rw[8], ld(a, QV_S + 3, m)));
        Fr g = aos_load(a.t, m);
#pragma unroll
        for (int k = 0; k < 3; k++) g = fr_add(g, fr_mul(a.zn[k], aos_load(a.t, (uint64_t)(k + 1) * a.n + m)));
        g = fr_add(g, fr_mul(a.v[0], r));
#pragma unroll
        for (int k = 0; k < 4; k++) g = fr_add(g, fr_mul(a.v[1 + k], ld(a, QV_W + k, m)));
#pragma unroll
        for (int k = 0; k < 3; k++) g = fr_add(g, fr_mul(a.v[5 + k], ld(a, QV_S + k, m)));
        Fr h = ld(a, QV_Z, m);
        h = fr_add(h, fr_mul(a.vs[0], ld(a, QV_W, m)));
        h = fr_add(h, fr_mul(a.vs[1], ld(a, QV_W + 1, m)));
        h = fr_add(h, fr_mul(a.vs[2], ld(a, QV_W + 3, m)));
        aos_store(a.out, m, g);
        aos_store(a.out, a.n + m, h);
        aos_store(a.out, 2 * a.n + m, r);
    }
};

// ---------------------------------------------------------------------------------------------------- synthetic inputs
PG_HD uint64_t splitmix64_at(uint64_t seed, uint64_t index1) {   // output number index1 (1-based) of SplitMix64(seed)
    uint64_t z = seed + index1 * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
struct SynthBody {
    struct Args { uint64_t seed; uint64_t n; int kind; uint32_t bits; uint4* dst; };
    PG_HD static void run(const Args& a, uint64_t i) {
        Fr lo, hi;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint64_t w0 = splitmix64_at(a.seed, 8 * i + j + 1), w1 = splitmix64_at(a.seed, 8 * i + 4 + j + 1);
            lo.v[2 * j] = (uint32_t)w0; lo.v[2 * j + 1] = (uint32_t)(w0 >> 32);
            hi.v[2 * j] = (uint32_t)w1; hi.v[2 * j + 1] = (uint32_t)(w1 >> 32);
        }
        int kind = a.kind;
        if (kind == 2) kind = (i & 1) ? 0 : 1;
        Fr out;
        if (kind == 0) {                                    // from_bytes_wide: lo*R2 + hi*R3 (Montgomery products)
            out = fr_add(fr_mul(fr_r2(), lo), fr_mul(fr_r3(), hi));
        } else {                                            // low `bits` bits of the draw (bits <= 254 < log2 q)
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const int rem = (int)a.bits - 32 * k;
                if (rem <= 0) lo.v[k] = 0; else if (rem < 32) lo.v[k] &= (1u << rem) - 1u;
            }
            if (kind == 3 && a.bits > 0) lo.v[(a.bits - 1) >> 5] |= 1u << ((a.bits - 1) & 31u);
            out = fr_mul(fr_r2(), lo);
        }
        aos_store(a.dst, i, out);
    }
};

// ---------------------------------------------------------------------------------------------------- wire format
// BlsScalar::to_bytes / from_bytes (dusk_bytes::Serializable<32>, used at /root/reference/src/range.rs:163): canonical
// little-endian 32 bytes <-> Montgomery limbs.  from_bytes rejects encodings >= q (counted; the output is then 0).
struct ToBytesBody {
    struct Args { const uint4* src; uint4* dst; uint64_t n; };
    PG_HD static void run(const Args& a, uint64_t i) { aos_store(a.dst, i, fr_from_mont(aos_load(a.src, i))); }
};
struct FromBytesBody {
    struct Args { const uint4* src; uint4* dst; uint64_t n; unsigned long long* counters; };
    PG_HD static void run(const Args& a, uint64_t i) {
        const Fr c = aos_load(a.src, i);
        const uint32_t q[8] = {PG_Q0, PG_Q1, PG_Q2, PG_Q3, PG_Q4, PG_Q5, PG_Q6, PG_Q7};
        Fr d;
        if (!fr_sub_limbs(d.v, c.v, q)) { counter_add(a.counters + CNT_N_ERR, 1ull); counter_min(a.counters + CNT_FIRST_ERR, (unsigned long long)i); aos_store(a.dst, i, fr_zero()); }
        else aos_store(a.dst, i, fr_to_mont(c));
    }
};

// ---------------------------------------------------------------------------------------------------- Fr self-test
struct FrOpBody {
    struct Args { int op; const uint4* a; const uint4* b; uint4* out; uint64_t n; };
    PG_HD static void run(const Args& g, uint64_t i) {
        const Fr a = aos_load(g.a, i);
        Fr b = fr_zero(); if (g.b) b = aos_load(g.b, i);
        Fr r;
        switch (g.op) {
            case 0: r = fr_mul(a, b); break;
            case 1: r = fr_add(a, b); break;
            case 2: r = fr_sub(a, b); break;
            case 3: r = fr_neg(a); break;
            case 5: r = fr_from_mont(a); break;
            case 6: r = fr_mul_cios(a, b); break;
            default: r = fr_zero(); break;
        }
        aos_store(g.out, i, r);
    }
};
}  // namespace pg
