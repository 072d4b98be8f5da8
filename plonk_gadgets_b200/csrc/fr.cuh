// fr.cuh -- BLS12-381 scalar field Fr for sm_100a: 8 x 32-bit little-endian limbs of the Montgomery form a*2^256 mod q.
//
// Memory image == dusk-bls12_381 `Scalar([u64;4])` (= dusk_plonk BlsScalar), so results are bit-comparable with the
// reference composer (uses: /root/reference/src/range.rs:62,:87,:102,:146,:152,:163; /root/reference/src/scalar.rs:73,:121,:122,:126).
// All outputs are fully reduced to [0,q): the reference type is always canonical in Montgomery form, and bit-exact
// parity needs the same representative.
//
// Two multipliers, same results:
//   fr_mul_cios  : portable C (64-bit intermediates), runs on host and device; used by host-side template building.
//   fr_mul       : device hot path.  Operand-scanning Montgomery with the partial products split into an "even" and an
//                  "odd" accumulator (limb-aligned and one-limb-shifted), so that every row of 32x32->64 products is one
//                  uninterrupted mad.lo.cc/madc.hi.cc carry chain that ptxas maps onto IMAD.WIDE.U32(.X) -- no carry
//                  save/restore between products.  q' = -q^-1 mod 2^32 = 0xffffffff, so m_i = -t_0 needs no multiply.
//   On the host the same even/odd algorithm runs through a carry-flag emulation (tests/emu), so its limb logic is
//   testable without a GPU.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define PG_HD __host__ __device__ __forceinline__
#define PG_D __device__ __forceinline__
#else
#define PG_HD inline
#define PG_D inline
// host-only builds (tests/emu): the two CUDA vector helpers the layout code uses
struct alignas(16) uint4 { uint32_t x, y, z, w; };
static inline uint4 make_uint4(uint32_t x, uint32_t y, uint32_t z, uint32_t w) { uint4 r = {x, y, z, w}; return r; }
#endif

// tests/emu defines PG_EMU_CHECKS: the host emulation then reports every place where a carry the device code drops
// (or adds into a limb assumed to have room) is not zero.
#if !defined(__CUDA_ARCH__) && defined(PG_EMU_CHECKS)
void pg_emu_carry_violation();
#define PG_EMU_VIOLATION() pg_emu_carry_violation()
#else
#define PG_EMU_VIOLATION() ((void)0)
#endif

namespace pg {

struct Fr { uint32_t v[8]; };

// q, little-endian 32-bit limbs
#define PG_Q0 0x00000001u
#define PG_Q1 0xffffffffu
#define PG_Q2 0xfffe5bfeu
#define PG_Q3 0x53bda402u
#define PG_Q4 0x09a1d805u
#define PG_Q5 0x3339d808u
#define PG_Q6 0x299d7d48u
#define PG_Q7 0x73eda753u

// The same limbs behind a __constant__ array: as immediates ptxas splits every reduction product into IMAD.HI + IMAD
// (6 multiplier-pipe cycles); as constant-bank operands they stay one IMAD.WIDE.U32.X (4 cycles).
#if defined(__CUDACC__)
__constant__ uint32_t c_q[8] = {PG_Q0, PG_Q1, PG_Q2, PG_Q3, PG_Q4, PG_Q5, PG_Q6, PG_Q7};
#endif
PG_HD uint32_t fr_qc(int i) {
#if defined(__CUDA_ARCH__)
    return c_q[i];
#else
    const uint32_t q[8] = {PG_Q0, PG_Q1, PG_Q2, PG_Q3, PG_Q4, PG_Q5, PG_Q6, PG_Q7};
    return q[i];
#endif
}
// Modulus limbs held in ordinary (vector) registers.  With a uniform-register / constant-bank operand ptxas cannot form
// IMAD.WIDE.U32.X (carry-in) and splits each reduction product into IMAD.X + IMAD.HI.U32.X (6 multiplier cycles instead of 4);
// the hot kernels therefore load q once per thread from shared memory into a QRegs and pass it down.
struct QRegs { uint32_t v[8]; };
PG_HD QRegs q_regs_default() { QRegs q; for (int i = 0; i < 8; i++) q.v[i] = fr_qc(i); return q; }
PG_HD uint32_t fr_q(int i) {
    switch (i) { case 0: return PG_Q0; case 1: return PG_Q1; case 2: return PG_Q2; case 3: return PG_Q3;
                 case 4: return PG_Q4; case 5: return PG_Q5; case 6: return PG_Q6; default: return PG_Q7; }
}
// R = 2^256 mod q  (Montgomery form of 1 == BlsScalar::one())
PG_HD Fr fr_one() { Fr r = {{0xfffffffeu, 0x00000001u, 0x00034802u, 0x5884b7fau, 0xecbc4ff5u, 0x998c4fefu, 0xacc5056fu, 0x1824b159u}}; return r; }
// R^2 mod q (to_montgomery multiplier; From<u64> == raw * R2)
PG_HD Fr fr_r2() { Fr r = {{0xf3f29c6du, 0xc999e990u, 0x87925c23u, 0x2b6cedcbu, 0x7254398fu, 0x05d31496u, 0x9f59ff11u, 0x0748d9d9u}}; return r; }
// R^3 mod q (from_bytes_wide high half multiplier)
PG_HD Fr fr_r3() { Fr r = {{0x439b73afu, 0xc62c1807u, 0x8cf06990u, 0x1b3e0d18u, 0xc7b5f418u, 0x73d13c71u, 0xc8db33e9u, 0x6e2a5bb9u}}; return r; }
PG_HD Fr fr_zero() { Fr r = {{0, 0, 0, 0, 0, 0, 0, 0}}; return r; }

PG_HD bool fr_is_zero(const Fr& a) { return (a.v[0] | a.v[1] | a.v[2] | a.v[3] | a.v[4] | a.v[5] | a.v[6] | a.v[7]) == 0; }
PG_HD bool fr_eq(const Fr& a, const Fr& b) {
    uint32_t d = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) d |= a.v[i] ^ b.v[i];
    return d == 0;
}

// ---- portable add/sub (host + device fallback) -------------------------------------------------------------------
PG_HD uint32_t fr_sub_limbs(uint32_t* r, const uint32_t* a, const uint32_t* b) {   // r = a - b, returns borrow (0/1)
    uint64_t bw = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { uint64_t t = (uint64_t)a[i] - b[i] - bw; r[i] = (uint32_t)t; bw = (t >> 32) & 1; }
    return (uint32_t)bw;
}
PG_HD uint32_t fr_add_limbs(uint32_t* r, const uint32_t* a, const uint32_t* b) {   // r = a + b, returns carry (0/1)
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { uint64_t t = (uint64_t)a[i] + b[i] + c; r[i] = (uint32_t)t; c = t >> 32; }
    return (uint32_t)c;
}

#if defined(__CUDA_ARCH__)
// ---- device add/sub with PTX carry chains (IADD3.X on the ALU pipe, off the IMAD pipe) -----------------------------
PG_D Fr fr_add(const Fr& a, const Fr& b) {
    Fr s, d; uint32_t bw;
    asm("add.cc.u32 %0, %8, %16;\n\taddc.cc.u32 %1, %9, %17;\n\taddc.cc.u32 %2, %10, %18;\n\taddc.cc.u32 %3, %11, %19;\n\t"
        "addc.cc.u32 %4, %12, %20;\n\taddc.cc.u32 %5, %13, %21;\n\taddc.cc.u32 %6, %14, %22;\n\taddc.u32 %7, %15, %23;"
        : "=&r"(s.v[0]), "=&r"(s.v[1]), "=&r"(s.v[2]), "=&r"(s.v[3]), "=&r"(s.v[4]), "=&r"(s.v[5]), "=&r"(s.v[6]), "=&r"(s.v[7])
        : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]),
          "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]), "r"(b.v[7]));
    // a,b < q < 2^255: the sum fits 256 bits.  d = s - q; keep s when that borrows.
    asm("sub.cc.u32 %0, %9, %17;\n\tsubc.cc.u32 %1, %10, %18;\n\tsubc.cc.u32 %2, %11, %19;\n\tsubc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\tsubc.cc.u32 %5, %14, %22;\n\tsubc.cc.u32 %6, %15, %23;\n\tsubc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=&r"(d.v[0]), "=&r"(d.v[1]), "=&r"(d.v[2]), "=&r"(d.v[3]), "=&r"(d.v[4]), "=&r"(d.v[5]), "=&r"(d.v[6]), "=&r"(d.v[7]), "=&r"(bw)
        : "r"(s.v[0]), "r"(s.v[1]), "r"(s.v[2]), "r"(s.v[3]), "r"(s.v[4]), "r"(s.v[5]), "r"(s.v[6]), "r"(s.v[7]),
          "r"(PG_Q0), "r"(PG_Q1), "r"(PG_Q2), "r"(PG_Q3), "r"(PG_Q4), "r"(PG_Q5), "r"(PG_Q6), "r"(PG_Q7));
#pragma unroll
    for (int i = 0; i < 8; i++) d.v[i] = bw ? s.v[i] : d.v[i];
    return d;
}
PG_D Fr fr_sub(const Fr& a, const Fr& b) {
    Fr d; uint32_t bw;
    asm("sub.cc.u32 %0, %9, %17;\n\tsubc.cc.u32 %1, %10, %18;\n\tsubc.cc.u32 %2, %11, %19;\n\tsubc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\tsubc.cc.u32 %5, %14, %22;\n\tsubc.cc.u32 %6, %15, %23;\n\tsubc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=&r"(d.v[0]), "=&r"(d.v[1]), "=&r"(d.v[2]), "=&r"(d.v[3]), "=&r"(d.v[4]), "=&r"(d.v[5]), "=&r"(d.v[6]), "=&r"(d.v[7]), "=&r"(bw)
        : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]),
          "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]), "r"(b.v[7]));
    // bw = 0xffffffff when a < b: add q back under the mask
    asm("add.cc.u32 %0, %0, %8;\n\taddc.cc.u32 %1, %1, %9;\n\taddc.cc.u32 %2, %2, %10;\n\taddc.cc.u32 %3, %3, %11;\n\t"
        "addc.cc.u32 %4, %4, %12;\n\taddc.cc.u32 %5, %5, %13;\n\taddc.cc.u32 %6, %6, %14;\n\taddc.u32 %7, %7, %15;"
        : "+r"(d.v[0]), "+r"(d.v[1]), "+r"(d.v[2]), "+r"(d.v[3]), "+r"(d.v[4]), "+r"(d.v[5]), "+r"(d.v[6]), "+r"(d.v[7])
        : "r"(PG_Q0 & bw), "r"(PG_Q1 & bw), "r"(PG_Q2 & bw), "r"(PG_Q3 & bw), "r"(PG_Q4 & bw), "r"(PG_Q5 & bw), "r"(PG_Q6 & bw), "r"(PG_Q7 & bw));
    return d;
}
#else
PG_HD Fr fr_add(const Fr& a, const Fr& b) {
    Fr s, d; const uint32_t q[8] = {PG_Q0, PG_Q1, PG_Q2, PG_Q3, PG_Q4, PG_Q5, PG_Q6, PG_Q7};
    fr_add_limbs(s.v, a.v, b.v);
    uint32_t bw = fr_sub_limbs(d.v, s.v, q);
    return bw ? s : d;
}
PG_HD Fr fr_sub(const Fr& a, const Fr& b) {
    Fr d, e; const uint32_t q[8] = {PG_Q0, PG_Q1, PG_Q2, PG_Q3, PG_Q4, PG_Q5, PG_Q6, PG_Q7};
    uint32_t bw = fr_sub_limbs(d.v, a.v, b.v);
    if (!bw) return d;
    fr_add_limbs(e.v, d.v, q);
    return e;
}
#endif
PG_HD Fr fr_neg(const Fr& a) { return fr_sub(fr_zero(), a); }   // q - a, and 0 for a == 0 (0 - 0 does not borrow)

// conditional final subtraction: t in [0, 2q) -> [0, q)
#if defined(__CUDA_ARCH__)
PG_D Fr fr_reduce_once(const Fr& t) {
    Fr d; uint32_t bw;
    asm("sub.cc.u32 %0, %9, %17;\n\tsubc.cc.u32 %1, %10, %18;\n\tsubc.cc.u32 %2, %11, %19;\n\tsubc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\tsubc.cc.u32 %5, %14, %22;\n\tsubc.cc.u32 %6, %15, %23;\n\tsubc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=&r"(d.v[0]), "=&r"(d.v[1]), "=&r"(d.v[2]), "=&r"(d.v[3]), "=&r"(d.v[4]), "=&r"(d.v[5]), "=&r"(d.v[6]), "=&r"(d.v[7]), "=&r"(bw)
        : "r"(t.v[0]), "r"(t.v[1]), "r"(t.v[2]), "r"(t.v[3]), "r"(t.v[4]), "r"(t.v[5]), "r"(t.v[6]), "r"(t.v[7]),
          "r"(PG_Q0), "r"(PG_Q1), "r"(PG_Q2), "r"(PG_Q3), "r"(PG_Q4), "r"(PG_Q5), "r"(PG_Q6), "r"(PG_Q7));
#pragma unroll
    for (int i = 0; i < 8; i++) d.v[i] = bw ? t.v[i] : d.v[i];
    return d;
}
#else
PG_HD Fr fr_reduce_once(const Fr& t) {
    Fr d; const uint32_t q[8] = {PG_Q0, PG_Q1, PG_Q2, PG_Q3, PG_Q4, PG_Q5, PG_Q6, PG_Q7};
    uint32_t bw = fr_sub_limbs(d.v, t.v, q);
    Fr r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = bw ? t.v[i] : d.v[i];
    return r;
}
#endif

// ---- portable CIOS Montgomery multiplication (host + device) --------------------------------------------------------
PG_HD Fr fr_mul_cios(const Fr& a, const Fr& b) {
    uint32_t t[10];
#pragma unroll
    for (int i = 0; i < 10; i++) t[i] = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint64_t c = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) { uint64_t s = (uint64_t)a.v[j] * b.v[i] + t[j] + c; t[j] = (uint32_t)s; c = s >> 32; }
        uint64_t s = (uint64_t)t[8] + c; t[8] = (uint32_t)s; t[9] = (uint32_t)(s >> 32);
        uint32_t m = 0u - t[0];                                   // t0 * (-q^-1 mod 2^32), q^-1 = 1 mod 2^32
        c = ((uint64_t)m * PG_Q0 + t[0]) >> 32;
#pragma unroll
        for (int j = 1; j < 8; j++) { uint64_t u = (uint64_t)m * fr_q(j) + t[j] + c; t[j - 1] = (uint32_t)u; c = u >> 32; }
        s = (uint64_t)t[8] + c; t[7] = (uint32_t)s; t[8] = t[9] + (uint32_t)(s >> 32);
    }
    Fr r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = t[i];
    return fr_reduce_once(r);                                     // t[8] == 0 here because the running value stays < 2q
}

// m = -t0 mod 2^32 (t0 * q' with q' = 2^32 - 1).  On the device the negation is kept inside an asm statement: when the
// compiler can see `0 - x` feeding the reduction rows it breaks every IMAD.WIDE.U32.X of the row into IMAD.X + IMAD.HI.U32.X
// (6 multiplier-pipe cycles per product instead of 4; found in SASS, see profiles/README.md).
PG_HD uint32_t mont_m(uint32_t t0) {
#if defined(__CUDA_ARCH__)
    uint32_t m;
    asm("sub.u32 %0, 0, %1;" : "=r"(m) : "r"(t0));
    return m;
#else
    return 0u - t0;
#endif
}

// ---- even/odd carry-chain primitives -------------------------------------------------------------------------------
// Each primitive is ONE asm statement holding ONE complete carry chain, so the condition-code register never has to
// survive between statements.  Host versions emulate the same dataflow with 64-bit arithmetic (tests/emu).
//
// chain A ("first row"):      acc[j],acc[j+1] = lo,hi(x[j]*y)                     j = 0,2,4,6
// chain B ("accumulate row"): acc[j],acc[j+1] += lo,hi(x[j]*y) with carry ripple  j = 0,2,4,6 ; top += carry_out
// chain C ("shifted row"):    e0 += y1 ; new o[j],o[j+1] = lo,hi(x[j]*y) + old o[j+2],o[j+3] + ripple (old o[8],o[9] = 0)
#if defined(__CUDA_ARCH__)
PG_D void mul_row(uint32_t* acc, uint32_t x0, uint32_t x2, uint32_t x4, uint32_t x6, uint32_t y) {
    asm("mul.lo.u32 %0, %8, %12;\n\tmul.hi.u32 %1, %8, %12;\n\tmul.lo.u32 %2, %9, %12;\n\tmul.hi.u32 %3, %9, %12;\n\t"
        "mul.lo.u32 %4, %10, %12;\n\tmul.hi.u32 %5, %10, %12;\n\tmul.lo.u32 %6, %11, %12;\n\tmul.hi.u32 %7, %11, %12;"
        : "=&r"(acc[0]), "=&r"(acc[1]), "=&r"(acc[2]), "=&r"(acc[3]), "=&r"(acc[4]), "=&r"(acc[5]), "=&r"(acc[6]), "=&r"(acc[7])
        : "r"(x0), "r"(x2), "r"(x4), "r"(x6), "r"(y));
}
// acc += (x0,x2,x4,x6 at limbs 0,2,4,6) * y ; top += carry out of acc[7]
PG_D void mad_row(uint32_t* acc, uint32_t& top, uint32_t x0, uint32_t x2, uint32_t x4, uint32_t x6, uint32_t y) {
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\tmadc.hi.cc.u32 %1, %9, %13, %1;\n\tmadc.lo.cc.u32 %2, %10, %13, %2;\n\tmadc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\tmadc.hi.cc.u32 %5, %11, %13, %5;\n\tmadc.lo.cc.u32 %6, %12, %13, %6;\n\tmadc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(top)
        : "r"(x0), "r"(x2), "r"(x4), "r"(x6), "r"(y));
}
// same, carry out of acc[7] known to be zero (dropped)
PG_D void mad_row_nc(uint32_t* acc, uint32_t x0, uint32_t x2, uint32_t x4, uint32_t x6, uint32_t y) {
    asm("mad.lo.cc.u32 %0, %8, %12, %0;\n\tmadc.hi.cc.u32 %1, %8, %12, %1;\n\tmadc.lo.cc.u32 %2, %9, %12, %2;\n\tmadc.hi.cc.u32 %3, %9, %12, %3;\n\t"
        "madc.lo.cc.u32 %4, %10, %12, %4;\n\tmadc.hi.cc.u32 %5, %10, %12, %5;\n\tmadc.lo.cc.u32 %6, %11, %12, %6;\n\tmadc.hi.u32 %7, %11, %12, %7;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7])
        : "r"(x0), "r"(x2), "r"(x4), "r"(x6), "r"(y));
}
// e0 += o[1]; o <- (o >> 2 limbs) + (x0,x2,x4,x6)*y with the carry of the first add rippling in
PG_D void mad_row_shift(uint32_t* o, uint32_t& e0, uint32_t x0, uint32_t x2, uint32_t x4, uint32_t x6, uint32_t y) {
    asm("add.cc.u32 %8, %8, %1;\n\t"
        "madc.lo.cc.u32 %0, %9, %13, %2;\n\tmadc.hi.cc.u32 %1, %9, %13, %3;\n\tmadc.lo.cc.u32 %2, %10, %13, %4;\n\tmadc.hi.cc.u32 %3, %10, %13, %5;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %6;\n\tmadc.hi.cc.u32 %5, %11, %13, %7;\n\tmadc.lo.cc.u32 %6, %12, %13, 0;\n\tmadc.hi.u32 %7, %12, %13, 0;"
        : "+r"(o[0]), "+r"(o[1]), "+r"(o[2]), "+r"(o[3]), "+r"(o[4]), "+r"(o[5]), "+r"(o[6]), "+r"(o[7]), "+r"(e0)
        : "r"(x0), "r"(x2), "r"(x4), "r"(x6), "r"(y));
}
// r[i] = e[i] + o[i+1] (i = 0..6), r[7] = e[7] + carry
PG_D void merge_even_odd(uint32_t* r, const uint32_t* e, const uint32_t* o) {
    asm("add.cc.u32 %0, %8, %16;\n\taddc.cc.u32 %1, %9, %17;\n\taddc.cc.u32 %2, %10, %18;\n\taddc.cc.u32 %3, %11, %19;\n\t"
        "addc.cc.u32 %4, %12, %20;\n\taddc.cc.u32 %5, %13, %21;\n\taddc.cc.u32 %6, %14, %22;\n\taddc.u32 %7, %15, 0;"
        : "=&r"(r[0]), "=&r"(r[1]), "=&r"(r[2]), "=&r"(r[3]), "=&r"(r[4]), "=&r"(r[5]), "=&r"(r[6]), "=&r"(r[7])
        : "r"(e[0]), "r"(e[1]), "r"(e[2]), "r"(e[3]), "r"(e[4]), "r"(e[5]), "r"(e[6]), "r"(e[7]),
          "r"(o[1]), "r"(o[2]), "r"(o[3]), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]));
}
#else
inline void mul_row(uint32_t* acc, uint32_t x0, uint32_t x2, uint32_t x4, uint32_t x6, uint32_t y) {
    const uint32_t x[4] = {x0, x2, x4, x6};
    for (int j = 0; j < 4; j++) { uint64_t p = (uint64_t)x[j] * y; acc[2 * j] = (uint32_t)p; acc[2 * j + 1] = (uint32_t)(p >> 32); }
}
inline uint32_t emu_mad_chain(uint32_t* acc, const uint32_t* x, uint32_t y, uint32_t cin) {
    uint32_t c = cin;
    for (int j = 0; j < 4; j++) {
        uint64_t p = (uint64_t)x[j] * y;
        uint64_t lo = (uint64_t)acc[2 * j] + (uint32_t)p + c; acc[2 * j] = (uint32_t)lo; c = (uint32_t)(lo >> 32);
        uint64_t hi = (uint64_t)acc[2 * j + 1] + (uint32_t)(p >> 32) + c; acc[2 * j + 1] = (uint32_t)hi; c = (uint32_t)(hi >> 32);
    }
    return c;
}
inline void mad_row(uint32_t* acc, uint32_t& top, uint32_t x0, uint32_t x2, uint32_t x4, uint32_t x6, uint32_t y) {
    const uint32_t x[4] = {x0, x2, x4, x6};
    uint32_t c = emu_mad_chain(acc, x, y, 0);
    if (top + c < top) PG_EMU_VIOLATION();   // the limb above must absorb the carry
    top += c;
}
inline void mad_row_nc(uint32_t* acc, uint32_t x0, uint32_t x2, uint32_t x4, uint32_t x6, uint32_t y) {
    const uint32_t x[4] = {x0, x2, x4, x6};
    uint32_t c = emu_mad_chain(acc, x, y, 0);
    if (c) PG_EMU_VIOLATION();   // tests/emu: the dropped carry must be 0
}
inline void mad_row_shift(uint32_t* o, uint32_t& e0, uint32_t x0, uint32_t x2, uint32_t x4, uint32_t x6, uint32_t y) {
    const uint32_t x[4] = {x0, x2, x4, x6};
    uint64_t s = (uint64_t)e0 + o[1]; e0 = (uint32_t)s; uint32_t c = (uint32_t)(s >> 32);
    uint32_t sh[8] = {o[2], o[3], o[4], o[5], o[6], o[7], 0, 0};
    c = emu_mad_chain(sh, x, y, c);
    if (c) PG_EMU_VIOLATION();
    for (int i = 0; i < 8; i++) o[i] = sh[i];
}
inline void merge_even_odd(uint32_t* r, const uint32_t* e, const uint32_t* o) {
    uint64_t c = 0;
    for (int i = 0; i < 7; i++) { uint64_t s = (uint64_t)e[i] + o[i + 1] + c; r[i] = (uint32_t)s; c = s >> 32; }
    if ((uint64_t)e[7] + c > 0xffffffffull) PG_EMU_VIOLATION();   // the result must fit 256 bits
    r[7] = e[7] + (uint32_t)c;
}
#endif

// One operand-scanning step: (X | Y) hold T = sum X[j] 2^(32j) + sum Y[j] 2^(32(j+1)).  Adds a*bi, then m*q with
// m = -T[0], leaving X[0] == 0; the caller swaps the roles of X and Y for the next step (division by 2^32).
// reduction rows of one step for m = -X[0]:  Y += m*(q1,q3,q5,q7) (m*q1 = (m << 32) - m by the adder, no carry out of Y[7]
// because q7 < 2^31),  X += m*(q0,q2,q4,q6) (m*q0 = m), carry -> Y[7]
#if defined(__CUDA_ARCH__)
PG_D void red_rows(uint32_t* X, uint32_t* Y, const QRegs& q) {
    const uint32_t m = mont_m(X[0]);
    uint32_t lo, hi;
    asm("sub.cc.u32 %0, 0, %2;\n\tsubc.u32 %1, %2, 0;" : "=&r"(lo), "=&r"(hi) : "r"(m));
    asm("add.cc.u32 %0, %0, %8;\n\taddc.cc.u32 %1, %1, %9;\n\tmadc.lo.cc.u32 %2, %10, %13, %2;\n\tmadc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\tmadc.hi.cc.u32 %5, %11, %13, %5;\n\tmadc.lo.cc.u32 %6, %12, %13, %6;\n\tmadc.hi.u32 %7, %12, %13, %7;"
        : "+r"(Y[0]), "+r"(Y[1]), "+r"(Y[2]), "+r"(Y[3]), "+r"(Y[4]), "+r"(Y[5]), "+r"(Y[6]), "+r"(Y[7])
        : "r"(lo), "r"(hi), "r"(q.v[3]), "r"(q.v[5]), "r"(q.v[7]), "r"(m));
    asm("add.cc.u32 %0, %0, %12;\n\taddc.cc.u32 %1, %1, 0;\n\tmadc.lo.cc.u32 %2, %9, %12, %2;\n\tmadc.hi.cc.u32 %3, %9, %12, %3;\n\t"
        "madc.lo.cc.u32 %4, %10, %12, %4;\n\tmadc.hi.cc.u32 %5, %10, %12, %5;\n\tmadc.lo.cc.u32 %6, %11, %12, %6;\n\tmadc.hi.cc.u32 %7, %11, %12, %7;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+r"(X[0]), "+r"(X[1]), "+r"(X[2]), "+r"(X[3]), "+r"(X[4]), "+r"(X[5]), "+r"(X[6]), "+r"(X[7]), "+r"(Y[7])
        : "r"(q.v[2]), "r"(q.v[4]), "r"(q.v[6]), "r"(m));
}
#else
inline void red_rows(uint32_t* X, uint32_t* Y, const QRegs& q) {
    const uint32_t m = mont_m(X[0]);
    mad_row_nc(Y, q.v[1], q.v[3], q.v[5], q.v[7], m);
    mad_row(X, Y[7], q.v[0], q.v[2], q.v[4], q.v[6], m);
}
#endif
PG_HD void mont_step_first(uint32_t* X, uint32_t* Y, const uint32_t* a, uint32_t bi, const QRegs& q) {
    mul_row(Y, a[1], a[3], a[5], a[7], bi);
    mul_row(X, a[0], a[2], a[4], a[6], bi);
    red_rows(X, Y, q);
}
PG_HD void mont_step(uint32_t* X, uint32_t* Y, const uint32_t* a, uint32_t bi, const QRegs& q) {
    mad_row_shift(Y, X[0], a[1], a[3], a[5], a[7], bi);       // X[0] += Y[1]; Y = (Y >> 64) + a_odd*bi
    mad_row(X, Y[7], a[0], a[2], a[4], a[6], bi);
    red_rows(X, Y, q);
}

PG_HD Fr fr_mul_eo(const Fr& a, const Fr& b, const QRegs& q) {
    uint32_t even[8], odd[8];
    mont_step_first(even, odd, a.v, b.v[0], q);
    mont_step(odd, even, a.v, b.v[1], q);
    mont_step(even, odd, a.v, b.v[2], q);
    mont_step(odd, even, a.v, b.v[3], q);
    mont_step(even, odd, a.v, b.v[4], q);
    mont_step(odd, even, a.v, b.v[5], q);
    mont_step(even, odd, a.v, b.v[6], q);
    mont_step(odd, even, a.v, b.v[7], q);
    Fr r;
    merge_even_odd(r.v, even, odd);                           // (even + odd>>32), odd[0] == 0
    return fr_reduce_once(r);
}
PG_HD Fr fr_mul_eo(const Fr& a, const Fr& b) { return fr_mul_eo(a, b, q_regs_default()); }

// ---- dot-product Montgomery: sum_p a_p*b_p with ONE interleaved reduction ----------------------------------------------
// The gate equation needs q_m*(ab) + q_l*a + q_r*b + q_o*c + q_4*d only up to "is it 0 mod q", so the five double-width
// products are accumulated into one running value that is reduced once per limb step (operand scanning over the b_p limbs):
//     for i in 0..8:  T += sum_p a_p * b_p[i];  m = -T[0];  T += m*q;  T >>= 32
// 5*64 + 8*6 multiplier instructions instead of 5*(64+64).  T is held as an even array X (limbs 0..7), an odd array Y
// (limbs 1..8) and a top word Z (limb 9): with K products T stays below (K+1)*q*(2^32+1) < 2^320, every carry out of limb 7
// or 8 is caught (X -> Y[7] -> Z, Y -> Z).  The reduction rows use the shape of q: q0 = 1 (m*q0 = m) and q1 = 2^32-1
// (m*q1 = m*2^32 - m) need no multiplier.  Result: 9 limbs r < (K+1)*q + small, congruent to sum_p a_p*b_p / 2^256 mod q.
#if defined(__CUDA_ARCH__)
// X[0..7] += (x0,x2,x4,x6)*y ; carry -> y7 -> z
PG_D void dmad_row_x(uint32_t* X, uint32_t& y7, uint32_t& z, uint32_t x0, uint32_t x2, uint32_t x4, uint32_t x6, uint32_t y) {
    asm("mad.lo.cc.u32 %0, %10, %14, %0;\n\tmadc.hi.cc.u32 %1, %10, %14, %1;\n\tmadc.lo.cc.u32 %2, %11, %14, %2;\n\tmadc.hi.cc.u32 %3, %11, %14, %3;\n\t"
        "madc.lo.cc.u32 %4, %12, %14, %4;\n\tmadc.hi.cc.u32 %5, %12, %14, %5;\n\tmadc.lo.cc.u32 %6, %13, %14, %6;\n\tmadc.hi.cc.u32 %7, %13, %14, %7;\n\t"
        "addc.cc.u32 %8, %8, 0;\n\taddc.u32 %9, %9, 0;"
        : "+r"(X[0]), "+r"(X[1]), "+r"(X[2]), "+r"(X[3]), "+r"(X[4]), "+r"(X[5]), "+r"(X[6]), "+r"(X[7]), "+r"(y7), "+r"(z)
        : "r"(x0), "r"(x2), "r"(x4), "r"(x6), "r"(y));
}
// Y[0..7] += (x1,x3,x5,x7)*y ; carry -> z
PG_D void dmad_row_y(uint32_t* Y, uint32_t& z, uint32_t x1, uint32_t x3, uint32_t x5, uint32_t x7, uint32_t y) {
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\tmadc.hi.cc.u32 %1, %9, %13, %1;\n\tmadc.lo.cc.u32 %2, %10, %13, %2;\n\tmadc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\tmadc.hi.cc.u32 %5, %11, %13, %5;\n\tmadc.lo.cc.u32 %6, %12, %13, %6;\n\tmadc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+r"(Y[0]), "+r"(Y[1]), "+r"(Y[2]), "+r"(Y[3]), "+r"(Y[4]), "+r"(Y[5]), "+r"(Y[6]), "+r"(Y[7]), "+r"(z)
        : "r"(x1), "r"(x3), "r"(x5), "r"(x7), "r"(y));
}
// division by 2^32 fused with the first odd row of the next step:
//   e0 += o[1];  o <- (o >> 2 limbs | z at the top) + (x1,x3,x5,x7)*y ;  z <- carry
PG_D void dmad_row_shift(uint32_t* o, uint32_t& e0, uint32_t& z, uint32_t x1, uint32_t x3, uint32_t x5, uint32_t x7, uint32_t y) {
    asm("add.cc.u32 %8, %8, %1;\n\t"
        "madc.lo.cc.u32 %0, %10, %14, %2;\n\tmadc.hi.cc.u32 %1, %10, %14, %3;\n\tmadc.lo.cc.u32 %2, %11, %14, %4;\n\tmadc.hi.cc.u32 %3, %11, %14, %5;\n\t"
        "madc.lo.cc.u32 %4, %12, %14, %6;\n\tmadc.hi.cc.u32 %5, %12, %14, %7;\n\tmadc.lo.cc.u32 %6, %13, %14, 0;\n\tmadc.hi.cc.u32 %7, %13, %14, %9;\n\t"
        "addc.u32 %9, 0, 0;"
        : "+r"(o[0]), "+r"(o[1]), "+r"(o[2]), "+r"(o[3]), "+r"(o[4]), "+r"(o[5]), "+r"(o[6]), "+r"(o[7]), "+r"(e0), "+r"(z)
        : "r"(x1), "r"(x3), "r"(x5), "r"(x7), "r"(y));
}
// reduction rows for m = -X[0]:  Y += m*(q1,q3,q5,q7) with m*q1 = (m<<32) - m done by the adder;  X += m*(q0,q2,q4,q6) with m*q0 = m
PG_D void dred_rows(uint32_t* X, uint32_t* Y, uint32_t& z, const QRegs& q) {
    const uint32_t m = mont_m(X[0]);
    uint32_t lo, hi;
    asm("sub.cc.u32 %0, 0, %2;\n\tsubc.u32 %1, %2, 0;" : "=&r"(lo), "=&r"(hi) : "r"(m));            // m*(2^32-1) = hi:lo
    asm("add.cc.u32 %0, %0, %9;\n\taddc.cc.u32 %1, %1, %10;\n\tmadc.lo.cc.u32 %2, %11, %14, %2;\n\tmadc.hi.cc.u32 %3, %11, %14, %3;\n\t"
        "madc.lo.cc.u32 %4, %12, %14, %4;\n\tmadc.hi.cc.u32 %5, %12, %14, %5;\n\tmadc.lo.cc.u32 %6, %13, %14, %6;\n\tmadc.hi.cc.u32 %7, %13, %14, %7;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+r"(Y[0]), "+r"(Y[1]), "+r"(Y[2]), "+r"(Y[3]), "+r"(Y[4]), "+r"(Y[5]), "+r"(Y[6]), "+r"(Y[7]), "+r"(z)
        : "r"(lo), "r"(hi), "r"(q.v[3]), "r"(q.v[5]), "r"(q.v[7]), "r"(m));
    asm("add.cc.u32 %0, %0, %13;\n\taddc.cc.u32 %1, %1, 0;\n\tmadc.lo.cc.u32 %2, %10, %13, %2;\n\tmadc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\tmadc.hi.cc.u32 %5, %11, %13, %5;\n\tmadc.lo.cc.u32 %6, %12, %13, %6;\n\tmadc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.cc.u32 %8, %8, 0;\n\taddc.u32 %9, %9, 0;"
        : "+r"(X[0]), "+r"(X[1]), "+r"(X[2]), "+r"(X[3]), "+r"(X[4]), "+r"(X[5]), "+r"(X[6]), "+r"(X[7]), "+r"(Y[7]), "+r"(z)
        : "r"(q.v[2]), "r"(q.v[4]), "r"(q.v[6]), "r"(m));
}
// r[0..8] = (X >> 32) + Y + (z << 256)
PG_D void dmerge(uint32_t* r, const uint32_t* X, const uint32_t* Y, uint32_t z) {
    asm("add.cc.u32 %0, %9, %17;\n\taddc.cc.u32 %1, %10, %18;\n\taddc.cc.u32 %2, %11, %19;\n\taddc.cc.u32 %3, %12, %20;\n\t"
        "addc.cc.u32 %4, %13, %21;\n\taddc.cc.u32 %5, %14, %22;\n\taddc.cc.u32 %6, %15, %23;\n\taddc.cc.u32 %7, %16, 0;\n\taddc.u32 %8, %24, 0;"
        : "=&r"(r[0]), "=&r"(r[1]), "=&r"(r[2]), "=&r"(r[3]), "=&r"(r[4]), "=&r"(r[5]), "=&r"(r[6]), "=&r"(r[7]), "=&r"(r[8])
        : "r"(Y[0]), "r"(Y[1]), "r"(Y[2]), "r"(Y[3]), "r"(Y[4]), "r"(Y[5]), "r"(Y[6]), "r"(Y[7]),
          "r"(X[1]), "r"(X[2]), "r"(X[3]), "r"(X[4]), "r"(X[5]), "r"(X[6]), "r"(X[7]), "r"(z));
}
// r[0..8] += a[0..7]   (no carry out of limb 8 by the bound on r)
PG_D void add9_fr(uint32_t* r, const Fr& a) {
    asm("add.cc.u32 %0, %0, %9;\n\taddc.cc.u32 %1, %1, %10;\n\taddc.cc.u32 %2, %2, %11;\n\taddc.cc.u32 %3, %3, %12;\n\t"
        "addc.cc.u32 %4, %4, %13;\n\taddc.cc.u32 %5, %5, %14;\n\taddc.cc.u32 %6, %6, %15;\n\taddc.cc.u32 %7, %7, %16;\n\taddc.u32 %8, %8, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8])
        : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]));
}
// r[0..8] -= a[0..7]   (the caller keeps r >= a: SparseProgBody starts every row at 7q)
PG_D void sub9_fr(uint32_t* r, const Fr& a) {
    asm("sub.cc.u32 %0, %0, %9;\n\tsubc.cc.u32 %1, %1, %10;\n\tsubc.cc.u32 %2, %2, %11;\n\tsubc.cc.u32 %3, %3, %12;\n\t"
        "subc.cc.u32 %4, %4, %13;\n\tsubc.cc.u32 %5, %5, %14;\n\tsubc.cc.u32 %6, %6, %15;\n\tsubc.cc.u32 %7, %7, %16;\n\tsubc.u32 %8, %8, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8])
        : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]));
}
#else
inline void dmad_row_x(uint32_t* X, uint32_t& y7, uint32_t& z, uint32_t x0, uint32_t x2, uint32_t x4, uint32_t x6, uint32_t y) {
    const uint32_t x[4] = {x0, x2, x4, x6};
    const uint32_t c = emu_mad_chain(X, x, y, 0);
    const uint64_t s = (uint64_t)y7 + c; y7 = (uint32_t)s;
    if (z + (uint32_t)(s >> 32) < z) PG_EMU_VIOLATION();
    z += (uint32_t)(s >> 32);
}
inline void dmad_row_y(uint32_t* Y, uint32_t& z, uint32_t x1, uint32_t x3, uint32_t x5, uint32_t x7, uint32_t y) {
    const uint32_t x[4] = {x1, x3, x5, x7};
    const uint32_t c = emu_mad_chain(Y, x, y, 0);
    if (z + c < z) PG_EMU_VIOLATION();
    z += c;
}
inline void dmad_row_shift(uint32_t* o, uint32_t& e0, uint32_t& z, uint32_t x1, uint32_t x3, uint32_t x5, uint32_t x7, uint32_t y) {
    const uint32_t x[4] = {x1, x3, x5, x7};
    if (o[0] != 0) PG_EMU_VIOLATION();                                  // the reduction must have cleared the lowest limb
    const uint64_t s = (uint64_t)e0 + o[1]; e0 = (uint32_t)s;
    uint32_t sh[8] = {o[2], o[3], o[4], o[5], o[6], o[7], 0, z};
    z = emu_mad_chain(sh, x, y, (uint32_t)(s >> 32));
    for (int i = 0; i < 8; i++) o[i] = sh[i];
}
inline void dred_rows(uint32_t* X, uint32_t* Y, uint32_t& z, const QRegs& q) {
    const uint32_t m = mont_m(X[0]);
    const uint32_t qo[4] = {q.v[1], q.v[3], q.v[5], q.v[7]}, qe[4] = {q.v[0], q.v[2], q.v[4], q.v[6]};
    uint32_t c = emu_mad_chain(Y, qo, m, 0);
    if (z + c < z) PG_EMU_VIOLATION();
    z += c;
    c = emu_mad_chain(X, qe, m, 0);
    const uint64_t s = (uint64_t)Y[7] + c; Y[7] = (uint32_t)s;
    if (z + (uint32_t)(s >> 32) < z) PG_EMU_VIOLATION();
    z += (uint32_t)(s >> 32);
}
inline void dmerge(uint32_t* r, const uint32_t* X, const uint32_t* Y, uint32_t z) {
    uint64_t c = 0;
    for (int i = 0; i < 7; i++) { const uint64_t s = (uint64_t)Y[i] + X[i + 1] + c; r[i] = (uint32_t)s; c = s >> 32; }
    const uint64_t s = (uint64_t)Y[7] + c; r[7] = (uint32_t)s;
    if ((uint64_t)z + (s >> 32) > 0xffffffffull) PG_EMU_VIOLATION();
    r[8] = z + (uint32_t)(s >> 32);
}
inline void add9_fr(uint32_t* r, const Fr& a) {
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) { const uint64_t s = (uint64_t)r[i] + a.v[i] + c; r[i] = (uint32_t)s; c = s >> 32; }
    if ((uint64_t)r[8] + c > 0xffffffffull) PG_EMU_VIOLATION();
    r[8] += (uint32_t)c;
}
inline void sub9_fr(uint32_t* r, const Fr& a) {
    uint64_t bw = 0;
    for (int i = 0; i < 8; i++) { const uint64_t d = (uint64_t)r[i] - a.v[i] - bw; r[i] = (uint32_t)d; bw = (d >> 32) & 1; }
    if (r[8] < bw) PG_EMU_VIOLATION();                                   // the accumulator must not go negative
    r[8] -= (uint32_t)bw;
}
#endif

// One limb step of the dot product for products p = 0..K-1: multiplicands a[p] (8 limbs), scanned limbs bi[p].
// (X | Y | z) as in mont_step; FIRST = the very first step (nothing to shift in).
template <int K, bool FIRST>
PG_HD void dot_step(uint32_t* X, uint32_t* Y, uint32_t& z, const Fr* a, const uint32_t* bi, const QRegs& q) {
    if (FIRST) {
        mul_row(Y, a[0].v[1], a[0].v[3], a[0].v[5], a[0].v[7], bi[0]);
        mul_row(X, a[0].v[0], a[0].v[2], a[0].v[4], a[0].v[6], bi[0]);
        z = 0;
    } else {
        dmad_row_shift(Y, X[0], z, a[0].v[1], a[0].v[3], a[0].v[5], a[0].v[7], bi[0]);   // X[0] += Y[1]; Y = (Y >> 64 | z) + a_odd*bi
        dmad_row_x(X, Y[7], z, a[0].v[0], a[0].v[2], a[0].v[4], a[0].v[6], bi[0]);
    }
#pragma unroll
    for (int p = 1; p < K; p++) {
        dmad_row_y(Y, z, a[p].v[1], a[p].v[3], a[p].v[5], a[p].v[7], bi[p]);
        dmad_row_x(X, Y[7], z, a[p].v[0], a[p].v[2], a[p].v[4], a[p].v[6], bi[p]);
    }
    dred_rows(X, Y, z, q);
}
// r[0..8] = (sum_p a[p]*b[p]) / 2^256 mod q up to a multiple of q:  r = (sum_p a[p]*b[p] + M*q) / 2^256 with M < 2^256, so
// r < q + sum_p a[p]*b[p] / 2^256  -- r < (K+1)*q for a[p] < q and any 256-bit b[p] (the generic row's u = q_m*b + q_l < 2q + 2^227),
// r < (2K+1)*q for a[p] < 2q, b[p] < 2q.
template <int K>
PG_HD void fr_dot_wide(uint32_t* r, const Fr* a, const Fr* b, const QRegs& q) {
    uint32_t even[8], odd[8], z, bi[K];
#define PG_DOT_STEP(I, XX, YY, FIRST)                          \
    _Pragma("unroll") for (int p = 0; p < K; p++) bi[p] = b[p].v[I]; \
    dot_step<K, FIRST>(XX, YY, z, a, bi, q);
    PG_DOT_STEP(0, even, odd, true)
    PG_DOT_STEP(1, odd, even, false)
    PG_DOT_STEP(2, even, odd, false)
    PG_DOT_STEP(3, odd, even, false)
    PG_DOT_STEP(4, even, odd, false)
    PG_DOT_STEP(5, odd, even, false)
    PG_DOT_STEP(6, even, odd, false)
    PG_DOT_STEP(7, odd, even, false)
#undef PG_DOT_STEP
    dmerge(r, odd, even, z);          // the last step cleared odd[0]: value = (odd >> 32) + even + (z << 256)
}
template <int K>
PG_HD void fr_dot_wide(uint32_t* r, const Fr* a, const Fr* b) { fr_dot_wide<K>(r, a, b, q_regs_default()); }

// ---- q_m*b with the reduction folded into per-selector constants -------------------------------------------------------
// For a selector s = q_m*R (Montgomery form) the host precomputes C[i] = q_m * 2^(32i+64) mod q, i = 0..7 (fr_fold_constants).
// For b as stored (any 256-bit value, limbs b[i])  U = sum_i b[i]*C[i]  is congruent to q_m*b*2^64: eight product rows at the same
// offset with no reduction between them (U < 8*2^32*q < 2^290: the ten limbs X | Y | z of the dot product).  Two Montgomery steps
// (m = -T[0], T += m*q, T >>= 32) leave  r == q_m*b == fr_mul_eo(s, b) (mod q)  with  r < q + 2^227:  8*8 + 2*6 = 76 wide products
// instead of fr_mul_eo's 112, and no conditional subtraction.  The result is NOT reduced.
#if defined(__CUDA_ARCH__)
// division by 2^32 between two reduction steps (o[0] == 0):  e0 += o[1];  o <- (o >> 2 limbs | z at the top), the odd array of the next step
PG_D void dshift_rows(uint32_t* o, uint32_t& e0, uint32_t z) {
    asm("add.cc.u32 %8, %8, %1;\n\taddc.cc.u32 %0, %2, 0;\n\taddc.cc.u32 %1, %3, 0;\n\taddc.cc.u32 %2, %4, 0;\n\taddc.cc.u32 %3, %5, 0;\n\t"
        "addc.cc.u32 %4, %6, 0;\n\taddc.cc.u32 %5, %7, 0;\n\taddc.u32 %6, 0, 0;"
        : "+r"(o[0]), "+r"(o[1]), "+r"(o[2]), "+r"(o[3]), "+r"(o[4]), "+r"(o[5]), "+r"(o[6]), "+r"(o[7]), "+r"(e0));
    o[7] = z;
}
// one 256-bit load of a fold constant (the table is 32-byte aligned and read-only while a kernel runs)
PG_D Fr fr_load_fold(const Fr* p) {
    Fr r;
    asm("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7]) : "l"(p));
    return r;
}
#else
inline void dshift_rows(uint32_t* o, uint32_t& e0, uint32_t z) {
    if (o[0] != 0) PG_EMU_VIOLATION();                                  // the reduction must have cleared the lowest limb
    const uint64_t s = (uint64_t)e0 + o[1]; e0 = (uint32_t)s;
    uint64_t c = s >> 32;
    for (int k = 0; k < 6; k++) { const uint64_t t = (uint64_t)o[k + 2] + c; o[k] = (uint32_t)t; c = t >> 32; }
    o[6] = (uint32_t)c; o[7] = z;
}
inline Fr fr_load_fold(const Fr* p) { return *p; }
#endif
// C[0..7] for the selector s (Montgomery form, < q): C[i] = mont(s, 2^(32i+64) mod q) = q_m * 2^(32i+64) mod q
PG_HD void fr_fold_constants(Fr* C, const Fr& s) {
    Fr p = {{0, 0, 1, 0, 0, 0, 0, 0}};                                     // 2^64 (a plain value below q)
    const Fr two32 = {{0, 1, 0, 0, 0, 0, 0, 0}};
    const Fr step = fr_mul_cios(two32, fr_r2());                           // 2^32*R: a Montgomery product with it multiplies by 2^32
    for (int i = 0; i < 8; i++) { C[i] = fr_mul_cios(s, p); p = fr_mul_cios(p, step); }
}
// r == s*b*R^-1 (mod q), r < q + 2^227, for the constants C = fr_fold_constants(s) (device: global memory) and any 256-bit b
PG_HD Fr fr_mul_folded(const Fr* C, const Fr& b, const QRegs& q) {
    uint32_t X[8], Y[8], z = 0;
    // One constant ahead: the address of C[p+1] is ORed with z >> 3, which is 0 (z < 8 after every row: U < 2^290) but not to ptxas, so
    // the load cannot be hoisted above row p-1.  Without it ptxas issues all eight loads early and k_check<0,0> spills at 96 registers.
    // (An OR on the low address word is one logic instruction; an added index would become an IMAD.WIDE on the multiplier pipe.)
    Fr c = fr_load_fold(C), cn = fr_load_fold(C + 1);
    mul_row(Y, c.v[1], c.v[3], c.v[5], c.v[7], b.v[0]);
    mul_row(X, c.v[0], c.v[2], c.v[4], c.v[6], b.v[0]);
#pragma unroll
    for (int p = 1; p < 8; p++) {
        c = cn;
        if (p < 7) cn = fr_load_fold(reinterpret_cast<const Fr*>(reinterpret_cast<uintptr_t>(C + p + 1) | (z >> 3)));
        dmad_row_y(Y, z, c.v[1], c.v[3], c.v[5], c.v[7], b.v[p]);
        dmad_row_x(X, Y[7], z, c.v[0], c.v[2], c.v[4], c.v[6], b.v[p]);
    }
    dred_rows(X, Y, z, q);             // T = U + m*q < 2^291
    dshift_rows(X, Y[0], z);           // T >>= 32 (< 2^259): Y even, X odd
    red_rows(Y, X, q);                 // T + m*q < 2^288: nothing leaves limb 8
    Fr r;
    merge_even_odd(r.v, X, Y);         // (X + Y>>32), Y[0] == 0
    return r;
}
// ---- the tensor-core part of the generic row: columns of the byte product -------------------------------------------------
// k_check_tc computes q_r*b + q_o*c + q_4*d (times R^-1, up to a multiple of q) as 32 s32 columns c[j] = sum over the 96 wire bytes
// of byte * (byte j of a byte-fold constant), c[j] <= 96*255*255 < 2^23, standing for L = sum_j c[j]*2^(8j) < 96*255*q.
// t[0..8] += L without a product:  P_k = c[4k] + (c[4k+1] << 8) and D_k = c[4k+2] + (c[4k+3] << 8) fit 32 bits, and
// L = sum_k P_k*2^(32k) + sum_k D_k*2^(32k+16), whose second sum has the limbs G_k = (D_k << 16) | (D_(k-1) >> 16):
// two 9-limb additions.
PG_HD void add_byte_columns(uint32_t* t, const uint32_t* c) {
    Fr P, G;
    uint32_t dprev = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
#if !defined(__CUDA_ARCH__)
        for (int j = 0; j < 4; j++) if (c[4 * k + j] >= (1u << 23)) PG_EMU_VIOLATION();   // the column bound the split relies on
#endif
#if defined(__CUDA_ARCH__)
        // x + (y << 8) written as a funnel shift: one LEA.HI on the integer ALU (as a shift and an add ptxas makes it an IMAD, which
        // would take the multiplier pipe the rest of the row is bound by)
        P.v[k] = c[4 * k] + __funnelshift_l(0u, c[4 * k + 1], 8);
        const uint32_t d = c[4 * k + 2] + __funnelshift_l(0u, c[4 * k + 3], 8);
        G.v[k] = __funnelshift_l(dprev, d, 16);
#else
        P.v[k] = c[4 * k] + (c[4 * k + 1] << 8);
        const uint32_t d = c[4 * k + 2] + (c[4 * k + 3] << 8);
        G.v[k] = (d << 16) | (dprev >> 16);
#endif
        dprev = d;
    }
    add9_fr(t, P);
    add9_fr(t, G);
#if !defined(__CUDA_ARCH__)
    if (t[8] + (dprev >> 16) < t[8]) PG_EMU_VIOLATION();
#endif
    t[8] += dprev >> 16;                                          // G_8
}
// t == 0 (mod q) for a 9-limb t < 2^15*q: since q = 1 (mod 2^32), t is a multiple of q iff t == k*q for k = t[0] < 2^15.
// k*q by eight wide products (k*q_i + carry is one IMAD.WIDE.U32 with a 64-bit addend each).
PG_HD bool limbs9_is_small_multiple_of_q(const uint32_t* t, const QRegs& q) {
    const uint32_t k = t[0] & 0x7fffu;
    uint32_t diff = t[0] >> 15;
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { c = (uint64_t)q.v[i] * k + (c >> 32); diff |= (uint32_t)c ^ t[i]; }
    diff |= (uint32_t)(c >> 32) ^ t[8];
    return diff == 0;
}
// plain 256-bit addition a + b (no reduction); the caller guarantees a + b < 2^256 (e.g. both < q)
PG_HD Fr fr_add_noreduce(const Fr& a, const Fr& b) {
    Fr r;
#if defined(__CUDA_ARCH__)
    asm("add.cc.u32 %0, %8, %16;\n\taddc.cc.u32 %1, %9, %17;\n\taddc.cc.u32 %2, %10, %18;\n\taddc.cc.u32 %3, %11, %19;\n\t"
        "addc.cc.u32 %4, %12, %20;\n\taddc.cc.u32 %5, %13, %21;\n\taddc.cc.u32 %6, %14, %22;\n\taddc.u32 %7, %15, %23;"
        : "=&r"(r.v[0]), "=&r"(r.v[1]), "=&r"(r.v[2]), "=&r"(r.v[3]), "=&r"(r.v[4]), "=&r"(r.v[5]), "=&r"(r.v[6]), "=&r"(r.v[7])
        : "r"(a.v[0]), "r"(a.v[1]), "r"(a.v[2]), "r"(a.v[3]), "r"(a.v[4]), "r"(a.v[5]), "r"(a.v[6]), "r"(a.v[7]),
          "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]), "r"(b.v[7]));
#else
    if (fr_add_limbs(r.v, a.v, b.v)) PG_EMU_VIOLATION();
#endif
    return r;
}
// a + t == b (mod q) for a, t, b < q, without reducing anything: s = a + t < 2q < 2^256, and s - b lies in (-q, 2q), so the
// congruence holds iff the 256-bit difference does not borrow and equals 0 or q (q0 = 1: the low limb tells which).
PG_HD bool fr_sum_equals(const Fr& a, const Fr& t, const Fr& b) {
    const Fr s = fr_add_noreduce(a, t);
    uint32_t d[8], bw;
#if defined(__CUDA_ARCH__)
    asm("sub.cc.u32 %0, %9, %17;\n\tsubc.cc.u32 %1, %10, %18;\n\tsubc.cc.u32 %2, %11, %19;\n\tsubc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\tsubc.cc.u32 %5, %14, %22;\n\tsubc.cc.u32 %6, %15, %23;\n\tsubc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=&r"(d[0]), "=&r"(d[1]), "=&r"(d[2]), "=&r"(d[3]), "=&r"(d[4]), "=&r"(d[5]), "=&r"(d[6]), "=&r"(d[7]), "=&r"(bw)
        : "r"(s.v[0]), "r"(s.v[1]), "r"(s.v[2]), "r"(s.v[3]), "r"(s.v[4]), "r"(s.v[5]), "r"(s.v[6]), "r"(s.v[7]),
          "r"(b.v[0]), "r"(b.v[1]), "r"(b.v[2]), "r"(b.v[3]), "r"(b.v[4]), "r"(b.v[5]), "r"(b.v[6]), "r"(b.v[7]));
#else
    bw = fr_sub_limbs(d, s.v, b.v);
#endif
    const uint32_t m = 0u - d[0];                      // d[0] == 1: all ones (compare with q); d[0] == 0: zero (compare with 0)
    uint32_t diff = bw | (d[0] >> 1);
    diff |= d[1] ^ (PG_Q1 & m); diff |= d[2] ^ (PG_Q2 & m); diff |= d[3] ^ (PG_Q3 & m); diff |= d[4] ^ (PG_Q4 & m);
    diff |= d[5] ^ (PG_Q5 & m); diff |= d[6] ^ (PG_Q6 & m); diff |= d[7] ^ (PG_Q7 & m);
    return diff == 0;
}
// k*q for k = 0..15 (9 limbs each): since q0 = 1, k*q = k (mod 2^32), so a 9-limb r is 0 mod q iff r == k*q for k = r[0] (r < 16q)
PG_HD bool limbs9_is_multiple_of_q(const uint32_t* r) {
    const uint32_t k = r[0];
    if (k > 15u) return false;
    const uint32_t q[8] = {PG_Q0, PG_Q1, PG_Q2, PG_Q3, PG_Q4, PG_Q5, PG_Q6, PG_Q7};
    uint32_t diff = 0; uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { const uint64_t t = (uint64_t)q[i] * k + c; diff |= (uint32_t)t ^ r[i]; c = t >> 32; }
    diff |= (uint32_t)c ^ r[8];
    return diff == 0;
}

#if defined(__CUDA_ARCH__)
PG_D Fr fr_mul(const Fr& a, const Fr& b) { return fr_mul_eo(a, b); }
#else
PG_HD Fr fr_mul(const Fr& a, const Fr& b) { return fr_mul_cios(a, b); }
#endif
PG_HD Fr fr_sqr(const Fr& a) { return fr_mul(a, a); }

// Montgomery form -> canonical integer limbs (BlsScalar::reduce / to_bytes): multiply by 1
PG_HD Fr fr_from_mont(const Fr& a) { Fr one = {{1, 0, 0, 0, 0, 0, 0, 0}}; return fr_mul(a, one); }
// canonical integer (< q) -> Montgomery form
PG_HD Fr fr_to_mont(const Fr& a) { return fr_mul(a, fr_r2()); }

// x^(q-2) with a 4-bit fixed window (255 squarings + <=64+14 multiplications).  x != 0.
PG_HD Fr fr_inv_fermat(const Fr& x) {
    const uint32_t e[8] = {0xffffffffu, 0xfffffffeu, 0xfffe5bfeu, 0x53bda402u, 0x09a1d805u, 0x3339d808u, 0x299d7d48u, 0x73eda753u};   // q - 2
    Fr tab[16];
    tab[0] = fr_one(); tab[1] = x;
#pragma unroll 1
    for (int i = 2; i < 16; i++) tab[i] = fr_mul(tab[i - 1], x);
    Fr r = fr_one();
#pragma unroll 1
    for (int w = 63; w >= 0; w--) {
        if (w != 63) { r = fr_sqr(r); r = fr_sqr(r); r = fr_sqr(r); r = fr_sqr(r); }
        uint32_t nib = (e[w >> 3] >> (4 * (w & 7))) & 0xf;
        if (nib) r = fr_mul(r, tab[nib]);
    }
    return r;
}

// The same inverse by the binary extended Euclidean algorithm (shifts, additions and subtractions only): about 370 short
// steps instead of 333 dependent multiplications -- a fifth of the instructions and of the latency of the Fermat chain, which
// is what the one-inversion-per-block step of the batch inversion waits on (kernels.cuh).  The inverse is unique, so the two
// functions return the same limbs (tests/test_emu_engine.py checks them against each other and against big ints).
// Variable time; meant for callers whose active lanes hold the SAME value (no divergence).  x != 0, Montgomery form in and out.
//   invariant:  s * x == u  and  t * x == v  (mod q), with x read as the integer it is stored as (x~ = x R);
//   u and v only lose bits; when they meet (u == v == gcd == 1) t is x~^-1, and one multiplication by R^3 puts it back in
//   Montgomery form:  mont(t, R^3) = x^-1 R^-1 * R^3 * R^-1 = x^-1 R.
PG_HD void fr_halve_mod_q(Fr& s) {          // s/2 mod q:  (s + q)/2 when s is odd (s + q < 2^256: both are below 2^255)
    const uint32_t odd = 0u - (s.v[0] & 1u);
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { c += (uint64_t)s.v[i] + (fr_q(i) & odd); s.v[i] = (uint32_t)c; c >>= 32; }
#pragma unroll
    for (int i = 0; i < 7; i++) s.v[i] = (s.v[i] >> 1) | (s.v[i + 1] << 31);
    s.v[7] >>= 1;
}
PG_HD Fr fr_inv_binary(const Fr& x) {
    Fr u = x, v, s = fr_zero(), t = fr_zero(), d;
    // 0 has no inverse (and would spin in the halving loop below): a caller that breaks the "x != 0" contract -- e.g. through an
    // unreduced table value equal to q, whose Montgomery product with anything is 0 -- gets 0 back, i.e. a wrong row, not a hung GPU.
    if (fr_is_zero(x)) return fr_zero();
#pragma unroll
    for (int i = 0; i < 8; i++) v.v[i] = fr_q(i);
    s.v[0] = 1;
    // every pass of the outer loop removes at least one bit from u + v (both below 2^256): 2*256 + 2 passes bound any input
#pragma unroll 1
    for (int pass = 0; pass < 2 * 256 + 2; pass++) {
#pragma unroll 1
        while (!(u.v[0] & 1u)) {
#pragma unroll
            for (int i = 0; i < 7; i++) u.v[i] = (u.v[i] >> 1) | (u.v[i + 1] << 31);
            u.v[7] >>= 1;
            fr_halve_mod_q(s);
        }
#pragma unroll 1
        while (!(v.v[0] & 1u)) {
#pragma unroll
            for (int i = 0; i < 7; i++) v.v[i] = (v.v[i] >> 1) | (v.v[i + 1] << 31);
            v.v[7] >>= 1;
            fr_halve_mod_q(t);
        }
        if (fr_sub_limbs(d.v, u.v, v.v)) {                    // u < v
            fr_sub_limbs(v.v, v.v, u.v);
            t = fr_sub(t, s);
        } else {
            u = d;
            if (fr_is_zero(u)) break;                         // u == v == 1
            s = fr_sub(s, t);
        }
    }
    return fr_mul(t, fr_r3());
}

}  // namespace pg
