// tests/emu/fold_emu.cpp -- host build of the folded q_m*b product of plonk_gadgets_b200/csrc/fr.cuh (TEST ONLY).
// fr_fold_constants / fr_mul_folded and the dot product they feed run through the carry-flag emulation, which counts every
// carry the device code drops (or adds into a limb assumed to have room) that is not zero.
#define PG_EMU_CHECKS 1
#include "../../plonk_gadgets_b200/csrc/fr.cuh"

static int g_violations = 0;
void pg_emu_carry_violation() { g_violations++; }

using pg::Fr;
extern "C" {
int emu_violations() { return g_violations; }
// C[8 * i .. 8 * i + 7] = fr_fold_constants(s[i])
void emu_fold_constants(uint64_t n, const Fr* s, Fr* C) { for (uint64_t i = 0; i < n; i++) pg::fr_fold_constants(C + 8 * i, s[i]); }
// u[i] = fr_mul_folded(constants of s[i], b[i]) + ql[i]  (the generic row's first dot-product operand, not reduced)
void emu_folded_u(uint64_t n, const Fr* s, const Fr* b, const Fr* ql, Fr* u) {
    for (uint64_t i = 0; i < n; i++) {
        Fr C[8];
        pg::fr_fold_constants(C, s[i]);
        u[i] = pg::fr_add_noreduce(pg::fr_mul_folded(C, b[i], pg::q_regs_default()), ql[i]);
    }
}
// r (9 limbs) = fr_dot_wide<4>(a[4i..4i+3], b[4i..4i+3])
void emu_dot4(uint64_t n, const Fr* a, const Fr* b, uint32_t* r9) { for (uint64_t i = 0; i < n; i++) pg::fr_dot_wide<4>(r9 + 9 * i, a + 4 * i, b + 4 * i); }
}
