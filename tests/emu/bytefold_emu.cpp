// tests/emu/bytefold_emu.cpp -- host build of the generic gate check's tensor-core row (TEST ONLY): the byte-fold blocks of
// plonk_gadgets_b200/csrc/layout.h, and the column merge and zero test of plonk_gadgets_b200/csrc/fr.cuh through the carry-flag
// emulation, which counts every carry the device code drops (or adds into a limb assumed to have room) that is not zero.  The
// MMA itself is modelled here by its definition: column j = sum over the 96 A bytes of A byte * B[k][j], B read through bf_offset.
#define PG_EMU_CHECKS 1
#include "../../plonk_gadgets_b200/csrc/layout.h"

static int g_violations = 0;
void pg_emu_carry_violation() { g_violations++; }

using pg::Fr;
extern "C" {
int emu_violations() { return g_violations; }
// blk[1024 * i ..] = byte_fold_block(s[i])
void emu_byte_fold_blocks(uint64_t n, const Fr* s, uint8_t* blk) { for (uint64_t i = 0; i < n; i++) pg::byte_fold_block(blk + 1024 * i, s[i]); }
// t9[9i ..] += columns c[32i ..]; ok[i] = limbs9_is_small_multiple_of_q(t9 after the addition)
void emu_add_columns(uint64_t n, uint32_t* t9, const uint32_t* c, uint8_t* ok) {
    for (uint64_t i = 0; i < n; i++) {
        pg::add_byte_columns(t9 + 9 * i, c + 32 * i);
        ok[i] = pg::limbs9_is_small_multiple_of_q(t9 + 9 * i, pg::q_regs_default());
    }
}
// One generic row as k_check_tc evaluates it: wires[4i ..] = a, b, c, d; sel[6i ..] = q_m, q_l, q_r, q_o, q_4 and q_c + PI (the two
// summed, below 2q).  The sum S (9 limbs) and the verdict come back.
void emu_generic_row(uint64_t n, const Fr* wires, const Fr* sel, uint32_t* S, uint8_t* ok) {
    for (uint64_t i = 0; i < n; i++) {
        const Fr* w = wires + 4 * i;        // a b c d
        const Fr* s = sel + 6 * i;
        Fr C[8];
        pg::fr_fold_constants(C, s[0]);
        const Fr u = pg::fr_add_noreduce(pg::fr_mul_folded(C, w[1], pg::q_regs_default()), s[1]);
        uint32_t* t = S + 9 * i;
        pg::fr_dot_wide<1>(t, w, &u);
        pg::add9_fr(t, s[5]);
        uint8_t B[3][1024];
        for (int k = 0; k < 3; k++) pg::byte_fold_block(B[k], s[2 + k]);
        uint32_t c[32];
        for (uint32_t j = 0; j < 32; j++) {
            uint32_t acc = 0;
            for (int k = 0; k < 3; k++)
                for (uint32_t kb = 0; kb < 32; kb++) acc += (uint32_t)((w[1 + k].v[kb >> 2] >> (8 * (kb & 3))) & 0xffu) * B[k][pg::bf_offset(j, kb)];
            c[j] = acc;
        }
        pg::add_byte_columns(t, c);
        ok[i] = pg::limbs9_is_small_multiple_of_q(t, pg::q_regs_default());
    }
}
}
