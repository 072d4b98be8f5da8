/*
 * oracle/permutation.c -- CPU restatement of the permutation argument: preprocessing's sigma polynomials and round 2 of
 * `Prover::prove`, the grand-product polynomial z(X) (SURVEY.md section 8f item 2, continued).
 *
 * TEST INFRASTRUCTURE ONLY (see oracle/fr.h).  Built by tests/permutation_model.py into tests/oracle_perm/_build; it reads the
 * oracle's composer (oracle/composer.h: the wire columns and the perm.variable_map lists) and shares no code with the kernels.  PARITY STATUS: "parity unpinned".  Restated from dusk-plonk 0.8
 * src/permutation/permutation.rs as recalled (compute_sigma_permutations, compute_permutation_lagrange,
 * compute_fast_permutation_poly, compute_permutation_poly) and permutation/constants.rs (K1 = 7, K2 = 13, K3 = 17):
 *   * sigma starts as the identity on 4 x size wire positions; every Variable's positions, in the order the gates entered them
 *     into perm.variable_map, form one cycle (each position maps to the next, the last to the first); padding rows stay fixed;
 *   * the identity of (row i, wire w) is k_w * omega^i, k = (1, K1, K2, K3); sigma_w(omega^i) = identity of sigma(i, w);
 *   * z_0 = 1, z_{i+1} = z_i * prod_w (v + beta*k_w*omega^i + gamma) / prod_w (v + beta*sigma_w(omega^i) + gamma).
 * Written from the definitions, independently of the CUDA kernels: the variable map is the oracle composer's own linked lists,
 * powers of omega (the caller passes omega, from the oracle's orc_domain_group_gen) are a running product, and the denominators
 * are inverted with one Montgomery batch inversion.
 */
#include "../../oracle/composer.h"
#include <stdlib.h>

static int fr_iszero(const fr_t *a) { return !(a->l[0] | a->l[1] | a->l[2] | a->l[3]); }

/* sigma[w * size + i] = successor (row*4 + wire) of position (i, w) */
static void sigma_positions(const orc_composer *c, uint64_t size, uint64_t *sigma) {
    for (int w = 0; w < 4; w++)
        for (uint64_t i = 0; i < size; i++) sigma[(uint64_t)w * size + i] = i * 4 + (uint64_t)w;
    for (uint64_t v = 0; v < c->n_vars; v++) {        /* the lists run newest -> oldest: newest's successor is the oldest */
        uint64_t e = c->perm_head.p[v];
        if (!e) continue;
        const uint64_t newest = c->perm_data.p[e - 1];
        uint64_t later = newest;
        for (e = c->perm_next.p[e - 1]; e; e = c->perm_next.p[e - 1]) {
            const uint64_t pos = c->perm_data.p[e - 1];
            sigma[(pos & 3) * size + (pos >> 2)] = later;
            later = pos;
        }
        sigma[(newest & 3) * size + (newest >> 2)] = later;
    }
}

/* variables: the composer's n_vars values (orc_dump_variables); omega: generator of the domain of 2^log_n points.
 * sig_eval: 4 x size sigma evaluations (may be NULL), z: size evaluations, *closing: product of all ratios.
 * Returns -1 when 2^log_n < n or log_n > 32, 1 + row of the first zero denominator, or 0. */
int perm_oracle_z(const orc_composer *c, const fr_t *variables, unsigned log_n, const fr_t *omega, const fr_t *beta, const fr_t *gamma,
                  fr_t *sig_eval, fr_t *z, fr_t *closing) {
    if (log_n > 32 || (1ull << log_n) < c->n) return -1;
    const uint64_t size = 1ull << log_n;
    uint64_t *sigma = malloc(4 * size * sizeof(uint64_t));
    fr_t *pw = malloc(size * sizeof(fr_t)), *num = malloc(size * sizeof(fr_t)), *den = malloc(size * sizeof(fr_t));
    sigma_positions(c, size, sigma);
    pw[0] = fr_one();
    for (uint64_t i = 1; i < size; i++) pw[i] = fr_mul(&pw[i - 1], omega);
    fr_t bk[4];
    for (int w = 0; w < 4; w++) { static const uint64_t k[4] = {1, 7, 13, 17}; fr_t kw = fr_from_u64(k[w]); bk[w] = fr_mul(beta, &kw); }
    int rc = 0;
    for (uint64_t i = 0; i < size; i++) {
        fr_t n_i = fr_one(), d_i = fr_one();
        for (int w = 0; w < 4; w++) {
            const fr_t v = i < c->n ? variables[c->w[w].p[i]] : fr_zero();
            const uint64_t s = sigma[(uint64_t)w * size + i];
            fr_t t = fr_mul(&bk[w], &pw[i]); t = fr_add(&t, &v); t = fr_add(&t, gamma); n_i = fr_mul(&n_i, &t);
            fr_t kw = fr_from_u64(s % 4 == 0 ? 1 : s % 4 == 1 ? 7 : s % 4 == 2 ? 13 : 17), se = fr_mul(&kw, &pw[s >> 2]);
            if (sig_eval) sig_eval[(uint64_t)w * size + i] = se;
            fr_t u = fr_mul(beta, &se); u = fr_add(&u, &v); u = fr_add(&u, gamma); d_i = fr_mul(&d_i, &u);
        }
        if (fr_iszero(&d_i) && !rc) rc = (int)(i + 1);
        num[i] = n_i; den[i] = d_i;
    }
    if (!rc) {
        /* batch inversion: pw is reused for the running products of the denominators */
        fr_t acc = fr_one();
        for (uint64_t i = 0; i < size; i++) { pw[i] = acc; acc = fr_mul(&acc, &den[i]); }
        fr_t inv; fr_invert(&acc, &inv);
        for (uint64_t i = size; i-- > 0;) { const fr_t d_inv = fr_mul(&inv, &pw[i]); inv = fr_mul(&inv, &den[i]); den[i] = d_inv; }
        fr_t zz = fr_one();
        for (uint64_t i = 0; i < size; i++) { z[i] = zz; fr_t r = fr_mul(&num[i], &den[i]); zz = fr_mul(&zz, &r); }
        *closing = zz;
    }
    free(sigma); free(pw); free(num); free(den);
    return rc;
}
