/*
 * tests/oracle_openings/openings.c -- CPU restatement of rounds 4 and 5 of `Prover::prove`: the evaluations at the challenge zeta,
 * the linearisation polynomial r(X) and the two opening witnesses W_zeta, W_zeta_w (SURVEY.md section 8f item 2, continued).
 *
 * TEST INFRASTRUCTURE ONLY (see oracle/fr.h).  Built by tests/opening_model.py into tests/oracle_openings/_build; it shares no code
 * with the kernels and works over coefficient vectors it is given (wires, z, sigma, selectors in the engine's QV order, t_1 .. t_4).
 * PARITY STATUS: "parity unpinned".  Restated from dusk-plonk 0.8 as recalled, keeping the crate's own operations (deliberately
 * not the engine's strided evaluation pass, fused combination or Ruffini scan):
 *   * Polynomial::evaluate: Horner from the top coefficient, one polynomial and one point at a time;
 *   * linearisation_poly::compute and the widgets' compute_linearisation: r as a sum of polynomials, each scaled by a scalar formed
 *     from the evaluations;
 *   * compute_quotient_opening_poly: t_1 + zeta^N t_2 + zeta^2N t_3 + zeta^3N t_4, scalar times polynomial and sums;
 *   * compute_aggregate_witness: sum_i challenge^i p_i, then Polynomial::ruffini: walk the coefficients from the top, push
 *     coeff + k and set k = point * (coeff + k), pop the last value (the remainder), reverse.
 */
#include "../../oracle/fr.h"
#include <stdlib.h>
#include <string.h>

enum { V_W = 0, V_Z = 4, V_S = 5, V_QM = 9, V_QL, V_QR, V_QO, V_Q4, V_QC, V_QARITH, V_QRANGE, V_N };

/* Polynomial::evaluate */
void open_evaluate(const fr_t *c, uint64_t n, const fr_t *x, fr_t *out) {
    fr_t acc = fr_zero();
    for (uint64_t i = n; i-- > 0;) { acc = fr_mul(&acc, x); acc = fr_add(&acc, &c[i]); }
    *out = acc;
}
/* Polynomial::ruffini: q has n coefficients, the last one zero (the n - 1 of the quotient, padded) */
void open_ruffini(const fr_t *f, uint64_t n, const fr_t *z, fr_t *q) {
    fr_t *quotient = malloc((n ? n : 1) * sizeof(fr_t));
    uint64_t len = 0;
    fr_t k = fr_zero();
    for (uint64_t i = n; i-- > 0;) { fr_t t = fr_add(&f[i], &k); quotient[len++] = t; k = fr_mul(z, &t); }
    if (len) len--;                                                  /* pop the remainder */
    for (uint64_t i = 0; i < len; i++) q[i] = quotient[len - 1 - i]; /* reverse */
    for (uint64_t i = len; i < n; i++) q[i] = fr_zero();
    free(quotient);
}
static void add_scaled(fr_t *acc, const fr_t *p, uint64_t n, const fr_t *s) {   /* acc += s * p */
    for (uint64_t i = 0; i < n; i++) { fr_t t = fr_mul(&p[i], s); acc[i] = fr_add(&acc[i], &t); }
}
static fr_t delta(const fr_t *f) {
    fr_t r = *f;
    for (uint64_t k = 1; k <= 3; k++) { fr_t kk = fr_from_u64(k), d = fr_sub(f, &kk); r = fr_mul(&r, &d); }
    return r;
}
static fr_t minus4(const fr_t *x, const fr_t *y) {                  /* x - 4y */
    fr_t f = fr_from_u64(4), t = fr_mul(&f, y);
    return fr_sub(x, &t);
}

/* vec: V_N coefficient vectors of n; t: 4 of n; ch: alpha beta gamma rho zeta v v'; omega generates the domain of n.
 * evals: 17 scalars in pg_proof_evaluations' order; dst: W_zeta, W_zeta_w, r (3 x n).  Returns -1 when zeta^n = 1, else 0. */
int open_oracle(const fr_t *vec, const fr_t *t, uint64_t n, const fr_t *ch, const fr_t *omega, fr_t *evals, fr_t *dst) {
    const fr_t *alpha = &ch[0], *beta = &ch[1], *gamma = &ch[2], *rho = &ch[3], *z = &ch[4], *v = &ch[5], *vs = &ch[6];
#define VEC(k) (vec + (uint64_t)(k) * n)
    fr_t zn = fr_one(), one = fr_one();
    for (uint64_t i = 0; i < n; i++) zn = fr_mul(&zn, z);
    if (fr_eq(&zn, &one)) return -1;
    fr_t zw = fr_mul(z, omega);
    fr_t a, b, c, d, aw, bw, dw, qa, qc, ql, qr, s1, s2, s3, perm;
    open_evaluate(VEC(V_W), n, z, &a); open_evaluate(VEC(V_W + 1), n, z, &b); open_evaluate(VEC(V_W + 2), n, z, &c); open_evaluate(VEC(V_W + 3), n, z, &d);
    open_evaluate(VEC(V_W), n, &zw, &aw); open_evaluate(VEC(V_W + 1), n, &zw, &bw); open_evaluate(VEC(V_W + 3), n, &zw, &dw);
    open_evaluate(VEC(V_QARITH), n, z, &qa); open_evaluate(VEC(V_QC), n, z, &qc); open_evaluate(VEC(V_QL), n, z, &ql); open_evaluate(VEC(V_QR), n, z, &qr);
    open_evaluate(VEC(V_S), n, z, &s1); open_evaluate(VEC(V_S + 1), n, z, &s2); open_evaluate(VEC(V_S + 2), n, z, &s3);
    open_evaluate(VEC(V_Z), n, &zw, &perm);
    /* compute_quotient_opening_poly */
    fr_t *quot = calloc(n, sizeof(fr_t));
    fr_t zp = fr_one();
    for (int r = 0; r < 4; r++) { add_scaled(quot, t + (uint64_t)r * n, n, &zp); zp = fr_mul(&zp, &zn); }
    fr_t quot_eval; open_evaluate(quot, n, z, &quot_eval);
    /* linearisation_poly::compute: arithmetic, range and permutation widgets */
    fr_t *lin = calloc(n, sizeof(fr_t));
    fr_t ab = fr_mul(&a, &b), w;
    w = fr_mul(&ab, &qa); add_scaled(lin, VEC(V_QM), n, &w);
    w = fr_mul(&a, &qa); add_scaled(lin, VEC(V_QL), n, &w);
    w = fr_mul(&b, &qa); add_scaled(lin, VEC(V_QR), n, &w);
    w = fr_mul(&c, &qa); add_scaled(lin, VEC(V_QO), n, &w);
    w = fr_mul(&d, &qa); add_scaled(lin, VEC(V_Q4), n, &w);
    add_scaled(lin, VEC(V_QC), n, &qa);
    fr_t kappa = fr_square(rho), kappa2 = fr_square(&kappa), kappa3 = fr_mul(&kappa2, &kappa), f, b1, b2, b3, b4;
    f = minus4(&c, &d); b1 = delta(&f);
    f = minus4(&b, &c); b2 = delta(&f); b2 = fr_mul(&b2, &kappa);
    f = minus4(&a, &b); b3 = delta(&f); b3 = fr_mul(&b3, &kappa2);
    f = minus4(&dw, &a); b4 = delta(&f); b4 = fr_mul(&b4, &kappa3);
    w = fr_add(&b1, &b2); w = fr_add(&w, &b3); w = fr_add(&w, &b4); w = fr_mul(&w, rho);
    add_scaled(lin, VEC(V_QRANGE), n, &w);
    static const uint64_t K[4] = {1, 7, 13, 17};
    const fr_t wv[4] = {a, b, c, d}, sv[3] = {s1, s2, s3};
    fr_t prod = fr_one(), prod_s = fr_one();
    for (int k = 0; k < 4; k++) {
        fr_t kk = fr_from_u64(K[k]), y = fr_mul(beta, &kk); y = fr_mul(&y, z); y = fr_add(&y, &wv[k]); y = fr_add(&y, gamma); prod = fr_mul(&prod, &y);
        if (k < 3) { fr_t q = fr_mul(beta, &sv[k]); q = fr_add(&q, &wv[k]); q = fr_add(&q, gamma); prod_s = fr_mul(&prod_s, &q); }
    }
    fr_t zh = fr_sub(&zn, &one), nf = fr_from_u64(n), zm1 = fr_sub(z, &one), den = fr_mul(&nf, &zm1), den_inv, l1, a2 = fr_square(alpha);
    fr_invert(&den, &den_inv); l1 = fr_mul(&zh, &den_inv);
    w = fr_mul(alpha, &prod); { fr_t u = fr_mul(&a2, &l1); w = fr_add(&w, &u); }
    add_scaled(lin, VEC(V_Z), n, &w);
    w = fr_mul(alpha, beta); w = fr_mul(&w, &perm); w = fr_mul(&w, &prod_s); w = fr_neg(&w);
    add_scaled(lin, VEC(V_S + 3), n, &w);
    fr_t lin_eval; open_evaluate(lin, n, z, &lin_eval);
    const fr_t ev[17] = {a, b, c, d, aw, bw, dw, qa, qc, ql, qr, s1, s2, s3, lin_eval, perm, quot_eval};
    memcpy(evals, ev, sizeof(ev));
    /* compute_aggregate_witness at zeta and at zeta*w */
    fr_t *agg = calloc(n, sizeof(fr_t));
    const fr_t *polys[9] = {quot, lin, VEC(V_W), VEC(V_W + 1), VEC(V_W + 2), VEC(V_W + 3), VEC(V_S), VEC(V_S + 1), VEC(V_S + 2)};
    fr_t pw = fr_one();
    for (int k = 0; k < 9; k++) { add_scaled(agg, polys[k], n, &pw); pw = fr_mul(&pw, v); }
    open_ruffini(agg, n, z, dst);
    memset(agg, 0, n * sizeof(fr_t));
    const fr_t *shifted[4] = {VEC(V_Z), VEC(V_W), VEC(V_W + 1), VEC(V_W + 3)};
    pw = fr_one();
    for (int k = 0; k < 4; k++) { add_scaled(agg, shifted[k], n, &pw); pw = fr_mul(&pw, vs); }
    open_ruffini(agg, n, &zw, dst + n);
    memcpy(dst + 2 * n, lin, n * sizeof(fr_t));
    free(agg); free(lin); free(quot);
#undef VEC
    return 0;
}
