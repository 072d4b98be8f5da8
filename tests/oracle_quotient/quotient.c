/*
 * tests/oracle_quotient/quotient.c -- CPU restatement of round 3 of `Prover::prove`, the quotient polynomial t(X)
 * (SURVEY.md section 8f item 2, continued).
 *
 * TEST INFRASTRUCTURE ONLY (see oracle/fr.h).  Built by tests/quotient_model.py into tests/oracle_quotient/_build together with
 * oracle/fft.c and oracle/composer.c; it reads the oracle's composer (oracle/composer.h) and shares no code with the kernels.
 * PARITY STATUS: "parity unpinned".  Restated from dusk-plonk 0.8 src/proof_system/quotient_poly.rs as recalled, keeping the
 * reference's own structure (deliberately not the engine's four size-N sub-cosets):
 *   * every component polynomial (wires, z, sigma, the selectors, PI; N coefficients) is evaluated on the whole coset g*<zeta> of
 *     the 4N domain by coset_fft (coefficient m times g^m, then one 4N-point transform), g = 7;
 *   * alpha^2 L_1 is coset_fft of compute_first_lagrange_poly_scaled(alpha^2) = ifft([alpha^2, 0, ..]) = alpha^2 / N everywhere;
 *   * "next" values are index i + 4 (mod 4N) of the same evaluation vector (omega = zeta^4);
 *   * the numerator is divided pointwise by v_h_coset_4n: x^N - 1 = g^N zeta^(iN) - 1, four values repeating;
 *   * coset_ifft (the 4N inverse transform, then coefficient m times g^-m) and split_tx_poly into four pieces of N.
 * z and the sigma evaluations come from tests/oracle_perm/permutation.c (perm_oracle_z).
 */
#include "../oracle_perm/permutation.c"
#include <string.h>

int orc_fft(fr_t *a, unsigned log_n, int inverse);
void orc_domain_group_gen(unsigned log_n, fr_t *out);

static void distribute_powers(fr_t *a, uint64_t n, const fr_t *g) {
    fr_t p = fr_one();
    for (uint64_t i = 0; i < n; i++) { a[i] = fr_mul(&a[i], &p); p = fr_mul(&p, g); }
}
static fr_t delta(const fr_t *f) {                  /* f (f - 1) (f - 2) (f - 3) */
    fr_t r = *f;
    for (uint64_t k = 1; k <= 3; k++) { fr_t kk = fr_from_u64(k), d = fr_sub(f, &kk); r = fr_mul(&r, &d); }
    return r;
}
static fr_t times4(const fr_t *x) { fr_t y = fr_add(x, x); return fr_add(&y, &y); }

enum { C_W = 0, C_Z = 4, C_S = 5, C_SEL = 9, C_PI = 17, C_L1 = 18, C_N = 19 };

/* variables: the composer's n_vars values; challenges: one Montgomery scalar each.  out: t_1 .. t_4, 4 x 2^log_n coefficients.
 * Returns -1 when 2^log_n < n or log_n > 30, 1 + row of the first zero z denominator, or 0. */
int quot_oracle_t(const orc_composer *c, const fr_t *variables, unsigned log_n, const fr_t *alpha, const fr_t *beta, const fr_t *gamma,
                  const fr_t *rho, fr_t *out) {
    if (log_n > 30 || (1ull << log_n) < c->n) return -1;
    const uint64_t n = 1ull << log_n, m = 4 * n;
    fr_t omega; orc_domain_group_gen(log_n, &omega);
    fr_t *coef = calloc((size_t)C_N * n, sizeof(fr_t));
    fr_t closing;
    int rc = perm_oracle_z(c, variables, log_n, &omega, beta, gamma, coef + (uint64_t)C_S * n, coef + (uint64_t)C_Z * n, &closing);
    if (rc) { free(coef); return rc; }
    fr_t *pi = malloc((c->n ? c->n : 1) * sizeof(fr_t));
    orc_dense_pi(c, pi);
    for (uint64_t i = 0; i < c->n; i++) {
        for (int w = 0; w < 4; w++) coef[(C_W + w) * n + i] = variables[c->w[w].p[i]];
        for (int k = 0; k < 8; k++) coef[(C_SEL + k) * n + i] = c->sel[k].p[i];
        coef[C_PI * n + i] = pi[i];
    }
    free(pi);
    for (int v = 0; v < C_L1; v++) orc_fft(coef + (uint64_t)v * n, log_n, 1);            /* padding rows are zero: domain.ifft */
    fr_t a2 = fr_square(alpha), n_fr = fr_from_u64(n), n_inv; fr_invert(&n_fr, &n_inv);
    const fr_t l1 = fr_mul(&a2, &n_inv);
    for (uint64_t i = 0; i < n; i++) coef[C_L1 * n + i] = l1;

    const fr_t g = fr_from_u64(7);
    fr_t *ev = calloc((size_t)C_N * m, sizeof(fr_t));
    for (int v = 0; v < C_N; v++) {                                                      /* domain_4n.coset_fft */
        fr_t *e = ev + (uint64_t)v * m;
        memcpy(e, coef + (uint64_t)v * n, n * sizeof(fr_t));
        distribute_powers(e, m, &g);
        orc_fft(e, log_n + 2, 0);
    }
    free(coef);
    fr_t zeta; orc_domain_group_gen(log_n + 2, &zeta);
    fr_t vh_inv[4], g_n = fr_one(), zeta_n = fr_one();
    for (uint64_t i = 0; i < n; i++) { g_n = fr_mul(&g_n, &g); zeta_n = fr_mul(&zeta_n, &zeta); }
    for (int i = 0; i < 4; i++) {                                                        /* v_h_coset_4n: g^N zeta^(iN) - 1 */
        fr_t p = g_n, one = fr_one();
        for (int k = 0; k < i; k++) p = fr_mul(&p, &zeta_n);
        p = fr_sub(&p, &one);
        fr_invert(&p, &vh_inv[i]);
    }
    fr_t bk[4];
    for (int w = 0; w < 4; w++) { static const uint64_t k[4] = {1, 7, 13, 17}; fr_t kw = fr_from_u64(k[w]); bk[w] = fr_mul(beta, &kw); }
    const fr_t kappa = fr_square(rho), kappa2 = fr_square(&kappa), kappa3 = fr_mul(&kappa2, &kappa), one = fr_one();
    fr_t *t = malloc(m * sizeof(fr_t));
    fr_t x = g;
    for (uint64_t i = 0; i < m; i++) {
        const uint64_t nx = (i + 4) % m;
#define EV(v, j) ev[(uint64_t)(v) * m + (j)]
        const fr_t a = EV(C_W, i), b = EV(C_W + 1, i), cc = EV(C_W + 2, i), d = EV(C_W + 3, i), d_next = EV(C_W + 3, nx);
        /* compute_circuit_satisfiability_equation: arithmetic widget (PI outside the q_arith factor) and range widget */
        fr_t s = fr_mul(&a, &b); s = fr_mul(&s, &EV(C_SEL + 0, i));
        fr_t u;
        u = fr_mul(&a, &EV(C_SEL + 1, i)); s = fr_add(&s, &u);
        u = fr_mul(&b, &EV(C_SEL + 2, i)); s = fr_add(&s, &u);
        u = fr_mul(&cc, &EV(C_SEL + 3, i)); s = fr_add(&s, &u);
        u = fr_mul(&d, &EV(C_SEL + 4, i)); s = fr_add(&s, &u);
        s = fr_add(&s, &EV(C_SEL + 5, i));
        s = fr_mul(&s, &EV(C_SEL + 6, i));
        s = fr_add(&s, &EV(C_PI, i));
        fr_t f, b1, b2, b3, b4;
        f = times4(&d); f = fr_sub(&cc, &f); b1 = delta(&f);
        f = times4(&cc); f = fr_sub(&b, &f); b2 = delta(&f); b2 = fr_mul(&b2, &kappa);
        f = times4(&b); f = fr_sub(&a, &f); b3 = delta(&f); b3 = fr_mul(&b3, &kappa2);
        f = times4(&a); f = fr_sub(&d_next, &f); b4 = delta(&f); b4 = fr_mul(&b4, &kappa3);
        fr_t r = fr_add(&b1, &b2); r = fr_add(&r, &b3); r = fr_add(&r, &b4);
        r = fr_mul(&r, &EV(C_SEL + 7, i)); r = fr_mul(&r, rho);
        s = fr_add(&s, &r);
        /* compute_permutation_checks: identity range check, copy range check, term check one */
        fr_t num = fr_one(), den = fr_one();
        for (int w = 0; w < 4; w++) {
            fr_t y = fr_mul(&bk[w], &x); y = fr_add(&y, &EV(C_W + w, i)); y = fr_add(&y, gamma); num = fr_mul(&num, &y);
            fr_t q = fr_mul(beta, &EV(C_S + w, i)); q = fr_add(&q, &EV(C_W + w, i)); q = fr_add(&q, gamma); den = fr_mul(&den, &q);
        }
        fr_t p1 = fr_mul(&num, &EV(C_Z, i)); p1 = fr_mul(&p1, alpha);
        fr_t p2 = fr_mul(&den, &EV(C_Z, nx)); p2 = fr_mul(&p2, alpha);
        fr_t p3 = fr_sub(&EV(C_Z, i), &one); p3 = fr_mul(&p3, &EV(C_L1, i));
        fr_t p = fr_sub(&p1, &p2); p = fr_add(&p, &p3);
        s = fr_add(&s, &p);
        t[i] = fr_mul(&s, &vh_inv[i % 4]);
        x = fr_mul(&x, &zeta);
#undef EV
    }
    free(ev);
    fr_t g_inv; fr_invert(&g, &g_inv);                                                   /* domain_4n.coset_ifft */
    orc_fft(t, log_n + 2, 1);
    distribute_powers(t, m, &g_inv);
    memcpy(out, t, m * sizeof(fr_t));                                                    /* split_tx_poly: t[rN .. (r+1)N) */
    free(t);
    return 0;
}

/* out = sum_i c[i] x^i */
void quot_horner(const fr_t *c, uint64_t n, const fr_t *x, fr_t *out) {
    fr_t acc = fr_zero();
    for (uint64_t i = n; i-- > 0;) { acc = fr_mul(&acc, x); acc = fr_add(&acc, &c[i]); }
    *out = acc;
}
