/*
 * tests/oracle_lagrange/group_fft.c -- CPU restatement of the Lagrange-basis SRS derived from the monomial powers:
 *     lagrange[i] = L_i(tau) G = (1/n) sum_j w^(-ij) powers_of_g[j],   i < n = 2^log_n.
 *
 * TEST INFRASTRUCTURE ONLY (see oracle/fr.h).  Built by tests/lagrange_model.py into tests/oracle_lagrange/_build; it takes its
 * field and group code from oracle/g1.c (Jacobian coordinates, jac_mul double-and-add) and shares no code with the kernels.
 * The textbook serial radix-2 inverse FFT of oracle/fft.c (serial_fft with group_gen^-1, then size^-1), with points in place of
 * scalars: bit-reversal permutation, log n stages of decimation-in-time butterflies a +- w b with w stepping by w_m = w^(-n/2m)
 * inside a half block and every twiddle applied by jac_mul, then every point multiplied by 1/n.  (The kernels instead take their
 * twiddles from the forward table, skip the twiddle 1, apply 1/n first and use a fixed window schedule.)
 */
#include "../../oracle/g1.c"

static const fr_t LAG_ROOT_OF_UNITY = {{0xb9b58d8c5f0e466aULL, 0x5b1b4c801819d7ecULL, 0x0af53ae352a31e64ULL, 0x5bf3adda19e9b27bULL}};

static uint64_t lag_bitreverse(uint64_t k, unsigned l) {
    uint64_t r = 0;
    for (unsigned i = 0; i < l; i++) { r = (r << 1) | (k & 1); k >>= 1; }
    return r;
}
static g1_jac_t lag_jac_neg(const g1_jac_t *p) { g1_jac_t r = *p; r.y = fp_neg(&p->y); return r; }

/* out[i] = (1/n) sum_j w^(-ij) powers[j], i < 2^log_n (log_n <= 32) */
void lag_group_ifft(const g1_affine_t *powers, unsigned log_n, g1_affine_t *out) {
    const uint64_t n = (uint64_t)1 << log_n;
    g1_jac_t *a = malloc(n * sizeof(g1_jac_t));
    for (uint64_t k = 0; k < n; k++) a[lag_bitreverse(k, log_n)] = jac_from_affine(&powers[k]);
    fr_t omega = LAG_ROOT_OF_UNITY, omega_inv;
    for (unsigned i = log_n; i < 32; i++) omega = fr_square(&omega);          /* EvaluationDomain::new: group_gen */
    fr_invert(&omega, &omega_inv);
    for (uint64_t m = 1; m < n; m *= 2) {
        const uint64_t e[4] = {n / (2 * m), 0, 0, 0};
        const fr_t w_m = fr_pow(&omega_inv, e);
        for (uint64_t k = 0; k < n; k += 2 * m) {
            fr_t w = fr_one();
            for (uint64_t j = 0; j < m; j++) {
                const g1_jac_t t = jac_mul(&a[k + j + m], &w), nt = lag_jac_neg(&t);
                a[k + j + m] = jac_add(&a[k + j], &nt);
                a[k + j] = jac_add(&a[k + j], &t);
                w = fr_mul(&w, &w_m);
            }
        }
    }
    fr_t size_inv;
    fr_t size = fr_from_u64(n);
    fr_invert(&size, &size_inv);
    for (uint64_t i = 0; i < n; i++) { const g1_jac_t s = jac_mul(&a[i], &size_inv); out[i] = jac_to_affine(&s); }
    free(a);
}
