"""The quotient polynomial's test oracles (TEST INFRASTRUCTURE ONLY), next to tests/permutation_model.py:

  * a defining big-int model over the big-int model's own composer (oracle/pymodel.py) and the permutation loops of
    tests/permutation_model.py: selector and public-input polynomials, the numerator polynomial N(X) of round 3 as an exact
    coefficient vector (evaluation at the 8N-th roots of unity, a plain domain, then interpolation), and t(X) = N(X) / (X^N - 1)
    by long division with the remainder checked;
  * quot_oracle_t: the C restatement tests/oracle_quotient/quotient.c over the C oracle's composer (one 4N coset transform, the
    reference's own structure), for domains the Python model is too slow for, and its Horner evaluator;
  * the generator of tests/golden/quotient.json:   python -m tests.quotient_model

[DEP] dusk-plonk 0.8 src/proof_system/quotient_poly.rs (compute, compute_circuit_satisfiability_equation,
compute_permutation_checks, split_tx_poly) and widget/range, recalled: parity unpinned (DESIGN.md §7).
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess

import numpy as np

from oracle import pymodel as pm
from oracle.gen_golden import coeff_digest, run_pymodel_composer
from tests import permutation_model as perm
from tests.programs import Q, hx, synth_wide

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GENERATOR = 7                                              # dusk-bls12_381 GENERATOR: the coset of the 4N domain
SELECTORS = ("q_m", "q_l", "q_r", "q_o", "q_4", "q_c", "q_arith", "q_range")


# ------------------------------------------------------------------------------------------------ big-int model
def fft(values, root):
    """sum_j a_j root^(jk) for k < len(values), recursive radix-2 on Python ints (len a power of two, root of that order)."""
    if len(values) == 1:
        return list(values)
    even, odd = fft(values[0::2], root * root % Q), fft(values[1::2], root * root % Q)
    out, h, t = [0] * len(values), len(values) // 2, 1
    for k in range(h):
        x = t * odd[k] % Q
        out[k], out[k + h] = (even[k] + x) % Q, (even[k] - x) % Q
        t = t * root % Q
    return out


def padded(col, size):
    return [v % Q for v in col] + [0] * (size - len(col))


def selector_evaluations(composer, log_n: int):
    """q_m q_l q_r q_o q_4 q_c q_arith q_range of rows 0 .. 2^log_n (padding rows zero): 8 lists of canonical ints."""
    return [padded(composer.sel[k], 1 << log_n) for k in SELECTORS]


def public_input_evaluations(composer, log_n: int):
    return padded(composer.construct_dense_pi_vec(), 1 << log_n)


def wire_evaluations(composer, log_n: int):
    return [padded([composer.variables[v] for v in wires], 1 << log_n) for wires in (composer.w_l, composer.w_r, composer.w_o, composer.w_4)]


def component_polynomials(composer, log_n: int, beta: int, gamma: int):
    """Coefficient vectors (N each) in the engine's order: 4 wires, z, 4 sigma, 8 selectors, PI."""
    z, closing = perm.permutation_z(composer, log_n, beta, gamma)
    evals = (wire_evaluations(composer, log_n) + [z] + perm.sigma_evaluations(composer, log_n) + selector_evaluations(composer, log_n)
             + [public_input_evaluations(composer, log_n)])
    return [perm.ifft(e) for e in evals]


def numerator_at(p, x, xn, l1, alpha, beta, gamma, rho):
    """The round-3 numerator at one point from the component values p (wires, z, sigma, selectors, PI at x) and xn (wires and z at
    x*w); l1 = L_1(x)."""
    a, b, c, d = p[0:4]
    z, sig = p[4], p[5:9]
    q_m, q_l, q_r, q_o, q_4, q_c, q_arith, q_range = p[9:17]
    pi = p[17]
    kappa = rho * rho % Q

    def delta(f):
        return f * (f - 1) * (f - 2) * (f - 3)
    arith = q_arith * (q_m * a * b + q_l * a + q_r * b + q_o * c + q_4 * d + q_c) + pi
    rng = rho * q_range * (delta(c - 4 * d) + kappa * delta(b - 4 * c) + kappa ** 2 * delta(a - 4 * b) + kappa ** 3 * delta(xn[3] - 4 * a))
    num = den = 1
    for w in range(4):
        num = num * (p[w] + beta * perm.PERM_K[w] * x + gamma) % Q
        den = den * (p[w] + beta * sig[w] + gamma) % Q
    permutation = alpha * z * num - alpha * xn[4] * den + alpha * alpha * l1 * (z - 1)
    return (arith + rng + permutation) % Q


def numerator_polynomial(polys, log_n: int, alpha: int, beta: int, gamma: int, rho: int):
    """N(X) as 8N coefficients: the components evaluated at the 8N-th roots of unity mu^i (x*w = mu^(i+8)), N(x) there, and the
    inverse transform.  deg N <= 5N - 5 < 8N, so the interpolation is exact."""
    n = 1 << log_n
    m = 8 * n
    mu = pm.group_gen(log_n + 3)
    ev = [fft(p + [0] * (m - n), mu) for p in polys]
    vals = []
    x = 1
    for i in range(m):
        xn_pow = pow(x, n, Q)
        l1 = (1 if x == 1 else 0) if xn_pow == 1 else (xn_pow - 1) * pow(n * (x - 1), Q - 2, Q) % Q
        nxt = (i + 8) % m
        vals.append(numerator_at([e[i] for e in ev], x, [ev[w][nxt] for w in range(4)] + [ev[4][nxt]], l1, alpha, beta, gamma, rho))
        x = x * mu % Q
    m_inv = pow(m, Q - 2, Q)
    return [v * m_inv % Q for v in fft(vals, pow(mu, Q - 2, Q))]


def divide_by_vanishing(num, n: int):
    """(t, remainder): num = t * (X^N - 1) + remainder, t_k = num_(k+N) + t_(k+N) from the top, remainder_k = num_k + t_k (k < N)."""
    t = [0] * len(num)
    for k in range(len(num) - n - 1, -1, -1):
        t[k] = (num[k + n] + (t[k + n] if k + n < len(num) else 0)) % Q
    rem = [(num[k] + t[k]) % Q for k in range(n)]
    return t, rem


def coset_interpolant_of_remainder(rem, log_n: int):
    """The polynomial of degree < 4N that takes the values r(x) / (x^N - 1) on the coset g<zeta> of the 4N domain, r = rem (deg < N):
    what a 4N-point coset interpolation of N(x) / (x^N - 1) adds to the quotient of the long division when the remainder is not zero
    (an unsatisfied composer).  coset_fft / coset_ifft written out: scale by g^m, transform, divide, transform back, scale by g^-m."""
    n, m = 1 << log_n, 4 << log_n
    zeta = pm.group_gen(log_n + 2)
    vals = fft([r * pow(GENERATOR, i, Q) % Q for i, r in enumerate(rem)] + [0] * (m - n), zeta)
    g_n = pow(GENERATOR, n, Q)
    iota = pow(zeta, n, Q)
    zh_inv = [pow((g_n * pow(iota, i % 4, Q) - 1) % Q, Q - 2, Q) for i in range(4)]         # x^N - 1 = g^N iota^i at x = g zeta^i
    vals = [v * zh_inv[i % 4] % Q for i, v in enumerate(vals)]
    m_inv, g_inv = pow(m, Q - 2, Q), pow(GENERATOR, Q - 2, Q)
    return [v * m_inv * pow(g_inv, i, Q) % Q for i, v in enumerate(fft(vals, pow(zeta, Q - 2, Q)))]


def quotient(composer, log_n: int, alpha: int, beta: int, gamma: int, rho: int):
    """(t_1 .. t_4 as 4 lists of N canonical ints, remainder of N(X) / (X^N - 1), N(X)).  On a composer whose constraints hold the
    remainder is zero and t is the exact quotient, of degree <= 4N - 5 (asserted).  Otherwise t(X) is not a polynomial; the engine's
    t is then the interpolant of N(x) / (x^N - 1) on the coset g<zeta>, which is the exact quotient plus
    coset_interpolant_of_remainder(remainder)."""
    n = 1 << log_n
    polys = component_polynomials(composer, log_n, beta, gamma)
    num = numerator_polynomial(polys, log_n, alpha, beta, gamma, rho)
    t, rem = divide_by_vanishing(num, n)
    t = t[:4 * n] + [0] * (4 * n - len(t))
    if not any(rem):
        assert not any(t[4 * n - 4:]), "deg t > 4N - 5"
    else:
        t = [(a + b) % Q for a, b in zip(t, coset_interpolant_of_remainder(rem, log_n))]
    return [t[r * n:(r + 1) * n] for r in range(4)], rem, num


def horner(coeffs, x):
    acc = 0
    for c in reversed(coeffs):
        acc = (acc * x + c) % Q
    return acc


# ------------------------------------------------------------------------------------------------ C restatement
_SRC = os.path.join(HERE, "oracle_quotient", "quotient.c")
_SO = os.path.join(HERE, "oracle_quotient", "_build", "libquot_oracle.so")
_lib = None


def _clib():
    global _lib
    if _lib is None:
        deps = [_SRC, os.path.join(HERE, "oracle_perm", "permutation.c")] + [os.path.join(ROOT, "oracle", f) for f in ("fft.c", "composer.c", "fr.h", "composer.h")]
        if not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.run(["gcc", "-O3", "-march=x86-64-v3", "-madx", "-fPIC", "-shared", "-std=gnu11", "-o", _SO, _SRC,
                            os.path.join(ROOT, "oracle", "fft.c"), os.path.join(ROOT, "oracle", "composer.c")], check=True)
        _lib = C.CDLL(_SO)
        vp = C.c_void_p
        _lib.quot_oracle_t.restype = C.c_int
        _lib.quot_oracle_t.argtypes = [vp, vp, C.c_uint, vp, vp, vp, vp, vp]
        _lib.quot_horner.restype = None
        _lib.quot_horner.argtypes = [vp, C.c_uint64, vp, vp]
    return _lib


def quot_oracle_t(binding, composer, log_n: int, alpha, beta, gamma, rho):
    """t_1 .. t_4 ((4, 2^log_n, 4) Montgomery limbs) by the C restatement for the oracle composer `composer` (oracle.binding.Composer);
    challenges: one Montgomery scalar each.  Raises ZeroDivisionError at a zero z denominator."""
    size = 1 << log_n
    out = np.zeros((4, size, 4), dtype=np.uint64)
    var = np.ascontiguousarray(composer.variables())
    ch = [np.ascontiguousarray(x, dtype=np.uint64).reshape(4) for x in (alpha, beta, gamma, rho)]
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = _clib().quot_oracle_t(composer._c, p(var), log_n, *map(p, ch), p(out))
    if rc < 0:
        raise ValueError(f"a domain of 2^{log_n} cannot hold {composer.n} rows (or is larger than 2^30)")
    if rc > 0:
        raise ZeroDivisionError(f"zero denominator at row {rc - 1}")
    return out


def horner_mont(coeffs, x):
    """sum_i coeffs[i] x^i for an (n, 4) Montgomery array (any memory layout numpy can make contiguous) and one Montgomery x."""
    c = np.ascontiguousarray(coeffs, dtype=np.uint64)
    xx = np.ascontiguousarray(x, dtype=np.uint64).reshape(4)
    out = np.zeros(4, dtype=np.uint64)
    _clib().quot_horner(c.ctypes.data_as(C.c_void_p), c.shape[0], xx.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    return out


# ------------------------------------------------------------------------------------------------ golden vectors
CHALLENGE_STREAM = 160


def challenges():
    """(alpha, beta, gamma, range_challenge) of the golden vectors, canonical ints."""
    return tuple(synth_wide(CHALLENGE_STREAM, 4))


def quotient_vectors(programs, max_domain: int = 1 << 12):
    """Per non-error golden program (domains up to max_domain): digests of the selector polynomials and PI (both forms) and of
    t_1 .. t_4 from the model above, at challenges()."""
    alpha, beta, gamma, rho = challenges()
    out = dict(alpha=hx(alpha), beta=hx(beta), gamma=hx(gamma), range_challenge=hx(rho), programs={})
    for name in sorted(programs):
        spec = programs[name]
        if spec["expected"]["error"] or (1 << pm.domain_log_size(spec["expected"]["n_rows"])) > max_domain:
            continue
        c = run_pymodel_composer(spec["program"])
        log_n = pm.domain_log_size(c.n)
        sel = selector_evaluations(c, log_n)
        pi = public_input_evaluations(c, log_n)
        t, rem, _num = quotient(c, log_n, alpha, beta, gamma, rho)
        assert any(rem) == bool(c.unsatisfied_rows()), name
        out["programs"][name] = dict(log_n=log_n, selector_evaluations=coeff_digest(sel), selector_coefficients=coeff_digest([perm.ifft(s) for s in sel]),
                                     pi_evaluations=coeff_digest([pi]), pi_coefficients=coeff_digest([perm.ifft(pi)]), t=coeff_digest(t))
    return out


def main():
    golden = os.path.join(HERE, "golden")
    with open(os.path.join(golden, "programs.json")) as f:
        programs = json.load(f)
    vec = quotient_vectors(programs)
    path = os.path.join(golden, "quotient.json")
    with open(path, "w") as f:
        json.dump(vec, f, indent=1, sort_keys=True)
    print(f"wrote {len(vec['programs'])} quotient digest sets to {path}")


if __name__ == "__main__":
    main()
