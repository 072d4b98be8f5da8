"""The openings' test oracles (TEST INFRASTRUCTURE ONLY), next to tests/quotient_model.py:

  * a big-int model over the big-int model's own composer: the component polynomials and t of tests/quotient_model.py, the
    evaluations by Horner, r(X) by its formula, the two aggregates and the textbook Ruffini division;
  * open_oracle / c_ruffini / c_evaluate: the C restatement tests/oracle_openings/openings.c (the crate's own operations:
    Polynomial::evaluate, scalar x polynomial sums, Polynomial::ruffini) over given coefficient vectors, for 2^18 and above;
  * the quotient identity and the pairing-free opening checks used by the tests;
  * the generator of tests/golden/openings.json:   python -m tests.opening_model

[DEP] dusk-plonk 0.8 Prover::prove (rounds 4 and 5), linearisation_poly::compute, the widgets' compute_linearisation,
compute_quotient_opening_poly / compute_aggregate_witness and Polynomial::ruffini, recalled: parity unpinned (DESIGN.md §7).
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
from tests import quotient_model as qm
from tests.programs import Q, hx, synth_wide

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
EVALUATIONS = ("a_eval", "b_eval", "c_eval", "d_eval", "a_next_eval", "b_next_eval", "d_next_eval", "q_arith_eval", "q_c_eval",
               "q_l_eval", "q_r_eval", "left_sigma_eval", "right_sigma_eval", "out_sigma_eval", "lin_poly_eval", "perm_eval", "quot_eval")
# component polynomial indices (tests/quotient_model.component_polynomials: 4 wires, z, 4 sigma, 8 selectors, PI)
W, Z, S, QM, QL, QR, QO, Q4, QC, QARITH, QRANGE, PI = 0, 4, 5, 9, 10, 11, 12, 13, 14, 15, 16, 17


# ------------------------------------------------------------------------------------------------ big-int model
horner = qm.horner


def ruffini(f, p):
    """The quotient of f by (X - p), remainder dropped: q_(n-2) = f_(n-1), q_(i-1) = f_i + p q_i; n coefficients, q_(n-1) = 0."""
    n = len(f)
    q, acc = [0] * n, 0
    for i in range(n - 1, 0, -1):
        acc = (f[i] + p * acc) % Q
        q[i - 1] = acc
    return q


def delta(f):
    return f * (f - 1) * (f - 2) * (f - 3) % Q


def lagrange_1(x, n):
    xn = pow(x, n, Q)
    return (xn - 1) * pow(n * (x - 1), Q - 2, Q) % Q


def linearisation_weights(ev, alpha, beta, gamma, rho, z, n):
    """The scalars r's polynomials are multiplied by: {index: weight} over q_m q_l q_r q_o q_4 q_c q_range z sigma_4."""
    a, b, c, d = ev["a_eval"], ev["b_eval"], ev["c_eval"], ev["d_eval"]
    qa, kappa = ev["q_arith_eval"], rho * rho % Q
    rng = rho * (delta(c - 4 * d) + kappa * delta(b - 4 * c) + kappa ** 2 * delta(a - 4 * b) + kappa ** 3 * delta(ev["d_next_eval"] - 4 * a))
    prod = 1
    for k, vw in zip(perm.PERM_K, (a, b, c, d)):
        prod = prod * (vw + beta * k * z + gamma) % Q
    sig = [ev["left_sigma_eval"], ev["right_sigma_eval"], ev["out_sigma_eval"]]
    prod_s = (a + beta * sig[0] + gamma) * (b + beta * sig[1] + gamma) * (c + beta * sig[2] + gamma) % Q
    return {QM: qa * a * b % Q, QL: qa * a % Q, QR: qa * b % Q, QO: qa * c % Q, Q4: qa * d % Q, QC: qa, QRANGE: rng % Q,
            Z: (alpha * prod + alpha * alpha * lagrange_1(z, n)) % Q, S + 3: -alpha * beta * ev["perm_eval"] * prod_s % Q}


def openings_from_polys(polys, t, log_n, alpha, beta, gamma, rho, z, v, vs):
    """(evaluations dict, r, W_z, W_zw, remainders) from the component polynomials (quotient_model order) and t_1 .. t_4."""
    n = 1 << log_n
    zw = z * pm.group_gen(log_n) % Q
    at = lambda i: horner(polys[i], z)
    zn = pow(z, n, Q)
    assert zn != 1, "zeta^N = 1"
    ev = dict(a_eval=at(W), b_eval=at(W + 1), c_eval=at(W + 2), d_eval=at(W + 3), a_next_eval=horner(polys[W], zw),
              b_next_eval=horner(polys[W + 1], zw), d_next_eval=horner(polys[W + 3], zw), q_arith_eval=at(QARITH), q_c_eval=at(QC),
              q_l_eval=at(QL), q_r_eval=at(QR), left_sigma_eval=at(S), right_sigma_eval=at(S + 1), out_sigma_eval=at(S + 2),
              perm_eval=horner(polys[Z], zw))
    quot = [sum(pow(zn, r, Q) * t[r][i] for r in range(4)) % Q for i in range(n)]
    ev["quot_eval"] = horner(quot, z)
    wts = linearisation_weights(ev, alpha, beta, gamma, rho, z, n)
    r = [sum(w * polys[k][i] for k, w in wts.items()) % Q for i in range(n)]
    ev["lin_poly_eval"] = horner(r, z)
    agg = [quot, r] + [polys[W + k] for k in range(4)] + [polys[S + k] for k in range(3)]
    agg_z = [sum(pow(v, k, Q) * p[i] for k, p in enumerate(agg)) % Q for i in range(n)]
    shifted = [polys[Z], polys[W], polys[W + 1], polys[W + 3]]
    agg_zw = [sum(pow(vs, k, Q) * p[i] for k, p in enumerate(shifted)) % Q for i in range(n)]
    return ev, r, ruffini(agg_z, z), ruffini(agg_zw, zw), (horner(agg_z, z), horner(agg_zw, zw))


def openings(composer, log_n, alpha, beta, gamma, rho, z, v, vs):
    """The model for a big-int composer: (evaluations, r, W_z, W_zw, remainders, t, PI(z))."""
    polys = qm.component_polynomials(composer, log_n, beta, gamma)
    t, _rem, _num = qm.quotient(composer, log_n, alpha, beta, gamma, rho)
    ev, r, wz, wzw, rems = openings_from_polys(polys, t, log_n, alpha, beta, gamma, rho, z, v, vs)
    return ev, r, wz, wzw, rems, t, horner(polys[PI], z)


def quotient_identity_holds(ev, pi_z, alpha, beta, gamma, z, n):
    """quot * Z_H(z) == lin + PI(z) - alpha^2 L_1(z) - alpha perm (a + beta s1 + gamma)(b + beta s2 + gamma)(c + beta s3 + gamma)(d + gamma)."""
    zh = (pow(z, n, Q) - 1) % Q
    prod = ((ev["a_eval"] + beta * ev["left_sigma_eval"] + gamma) * (ev["b_eval"] + beta * ev["right_sigma_eval"] + gamma)
            * (ev["c_eval"] + beta * ev["out_sigma_eval"] + gamma) * (ev["d_eval"] + gamma))
    rhs = ev["lin_poly_eval"] + pi_z - alpha * alpha * lagrange_1(z, n) - alpha * ev["perm_eval"] * prod
    return ev["quot_eval"] * zh % Q == rhs % Q


def aggregate_values(ev, z, n, v, vs):
    """The aggregates' values at z and z*w from the evaluations: sum v^i p_i(z) and sum v'^i p_i(z w)."""
    at_z = [ev["quot_eval"], ev["lin_poly_eval"], ev["a_eval"], ev["b_eval"], ev["c_eval"], ev["d_eval"], ev["left_sigma_eval"],
            ev["right_sigma_eval"], ev["out_sigma_eval"]]
    at_zw = [ev["perm_eval"], ev["a_next_eval"], ev["b_next_eval"], ev["d_next_eval"]]
    return (sum(pow(v, k, Q) * x for k, x in enumerate(at_z)) % Q, sum(pow(vs, k, Q) * x for k, x in enumerate(at_zw)) % Q)


# ------------------------------------------------------------------------------------------------ C restatement
_SRC = os.path.join(HERE, "oracle_openings", "openings.c")
_SO = os.path.join(HERE, "oracle_openings", "_build", "libopen_oracle.so")
_lib = None


def _clib():
    global _lib
    if _lib is None:
        deps = [_SRC, os.path.join(ROOT, "oracle", "fr.h")]
        if not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.run(["gcc", "-O3", "-march=x86-64-v3", "-madx", "-fPIC", "-shared", "-std=gnu11", "-o", _SO, _SRC], check=True)
        _lib = C.CDLL(_SO)
        vp = C.c_void_p
        _lib.open_oracle.restype = C.c_int
        _lib.open_oracle.argtypes = [vp, vp, C.c_uint64, vp, vp, vp, vp]
        _lib.open_ruffini.restype = None
        _lib.open_ruffini.argtypes = [vp, C.c_uint64, vp, vp]
        _lib.open_evaluate.restype = None
        _lib.open_evaluate.argtypes = [vp, C.c_uint64, vp, vp]
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def open_oracle(oracle, vec, t, log_n, challenges):
    """(evaluations (17, 4), [W_z, W_zw, r] (3, N, 4)) by the C restatement; vec: (17, N, 4) coefficient vectors in the engine's order
    (wires, z, sigma, selectors), t: (4, N, 4), challenges: 7 Montgomery scalars alpha beta gamma rho z v v'."""
    n = 1 << log_n
    vec = np.ascontiguousarray(vec, dtype=np.uint64)
    t = np.ascontiguousarray(t, dtype=np.uint64)
    assert vec.shape == (17, n, 4) and t.shape == (4, n, 4)
    ch = np.ascontiguousarray(np.stack([np.asarray(x, dtype=np.uint64).reshape(4) for x in challenges]))
    omega = oracle.from_ints([pm.group_gen(log_n)])[0]
    ev = np.zeros((17, 4), dtype=np.uint64)
    dst = np.zeros((3, n, 4), dtype=np.uint64)
    if _clib().open_oracle(_p(vec), _p(t), n, _p(ch), _p(np.ascontiguousarray(omega)), _p(ev), _p(dst)):
        raise ValueError("zeta^N = 1")
    return ev, dst


def c_ruffini(f, p):
    f = np.ascontiguousarray(f, dtype=np.uint64)
    out = np.zeros_like(f)
    _clib().open_ruffini(_p(f), f.shape[0], _p(np.ascontiguousarray(p, dtype=np.uint64).reshape(4)), _p(out))
    return out


def c_evaluate(f, x):
    f = np.ascontiguousarray(f, dtype=np.uint64)
    out = np.zeros(4, dtype=np.uint64)
    _clib().open_evaluate(_p(f), f.shape[0], _p(np.ascontiguousarray(x, dtype=np.uint64).reshape(4)), _p(out))
    return out


# ------------------------------------------------------------------------------------------------ golden vectors
CHALLENGE_STREAM = 180


def challenges():
    """(alpha, beta, gamma, range_challenge, z, v, v') of the golden vectors, canonical ints."""
    return tuple(synth_wide(CHALLENGE_STREAM, 7))


def opening_vectors(programs, max_domain: int = 1 << 12):
    """Per non-error golden program (domains up to max_domain): digests of the evaluations, r, W_z and W_zw from the model above."""
    ch = challenges()
    out = dict(challenges=[hx(x) for x in ch], programs={})
    for name in sorted(programs):
        spec = programs[name]
        if spec["expected"]["error"] or (1 << pm.domain_log_size(spec["expected"]["n_rows"])) > max_domain:
            continue
        c = run_pymodel_composer(spec["program"])
        log_n = pm.domain_log_size(c.n)
        ev, r, wz, wzw, _rems, _t, pi_z = openings(c, log_n, *ch)
        honest = not c.unsatisfied_rows()
        assert quotient_identity_holds(ev, pi_z, ch[0], ch[1], ch[2], ch[4], 1 << log_n) == honest, name
        out["programs"][name] = dict(log_n=log_n, evaluations=coeff_digest([[ev[k] for k in EVALUATIONS]]), r=coeff_digest([r]),
                                     w_z=coeff_digest([wz]), w_zw=coeff_digest([wzw]))
    return out


def main():
    golden = os.path.join(HERE, "golden")
    with open(os.path.join(golden, "programs.json")) as f:
        programs = json.load(f)
    vec = opening_vectors(programs)
    path = os.path.join(golden, "openings.json")
    with open(path, "w") as f:
        json.dump(vec, f, indent=1, sort_keys=True)
    print(f"wrote {len(vec['programs'])} opening digest sets to {path}")


if __name__ == "__main__":
    main()
