"""The permutation argument's test oracles (TEST INFRASTRUCTURE ONLY), next to the gadget oracles of oracle/:

  * defining loops on Python ints over the big-int model's own variable map (oracle/pymodel.py StandardComposer.perm_map):
    sigma_evaluations, permutation_z, exclusive_prefix_product, and an O(n log n) inverse transform for the coefficient forms;
  * perm_oracle_z: the C restatement tests/oracle_perm/permutation.c over the C oracle's composer (oracle/binding.py), for domains
    the Python loops are too slow for;
  * the generator of tests/golden/permutation.json:   python -m tests.permutation_model

[DEP] dusk-plonk 0.8 src/permutation/permutation.rs (compute_sigma_permutations, compute_permutation_lagrange,
compute_fast_permutation_poly, compute_permutation_poly) and permutation/constants.rs, recalled: parity unpinned (DESIGN.md §7).
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess

import numpy as np

from oracle import pymodel as pm
from oracle.gen_golden import coeff_digest, run_pymodel_composer
from tests.programs import Q, hx, synth_wide

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PERM_K = (1, 7, 13, 17)                                    # permutation/constants.rs: 1, K1, K2, K3 for w_l, w_r, w_o, w_4


# ------------------------------------------------------------------------------------------------ big-int model
def sigma_positions(composer, log_n: int):
    """[w][i] -> cycle successor (row, wire) of position (i, w); padding rows and positions outside the map are fixed points."""
    size = 1 << log_n
    assert composer.n <= size
    succ = [[(i, w) for i in range(size)] for w in range(4)]
    for uses in composer.perm_map.values():
        for k, (r, w) in enumerate(uses):
            succ[w][r] = uses[(k + 1) % len(uses)]
    return succ


def sigma_evaluations(composer, log_n: int):
    """sigma_w(w^i) = k_{w'} * w^{r'} for the successor (r', w') of (i, w): 4 lists of 2^log_n canonical ints."""
    g = pm.group_gen(log_n)
    return [[PERM_K[w2] * pow(g, r2, Q) % Q for (r2, w2) in col] for col in sigma_positions(composer, log_n)]


def exclusive_prefix_product(values):
    """out[0] = 1, out[i] = values[0] * .. * values[i-1]; and the product of all of them."""
    out, acc = [], 1
    for v in values:
        out.append(acc)
        acc = acc * v % Q
    return out, acc


def permutation_z(composer, log_n: int, beta: int, gamma: int):
    """(z evaluations, closing): z_0 = 1, z_{i+1} = z_i * num_i / den_i over the domain 2^log_n, closing = prod of all ratios.
    Raises ZeroDivisionError at the first row whose denominator is zero (the reference's invert().unwrap() panics)."""
    size = 1 << log_n
    g = pm.group_gen(log_n)
    sig = sigma_evaluations(composer, log_n)
    cols = [[composer.variables[v] for v in wires] + [0] * (size - composer.n)
            for wires in (composer.w_l, composer.w_r, composer.w_o, composer.w_4)]
    ratios = []
    for i in range(size):
        gi = pow(g, i, Q)
        num = den = 1
        for w in range(4):
            num = num * (cols[w][i] + beta * PERM_K[w] * gi + gamma) % Q
            den = den * (cols[w][i] + beta * sig[w][i] + gamma) % Q
        if den == 0:
            raise ZeroDivisionError(f"zero denominator at row {i}")
        ratios.append(num * pow(den, Q - 2, Q) % Q)
    return exclusive_prefix_product(ratios)


def ifft(values):
    """domain.ifft by recursive radix-2 decimation in time on Python ints (the same result as pymodel.dft, O(n log n))."""
    n = len(values)

    def rec(a, w):
        if len(a) == 1:
            return a
        even, odd = rec(a[0::2], w * w % Q), rec(a[1::2], w * w % Q)
        out, h, t = [0] * len(a), len(a) // 2, 1
        for k in range(h):
            x = t * odd[k] % Q
            out[k], out[k + h] = (even[k] + x) % Q, (even[k] - x) % Q
            t = t * w % Q
        return out
    n_inv = pow(n, Q - 2, Q)
    return [v * n_inv % Q for v in rec(list(values), pow(pm.group_gen(n.bit_length() - 1), Q - 2, Q))]


# ------------------------------------------------------------------------------------------------ C restatement
_SRC = os.path.join(HERE, "oracle_perm", "permutation.c")
_SO = os.path.join(HERE, "oracle_perm", "_build", "libperm_oracle.so")
_lib = None


def _clib():
    global _lib
    if _lib is None:
        deps = [_SRC, os.path.join(ROOT, "oracle", "fr.h"), os.path.join(ROOT, "oracle", "composer.h")]
        if not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.run(["gcc", "-O3", "-march=x86-64-v3", "-madx", "-fPIC", "-shared", "-std=gnu11", "-o", _SO, _SRC], check=True)
        _lib = C.CDLL(_SO)
        vp = C.c_void_p
        _lib.perm_oracle_z.restype = C.c_int
        _lib.perm_oracle_z.argtypes = [vp, vp, C.c_uint, vp, vp, vp, vp, vp, vp]
    return _lib


def perm_oracle_z(binding, composer, log_n: int, beta, gamma):
    """(sigma evaluations (4, 2^log_n, 4), z evaluations (2^log_n, 4), closing (4,)) in Montgomery limbs for the oracle composer
    `composer` (oracle.binding.Composer); beta, gamma: one Montgomery scalar each.  Raises ZeroDivisionError at a zero denominator."""
    size = 1 << log_n
    sig = np.zeros((4, size, 4), dtype=np.uint64); z = np.zeros((size, 4), dtype=np.uint64); closing = np.zeros(4, dtype=np.uint64)
    var = np.ascontiguousarray(composer.variables())
    omega = binding.from_ints([binding.domain_group_gen(log_n)])[0]
    b = np.ascontiguousarray(beta, dtype=np.uint64).reshape(4); g = np.ascontiguousarray(gamma, dtype=np.uint64).reshape(4)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = _clib().perm_oracle_z(composer._c, p(var), log_n, p(omega), p(b), p(g), p(sig), p(z), p(closing))
    if rc < 0:
        raise ValueError(f"a domain of 2^{log_n} cannot hold {composer.n} rows")
    if rc > 0:
        raise ZeroDivisionError(f"zero denominator at row {rc - 1}")
    return sig, z, closing


# ------------------------------------------------------------------------------------------------ golden vectors
BETA_GAMMA_STREAM = 110


def permutation_vectors(programs, max_domain: int = 1 << 13):
    """Per non-error golden program (domains up to max_domain): digests of the sigma evaluations and coefficients and of z's
    evaluations and coefficients from the loops above, at one (beta, gamma) drawn from SEED.  The closing product is 1 on every one."""
    beta, gamma = synth_wide(BETA_GAMMA_STREAM, 2)
    out = dict(beta=hx(beta), gamma=hx(gamma), programs={})
    for name in sorted(programs):
        spec = programs[name]
        if spec["expected"]["error"] or (1 << pm.domain_log_size(spec["expected"]["n_rows"])) > max_domain:
            continue
        c = run_pymodel_composer(spec["program"])
        log_n = pm.domain_log_size(c.n)
        sig = sigma_evaluations(c, log_n)
        z, closing = permutation_z(c, log_n, beta, gamma)
        assert closing == 1, name
        out["programs"][name] = dict(log_n=log_n, sigma_evaluations=coeff_digest(sig), sigma_coefficients=coeff_digest([ifft(col) for col in sig]),
                                     z_evaluations=coeff_digest([z]), z_coefficients=coeff_digest([ifft(z)]), z_head=[hx(v) for v in z[:3]])
    return out


def main():
    golden = os.path.join(HERE, "golden")
    with open(os.path.join(golden, "programs.json")) as f:
        programs = json.load(f)
    vec = permutation_vectors(programs)
    path = os.path.join(golden, "permutation.json")
    with open(path, "w") as f:
        json.dump(vec, f, indent=1, sort_keys=True)
    print(f"wrote {len(vec['programs'])} permutation-argument digest sets to {path}")


if __name__ == "__main__":
    main()
