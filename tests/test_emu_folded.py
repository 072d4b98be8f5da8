"""CPU tests of the folded q_m*b product of the generic gate check (fr.cuh fr_fold_constants / fr_mul_folded) through its host
emulation: the constants, the product against big ints for edge and random operands, the bound on the result, and no dropped
carry that is not zero -- also in the dot product that takes the result as its first operand."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

from tests.programs import Q

HERE = os.path.dirname(os.path.abspath(__file__))
EMU_DIR = os.path.join(HERE, "emu")
ROOT = os.path.dirname(HERE)
R = (1 << 256) % Q
RINV = pow(R, -1, Q)
U_BOUND = 2 * Q + 2 ** 227          # u = q_m*b + q_l: below q + 2^227, plus q_l < q


@pytest.fixture(scope="module")
def lib():
    out = os.path.join(EMU_DIR, "_build", "libfold_emu.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    src = os.path.join(EMU_DIR, "fold_emu.cpp")
    deps = [src, os.path.join(ROOT, "plonk_gadgets_b200", "csrc", "fr.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out, src], check=True)
    return C.CDLL(out)


def pack(vs):
    return np.frombuffer(b"".join(v.to_bytes(32, "little") for v in vs), dtype=np.uint64).reshape(-1, 4).copy()


def unpack(a):
    return [int.from_bytes(a[i].tobytes(), "little") for i in range(a.shape[0])]


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def selectors(rng):
    """Pool entries (Montgomery form) of q_m: 0, 1, -1, 2^i (as field elements), the raw values 1 and q - 1, random."""
    mont = lambda x: x * R % Q
    return ([0, 1, Q - 1, mont(1), mont(Q - 1)] + [mont(2 ** i) for i in (1, 31, 32, 33, 64, 128, 200, 254)] +
            [rng.randrange(Q) for _ in range(24)])


def operands(rng):
    """b as stored: below q (edge: 0, 1, q - 1, all-ones limbs below q), and any 256-bit value (the scanned operand need not be reduced)."""
    ones = [(1 << k) - 1 for k in (32, 64, 128, 224, 254)]
    return ([0, 1, 2, Q - 1, Q - 2, R] + ones + [2 ** 256 - 1, 2 ** 256 - 2 ** 32, 2 * Q - 1] +
            [rng.randrange(Q) for _ in range(24)] + [rng.randrange(2 ** 256) for _ in range(8)])


def test_fold_constants(lib):
    rng = random.Random(11)
    s = selectors(rng)
    out = np.zeros((8 * len(s), 4), dtype=np.uint64)
    lib.emu_fold_constants(C.c_uint64(len(s)), vp(pack(s)), vp(out))
    got = unpack(out)
    for k, sv in enumerate(s):
        assert got[8 * k:8 * k + 8] == [sv * RINV * 2 ** (32 * i + 64) % Q for i in range(8)], k


def test_folded_product_matches_big_ints(lib):
    rng = random.Random(12)
    ql_vals = [0, 1, Q - 1, rng.randrange(Q)]
    cases = [(sv, b, rng.choice(ql_vals)) for sv in selectors(rng) for b in operands(rng)]
    cases += [(rng.randrange(Q), rng.randrange(2 ** 256), rng.randrange(Q)) for _ in range(3000)]
    s, b, ql = (pack([c[k] for c in cases]) for k in range(3))
    out = np.zeros_like(s)
    lib.emu_folded_u(C.c_uint64(len(cases)), vp(s), vp(b), vp(ql), vp(out))
    assert lib.emu_violations() == 0
    u = unpack(out)
    for (sv, bv, qv), uv in zip(cases, u):
        assert uv % Q == (sv * bv * RINV + qv) % Q, (hex(sv), hex(bv), hex(qv))
        assert uv < U_BOUND
    worst = max(u)
    assert worst > Q                     # the sum is not reduced: the check below runs at the new maximum


def test_dot_product_takes_the_wider_operand(lib):
    """fr_dot_wide<4> with u at and near its bound in the first slot: no dropped carry, the residue is right, and the result plus q_c and
    PI (each below q) stays below 16q -- the range of the k*q table the zero test reads."""
    rng = random.Random(13)
    us = [U_BOUND - 1, U_BOUND - 2 ** 200, 2 ** 256 - 1, Q + 2 ** 227 - 1] + [rng.randrange(U_BOUND) for _ in range(200)]
    rows = []
    for u in us:
        wires = [rng.choice([Q - 1, rng.randrange(Q)]) for _ in range(4)]
        sels = [u] + [rng.choice([Q - 1, rng.randrange(Q)]) for _ in range(3)]
        rows.append((wires, sels))
    A = pack([w for r in rows for w in r[0]])
    B = pack([x for r in rows for x in r[1]])
    r9 = np.zeros((len(rows), 9), dtype=np.uint32)
    lib.emu_dot4(C.c_uint64(len(rows)), vp(A), vp(B), r9.ctypes.data_as(C.c_void_p))
    assert lib.emu_violations() == 0
    for (wires, sels), limbs in zip(rows, r9):
        r = sum(int(x) << (32 * k) for k, x in enumerate(limbs))
        assert r % Q == sum(a * b for a, b in zip(wires, sels)) * RINV % Q
        assert r + 2 * (Q - 1) < 16 * Q
