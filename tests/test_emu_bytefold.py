"""CPU tests of the generic gate check's tensor-core row (kernels.cuh k_check_tc) through its host emulation: the byte-fold blocks
(layout.h byte_fold_block) against big ints and an independent model of the MMA's shared-memory layout, the column merge and the
zero test (fr.cuh add_byte_columns, limbs9_is_small_multiple_of_q) with no dropped carry, and whole rows against big-int verdicts."""
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
COL_MAX = 96 * 255 * 255            # one s32 column of the 128 x 96 x 32 u8 product
S_BOUND = 24484 * Q                 # a*u < 2q, the columns < 96*255*q, q_c + PI < 2q


@pytest.fixture(scope="module")
def lib():
    out = os.path.join(EMU_DIR, "_build", "libbytefold_emu.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    src = os.path.join(EMU_DIR, "bytefold_emu.cpp")
    deps = [src] + [os.path.join(ROOT, "plonk_gadgets_b200", "csrc", f) for f in ("fr.cuh", "layout.h")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out, src], check=True)
    return C.CDLL(out)


def pack(vs):
    return np.frombuffer(b"".join(v.to_bytes(32, "little") for v in vs), dtype=np.uint64).reshape(-1, 4).copy()


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def limbs9(v):
    return np.array([(v >> (32 * k)) & 0xffffffff for k in range(9)], dtype=np.uint32)


def value9(a):
    return sum(int(x) << (32 * k) for k, x in enumerate(a))


def selectors(rng):
    """Pool entries (Montgomery form): 0, 1 and -1 as field elements, the raw values 1 and q - 1, powers of two, random."""
    mont = lambda x: x * R % Q
    return [0, mont(1), mont(Q - 1), 1, Q - 1] + [mont(2 ** i) for i in (1, 63, 200)] + [rng.randrange(Q) for _ in range(12)]


def model_block(s):
    """The B operand of one selector as the int8 MMA reads it: K-major, no swizzle, core matrices of 8 rows (output byte j) x 16
    bytes (K index k); the core matrices along j are 128 bytes apart (SBO), the two 16-byte K chunks 512 bytes apart (LBO)."""
    blk = bytearray(1024)
    for k in range(32):
        f = s * 2 ** (8 * k) * RINV % Q
        for j in range(32):
            blk[(k // 16) * 512 + (j // 8) * 128 + (j % 8) * 16 + k % 16] = (f >> (8 * j)) & 0xff
    return bytes(blk)


def test_byte_fold_blocks_match_the_model(lib):
    s = selectors(random.Random(21))
    out = np.zeros(1024 * len(s), dtype=np.uint8)
    lib.emu_byte_fold_blocks(C.c_uint64(len(s)), vp(pack(s)), vp(out))
    for i, sv in enumerate(s):
        assert out[1024 * i:1024 * (i + 1)].tobytes() == model_block(sv), hex(sv)


def test_byte_fold_identity():
    """sum_k w_k * F_k == s*w*R^-1 (mod q) for any 256-bit w, and the value is below 255*32*q (F_k < q)."""
    rng = random.Random(22)
    for s in selectors(rng):
        F = [s * 2 ** (8 * k) * RINV % Q for k in range(32)]
        for w in [0, 1, Q - 1, R, 2 ** 256 - 1] + [rng.randrange(2 ** 256) for _ in range(4)]:
            L = sum(((w >> (8 * k)) & 0xff) * F[k] for k in range(32))
            assert L % Q == s * w * RINV % Q and L < 255 * 32 * Q


def test_column_merge_and_zero_test(lib):
    """add_byte_columns adds exactly sum_j c_j*2^(8j) with no dropped carry, for columns at their maximum and random ones, on top of a
    start value at the bound of the integer part (below 4q); below 2^15*q the zero test agrees with big ints on multiples of q and
    their neighbours."""
    rng = random.Random(23)
    cols, starts = [], []
    for _ in range(400):
        kind = rng.randrange(4)
        c = ([COL_MAX] * 32 if kind == 0 else [rng.randrange(COL_MAX + 1) for _ in range(32)] if kind == 1 else
             [rng.choice([0, COL_MAX, COL_MAX - 1]) for _ in range(32)] if kind == 2 else [rng.randrange(256) for _ in range(32)])
        L = sum(x << (8 * j) for j, x in enumerate(c))
        t0 = rng.choice([0, 4 * Q - 1, rng.randrange(4 * Q)])
        if rng.random() < 0.5:       # make the sum a multiple of q, or one off it
            t0 = (t0 - (t0 + L) % Q) + rng.choice([0, 0, 1, -1, Q])
            if t0 < 0:
                t0 += Q
        cols.append(c)
        starts.append(t0)
    t9 = np.stack([limbs9(v) for v in starts])
    cc = np.array(cols, dtype=np.uint32)
    ok = np.zeros(len(cols), dtype=np.uint8)
    lib.emu_add_columns(C.c_uint64(len(cols)), vp(t9), vp(cc), vp(ok))
    assert lib.emu_violations() == 0
    n_zero = 0
    for k, (c, t0) in enumerate(zip(cols, starts)):
        S = t0 + sum(x << (8 * j) for j, x in enumerate(c))
        assert value9(t9[k]) == S
        if S < 2 ** 15 * Q:          # the range of the zero test (arbitrary columns go beyond what a row can produce)
            assert bool(ok[k]) == (S % Q == 0), k
            n_zero += S % Q == 0
    assert n_zero > 50


def test_zero_test_range():
    """S == k*q with k = S[0] < 2^15 is the whole range the merged sum can take: 24484*q < 2^15*q."""
    assert S_BOUND < 2 ** 15 * Q and 24484 * Q < 2 ** 270


def test_generic_rows_match_big_ints(lib):
    """Whole rows (folded q_m*b, the dot product, the modelled MMA columns, q_c + PI, zero test) with edge and random wires and
    selectors, satisfied and unsatisfied, against a big-int evaluation of the gate; S stays below 24484*q."""
    rng = random.Random(24)
    sels = selectors(rng)
    a_vals = [0, 1, Q - 1, R]
    w_vals = [0, 1, Q - 1, R, 2 ** 256 - 1, 2 * Q - 1]
    rows = []
    for n in range(1500):
        a = rng.choice(a_vals + [rng.randrange(Q)])
        b, c, d = (rng.choice(w_vals + [rng.randrange(Q), rng.randrange(2 ** 256)]) for _ in range(3))
        qm, ql, qr, qo, q4 = (rng.choice(sels) for _ in range(5))
        if n < 40:                                           # all at their extremes
            a, b, c, d, qm, ql, qr, qo, q4 = Q - 1, 2 ** 256 - 1, 2 ** 256 - 1, 2 ** 256 - 1, Q - 1, Q - 1, Q - 1, Q - 1, Q - 1
        rest = (a * (qm * b * RINV + ql) * RINV + (qr * b + qo * c + q4 * d) * RINV) % Q
        qc_pi = (Q - rest) % Q + rng.choice([0, 0, Q, 1, rng.randrange(1, Q)])
        rows.append(((a, b, c, d), (qm, ql, qr, qo, q4, qc_pi)))
    W = pack([x for r in rows for x in r[0]])
    Sx = pack([x for r in rows for x in r[1]])
    S = np.zeros((len(rows), 9), dtype=np.uint32)
    ok = np.zeros(len(rows), dtype=np.uint8)
    lib.emu_generic_row(C.c_uint64(len(rows)), vp(W), vp(Sx), vp(S), vp(ok))
    assert lib.emu_violations() == 0
    n_ok = 0
    for k, ((a, b, c, d), (qm, ql, qr, qo, q4, qc_pi)) in enumerate(rows):
        gate = (a * (qm * b * RINV + ql) * RINV + (qr * b + qo * c + q4 * d) * RINV + qc_pi) % Q
        s = value9(S[k])
        assert s % Q == gate and s < S_BOUND
        assert bool(ok[k]) == (gate == 0), k
        n_ok += gate == 0
    assert 100 < n_ok < len(rows) - 100
