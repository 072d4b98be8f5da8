"""CPU tests of pg_srs_lagrange_from_powers (the group inverse FFT of g1fft.cuh) through tests/emu: the ingest, stage and
normalisation bodies and the fixed-window scalar multiplication run on the loop backend, for domains up to 2^7, against the
big-int model (oracle/pymodel.py), pg_srs_lagrange, the C restatement tests/oracle_lagrange/group_fft.c and the definition sum.
The CUDA launches are checked on the B200 by tests/test_gpu_srs_lagrange.py."""
import ctypes as C
import random

import numpy as np
import pytest

import plonk_gadgets_b200 as pg
from oracle import pymodel as pm
from tests import lagrange_model as lm
from tests.engine_runner import run_engine
from tests.programs import Q
from tests.test_emu_engine import emu  # noqa: F401  (fixture)
from tests.test_emu_msm import to_engine, to_oracle

BETA = 0x2c5e1f0a9b8d7c6e5f4a3b2c1d0e9f8a7b6c5d4e3f2a1b0c9d8e7f6a5b4c3d2e % Q


@pytest.mark.parametrize("log_n", [0, 1, 2, 3, 4, 6])
def test_emu_from_powers_equals_srs_lagrange(emu, oracle, log_n):
    """srs_powers(beta, base) -> the Lagrange form equals pymodel.srs_lagrange and pg_srs_lagrange, for a random beta, beta = 0
    (powers G, O, O, ...: every output is G/n) and beta = 2, with the generator and with another base."""
    c = pg.StandardComposer(_cdll=emu)
    n = 1 << log_n
    other = pm.g1_mul(0x1234567, pm.G1_GENERATOR)
    for beta in (BETA, 0, 2):
        b = oracle.from_ints([beta])[0]
        for base in (None, other):
            eb = None if base is None else to_engine(oracle.g1_from_ints([base]))[0]
            got = c.srs_lagrange_from_powers(c.srs_powers(b, n, base=eb), log_n)
            assert oracle.g1_to_ints(to_oracle(got)) == pm.srs_lagrange(beta, log_n, base or pm.G1_GENERATOR), (beta, base, log_n)
            assert np.array_equal(got, c.srs_lagrange(b, log_n, base=eb)), (beta, base, log_n)


@pytest.mark.parametrize("log_n", [2, 4, 6])
def test_emu_arbitrary_points(emu, oracle, log_n):
    """P_j = k_j G with infinity and opposite pairs among them: the output is (ifft k)_i G, and equals the C restatement (and, up
    to 2^4, the big-int definition sum)."""
    c = pg.StandardComposer(_cdll=emu)
    n = 1 << log_n
    rnd = random.Random(100 + log_n)
    ks = [rnd.randrange(Q) for _ in range(n)]
    ks[0] = 0                                                   # infinity
    ks[1] = Q - ks[n - 1]                                       # P_1 = -P_(n-1)
    if n >= 8:
        ks[5] = 0; ks[3] = ks[2]; ks[6] = Q - ks[2]             # a repeated point and its opposite
    pts13 = oracle.g1_mul(np.repeat(oracle.g1_generator(), n, axis=0), oracle.from_ints(ks))
    got = c.srs_lagrange_from_powers(to_engine(pts13), log_n)
    want = c.g1_fixed_base_mul(oracle.from_ints(lm.scalar_ifft(ks, log_n)))
    assert np.array_equal(got, want)
    assert np.array_equal(to_oracle(got), lm.group_ifft(pts13, log_n))
    if log_n <= 4:
        assert oracle.g1_to_ints(to_oracle(got)) == lm.definition_sum(oracle.g1_to_ints(pts13), log_n)


def test_emu_reads_only_the_first_n_powers(emu, oracle):
    c = pg.StandardComposer(_cdll=emu)
    powers = c.srs_powers(oracle.from_ints([BETA])[0], 16 + 5)
    tail = powers.copy(); tail[16:] = to_engine(oracle.g1_mul(oracle.g1_generator(), oracle.from_ints([77])))
    want = c.srs_lagrange_from_powers(powers[:16], 4)
    assert np.array_equal(c.srs_lagrange_from_powers(powers, 4), want)
    assert np.array_equal(c.srs_lagrange_from_powers(tail, 4), want)
    assert np.array_equal(c.srs_lagrange_from_powers(powers, 0), powers[:1])        # log_n = 0 copies powers_of_g[0]


def test_emu_argument_errors(emu, oracle):
    c = pg.StandardComposer(_cdll=emu)
    powers = c.srs_powers(oracle.from_ints([BETA])[0], 8)
    out = np.zeros((8, 12), dtype=np.uint64)
    pp, op = powers.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)
    f = c._L.pg_srs_lagrange_from_powers
    assert f(c._ctx, 3, None, 8, 0, op, 0) == -2                # null powers
    assert f(c._ctx, 3, pp, 8, 0, None, 0) == -2                # null output
    assert f(c._ctx, 33, pp, 8, 0, op, 0) == -2                 # beyond the two-adicity of Fr
    assert f(c._ctx, 3, pp, 7, 0, op, 0) == -2                  # fewer powers than the domain
    assert f(c._ctx, 3, pp, 8, 0, op, 0) == 0
    with pytest.raises(pg.EngineError) as e:
        c.srs_lagrange_from_powers(powers[:4], 3)
    assert e.value.code == -2


def test_emu_commitments_from_derived_basis(emu, oracle, golden):
    """The wire commitments taken from the wire values against the derived Lagrange form equal those of the wire polynomials
    against the monomial powers."""
    _snap, c = run_engine(golden["kat_range_check_0_ok"]["program"], lambda: pg.StandardComposer(_cdll=emu), oracle, return_composer=True)
    k = c.domain_log_size()
    mono = c.srs_powers(oracle.from_ints([BETA])[0], 1 << k)
    assert np.array_equal(c.commit_wire_evaluations(c.srs_lagrange_from_powers(mono, k)), c.commit_wire_polynomials(mono))


def test_c_restatement_matches_definition(oracle):
    """The C restatement against the big-int definition sum, on random points with infinity and an opposite pair."""
    rnd = random.Random(5)
    for log_n in (0, 1, 3):
        n = 1 << log_n
        pts = [pm.g1_mul(rnd.randrange(Q), pm.G1_GENERATOR) for _ in range(n)]
        if n >= 8:
            pts[2] = None
            pts[4] = pm.g1_neg(pts[6])
        got = oracle.g1_to_ints(lm.group_ifft(oracle.g1_from_ints(pts), log_n))
        assert got == lm.definition_sum(pts, log_n), log_n
