"""CPU tests of the quotient polynomial (pg_selector_polynomials, pg_public_input_polynomial, pg_quotient) through tests/emu: the
engine's host logic, the coset shift of the transform's first pass (ntt_pass_host) and the bodies QuotientBody / QuotientSplitBody run
on the loop backend and are compared with the big-int model of tests/quotient_model.py (its own composer, exact division by X^N - 1)
and the digests of tests/golden/quotient.json.  The CUDA kernels (k_ntt_coset_pass, k_simple<QuotientBody>, k_simple<QuotientSplitBody>)
are checked on the B200 by tests/test_gpu_quotient.py."""
import json
import os
import random

import numpy as np
import pytest

import plonk_gadgets_b200 as pg
from oracle.gen_golden import coeff_digest, run_pymodel_composer
from tests import permutation_model as perm
from tests import quotient_model as qm
from tests.engine_runner import run_engine
from tests.programs import Q, hx, synth_wide, unhx
from tests.test_emu_engine import emu  # noqa: F401  (fixture)

COEFF = pg.api.FORM_COEFFICIENTS


@pytest.fixture(scope="module")
def golden_quot():
    with open(os.path.join(os.path.dirname(__file__), "golden", "quotient.json")) as f:
        return json.load(f)


def _challenges(oracle, golden_quot):
    return [oracle.from_ints([unhx(golden_quot[k])])[0] for k in ("alpha", "beta", "gamma", "range_challenge")]


def _ints(oracle, a):
    return [oracle.to_ints(col) for col in a]


def test_emu_quotient_golden(emu, oracle, golden, golden_quot):
    """Every non-error golden program: selectors and PI in both forms and t_1 .. t_4 equal the model's digests; t_4's top four
    coefficients are zero exactly on the programs whose constraints hold."""
    ch = _challenges(oracle, golden_quot)
    names = [name for name, spec in sorted(golden.items()) if not spec["expected"]["error"]]
    assert sorted(golden_quot["programs"]) == names
    for name in names:
        exp = golden_quot["programs"][name]
        _snap, c = run_engine(golden[name]["program"], lambda: pg.StandardComposer(_cdll=emu), oracle, return_composer=True)
        assert c.domain_log_size() == exp["log_n"], name
        assert coeff_digest(_ints(oracle, c.selector_polynomials())) == exp["selector_evaluations"], name
        assert coeff_digest(_ints(oracle, c.selector_polynomials(form=COEFF))) == exp["selector_coefficients"], name
        assert coeff_digest([oracle.to_ints(c.public_input_polynomial())]) == exp["pi_evaluations"], name
        assert coeff_digest([oracle.to_ints(c.public_input_polynomial(form=COEFF))]) == exp["pi_coefficients"], name
        t = c.quotient(*ch)
        assert coeff_digest(_ints(oracle, t)) == exp["t"], name
        honest = not golden[name]["expected"]["unsat"]
        assert (not t[3, -4:].any()) == honest, name


@pytest.mark.parametrize("name", ["kat_range_check_0_ok", "kat_range_gate_8bits_ok", "batch_mixed_circuit", "batch_is_non_zero_maybe_equal"])
def test_emu_quotient_model(emu, oracle, golden, name):
    """Element by element against the model, at the program's domain and one size larger."""
    al, be, ga, rh = synth_wide(161, 4)
    ch = [oracle.from_ints([v])[0] for v in (al, be, ga, rh)]
    m = run_pymodel_composer(golden[name]["program"])
    _snap, c = run_engine(golden[name]["program"], lambda: pg.StandardComposer(_cdll=emu), oracle, return_composer=True)
    for log_n in (c.domain_log_size(), c.domain_log_size() + 1):
        sel = qm.selector_evaluations(m, log_n)
        assert _ints(oracle, c.selector_polynomials(log_n)) == sel
        assert _ints(oracle, c.selector_polynomials(log_n, form=COEFF)) == [perm.ifft(s) for s in sel]
        pi = qm.public_input_evaluations(m, log_n)
        assert oracle.to_ints(c.public_input_polynomial(log_n)) == pi
        assert oracle.to_ints(c.public_input_polynomial(log_n, form=COEFF)) == perm.ifft(pi)
        t, _rem, _num = qm.quotient(m, log_n, al, be, ga, rh)
        assert _ints(oracle, c.quotient(*ch, log_n=log_n)) == t


def _identity_holds(oracle, t, num, log_n, x):
    """(t_1(x) + x^N t_2(x) + x^2N t_3(x) + x^3N t_4(x)) (x^N - 1) == N(x), with N(X) the model's numerator polynomial."""
    n = 1 << log_n
    xn = pow(x, n, Q)
    parts = [qm.horner(oracle.to_ints(t[r]), x) for r in range(4)]
    lhs = sum(p * pow(xn, r, Q) for r, p in enumerate(parts)) * (xn - 1) % Q
    return lhs == qm.horner(num, x)


def _two_range_checks():
    vals = [v & ((1 << 64) - 1) for v in synth_wide(162, 2)]
    return [dict(op="add_input", values=[hx(v) for v in vals]), dict(op="range_check", min=hx(0), max=hx(1 << 64), witness=0)]


# Stored Variables of _two_range_checks (k = 65 bits: 653 Variables per instance after the 5 of the fresh composer and the 2 inputs;
# offset 0 is V, 1 .. 256 the packed bits, then the accumulators, the last one U): the inputs, and V, an accumulator and U of the first
# and of the last instance of the segment
POKES = [5, 6] + [7 + 653 * i + off for i in (0, 1) for off in (0, 259, 652)]


def test_emu_quotient_degree_and_identity(emu, oracle):
    """Honest: the top four coefficients of t_4 are zero, the model's division is exact and the identity holds at a seeded random point.
    After a poke of a stored Variable (V, an accumulator, U; first and last instance of the segment): top coefficients non-zero, the
    model's remainder non-zero, the identity fails."""
    al, be, ga, rh = synth_wide(163, 4)
    ch = [oracle.from_ints([v])[0] for v in (al, be, ga, rh)]
    prog = _two_range_checks()
    x = random.Random(164).randrange(Q)
    _snap, c = run_engine(prog, lambda: pg.StandardComposer(_cdll=emu), oracle, return_composer=True)
    log_n = c.domain_log_size()
    m = run_pymodel_composer(prog)
    t = c.quotient(*ch)
    _tm, rem, num = qm.quotient(m, log_n, al, be, ga, rh)
    assert not any(rem) and not t[3, -4:].any() and _identity_holds(oracle, t, num, log_n, x)
    for var in POKES:
        _snap, c = run_engine(prog, lambda: pg.StandardComposer(_cdll=emu), oracle, return_composer=True)
        m = run_pymodel_composer(prog)
        value = (m.variables[var] + 3) % Q
        c.poke_variable(var, oracle.from_ints([value])[0])
        m.variables[var] = value
        t = c.quotient(*ch)
        _tm, rem, num = qm.quotient(m, log_n, al, be, ga, rh)
        assert any(rem), var
        assert t[3, -4:].any(), var
        assert not _identity_holds(oracle, t, num, log_n, x), var


def test_emu_quotient_errors(emu, oracle, golden):
    spec = golden["kat_range_check_0_ok"]
    _snap, c = run_engine(spec["program"], lambda: pg.StandardComposer(_cdll=emu), oracle, return_composer=True)
    k = c.domain_log_size()
    ch = [oracle.from_ints([v])[0] for v in synth_wide(165, 4)]
    for bad_log_n in (k - 1, 31, 33):
        with pytest.raises(pg.EngineError) as e:
            c.quotient(*ch, log_n=bad_log_n)
        assert e.value.code == -2, bad_log_n
    small = np.zeros((4, 1 << k, 4), dtype=np.uint64)          # the engine itself refuses before it writes anything
    vp = lambda a: a.ctypes.data_as(pg.api.C.c_void_p)
    for bad_log_n in (31, 33):
        assert c._L.pg_quotient(c._ctx, bad_log_n, *map(vp, ch), vp(small), 0) == -2
        assert "2^30" in c._L.pg_last_error(c._ctx).decode()
    for fn in (c.selector_polynomials, c.public_input_polynomial):
        with pytest.raises(pg.EngineError) as e:
            fn(k - 1)
        assert e.value.code == -2
    unreduced = np.array([0xFFFFFFFF00000001, 0x53BDA402FFFE5BFE, 0x3339D80809A1D805, 0x73EDA753299D7D48], dtype=np.uint64)   # q itself
    for i in range(4):
        bad = list(ch); bad[i] = unreduced
        with pytest.raises(pg.EngineError) as e:
            c.quotient(*bad)
        assert e.value.code == -2 and "reduced" in str(e.value), i
    zero = oracle.from_ints([0])[0]
    with pytest.raises(pg.EngineError) as e:                   # beta = gamma = 0: the zero variable's rows have a zero z denominator
        c.quotient(ch[0], zero, zero, ch[3])
    assert e.value.code == -2 and "zero denominator" in str(e.value) and "first at row 0" in str(e.value)
    t = c.quotient(*ch)                                        # afterwards the ctx still computes
    assert t.shape == (4, 1 << k, 4) and not t[3, -4:].any() and t.any()
