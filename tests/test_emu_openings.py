"""CPU tests of prover rounds 4 and 5 (pg_prover_openings, pg_fr_op 8) through tests/emu: the engine's host logic and the bodies
OpenEvalBody / OpenSumBody / OpenCombineBody run on the loop backend, the Ruffini division as its defining serial body
(FrRuffiniSerialBody), all compared with the big-int model of tests/opening_model.py and the digests of tests/golden/openings.json.
The CUDA kernels (the k_simple instantiations and the Ruffini scan k_fr_ruffini_reduce / k_fr_ruffini_apply) are checked on the B200
by tests/test_gpu_openings.py."""
import json
import os
import random

import numpy as np
import pytest

import plonk_gadgets_b200 as pg
from oracle import pymodel as pm
from oracle.gen_golden import coeff_digest, run_pymodel_composer
from tests import opening_model as om
from tests.engine_runner import run_engine
from tests.programs import Q, synth_wide, unhx
from tests.test_emu_engine import emu  # noqa: F401  (fixture)
from tests.test_emu_quotient import POKES, _two_range_checks

COEFF = pg.api.FORM_COEFFICIENTS


@pytest.fixture(scope="module")
def golden_open():
    with open(os.path.join(os.path.dirname(__file__), "golden", "openings.json")) as f:
        return json.load(f)


def _ev_ints(oracle, ev):
    return {k: oracle.to_ints(ev[k][None])[0] for k in om.EVALUATIONS}


def _composer(emu, program, oracle):
    _snap, c = run_engine(program, lambda: pg.StandardComposer(_cdll=emu), oracle, return_composer=True)
    return c


def test_emu_openings_golden(emu, oracle, golden, golden_open):
    """Every non-error golden program: the evaluations, r, W_z and W_zw equal the model's digests; the quotient identity holds exactly
    on the programs whose constraints hold."""
    ints = [unhx(x) for x in golden_open["challenges"]]
    ch = [oracle.from_ints([v])[0] for v in ints]
    names = [name for name, spec in sorted(golden.items()) if not spec["expected"]["error"]]
    assert sorted(golden_open["programs"]) == names
    for name in names:
        exp = golden_open["programs"][name]
        c = _composer(emu, golden[name]["program"], oracle)
        t = c.quotient(*ch[:4])
        ev, out = c.prover_openings(t, *ch)
        evi = _ev_ints(oracle, ev)
        assert coeff_digest([[evi[k] for k in om.EVALUATIONS]]) == exp["evaluations"], name
        assert coeff_digest([oracle.to_ints(out[2])]) == exp["r"], name
        assert coeff_digest([oracle.to_ints(out[0])]) == exp["w_z"], name
        assert coeff_digest([oracle.to_ints(out[1])]) == exp["w_zw"], name
        n = 1 << exp["log_n"]
        pi_z = om.horner(oracle.to_ints(c.public_input_polynomial(form=COEFF)), ints[4])
        assert om.quotient_identity_holds(evi, pi_z, ints[0], ints[1], ints[2], ints[4], n) == (not golden[name]["expected"]["unsat"]), name


@pytest.mark.parametrize("name", ["kat_range_check_0_ok", "kat_range_gate_8bits_ok", "batch_mixed_circuit", "batch_is_non_zero_maybe_equal"])
def test_emu_openings_model(emu, oracle, golden, name):
    """Element by element against the model, at the program's domain and one size larger."""
    ints = synth_wide(181, 7)
    ch = [oracle.from_ints([v])[0] for v in ints]
    m = run_pymodel_composer(golden[name]["program"])
    c = _composer(emu, golden[name]["program"], oracle)
    for log_n in (c.domain_log_size(), c.domain_log_size() + 1):
        ev_m, r, wz, wzw, _rems, t, _pi = om.openings(m, log_n, *ints)
        t_mont = np.stack([oracle.from_ints(col) for col in t])
        ev, out = c.prover_openings(t_mont, *ch, log_n=log_n)
        assert _ev_ints(oracle, ev) == ev_m
        assert [oracle.to_ints(col) for col in out] == [wz, wzw, r]


@pytest.mark.parametrize("n", [1, 2, 1023, 1024, 1025, 3 * 1024 + 7])
def test_emu_fr_op_ruffini(emu, oracle, n):
    """pg_fr_op 8 (in place on its staged copy) against the textbook division and Horner, for p in {0, 1, -1, w, random}."""
    c = pg.StandardComposer(_cdll=emu)
    vals = synth_wide(182 + n, n)
    a = oracle.from_ints(vals)
    for p in (0, 1, Q - 1, pm.group_gen(10), synth_wide(183, 1)[0]):
        got = oracle.to_ints(c.fr_op(8, a, oracle.from_ints([p])))
        assert got[:n - 1] == om.ruffini(vals, p)[:n - 1], p
        assert got[n - 1] == om.horner(vals, p), p
    c.close()


def _engine_polys(c, oracle, ch, log_n):
    """The engine's coefficient vectors as ints: wires, z, sigma (each checked against the oracles by the earlier tests)."""
    return ([oracle.to_ints(x) for x in c.wire_polynomials(log_n)] + [oracle.to_ints(c.permutation_z(ch[1], ch[2], log_n, form=COEFF)[0])]
            + [oracle.to_ints(x) for x in c.sigma_polynomials(log_n, form=COEFF)])


def _openings_hold(oracle, c, t, ev, out, ints, ch, log_n, x):
    """(x - p) W(x) == agg(x) - agg(p) at both points, agg(p) formed from the evaluations."""
    n = 1 << log_n
    z, v, vs = ints[4], ints[5], ints[6]
    zw = z * pm.group_gen(log_n) % Q
    polys = _engine_polys(c, oracle, ch, log_n)
    h = lambda p: om.horner(p, x)
    zn = pow(z, n, Q)
    quot = sum(pow(zn, r, Q) * h(oracle.to_ints(t[r])) for r in range(4))
    at_x = [quot, h(oracle.to_ints(out[2]))] + [h(polys[k]) for k in range(4)] + [h(polys[5 + k]) for k in range(3)]
    agg_x = sum(pow(v, k, Q) * y for k, y in enumerate(at_x)) % Q
    agg_xw = sum(pow(vs, k, Q) * y for k, y in enumerate([h(polys[4]), h(polys[0]), h(polys[1]), h(polys[3])])) % Q
    agg_z, agg_zw = om.aggregate_values(_ev_ints(oracle, ev), z, n, v, vs)
    ok_z = (x - z) * h(oracle.to_ints(out[0])) % Q == (agg_x - agg_z) % Q
    ok_zw = (x - zw) * h(oracle.to_ints(out[1])) % Q == (agg_xw - agg_zw) % Q
    return ok_z and ok_zw


def test_emu_openings_identities(emu, oracle):
    """Honest: the quotient identity and both opening identities hold (seeded random x).  After each poke of test_emu_quotient.py's
    POKES: the openings still hold (they are exact divisions of whatever was committed) and the quotient identity fails."""
    ints = synth_wide(184, 7)
    ch = [oracle.from_ints([v])[0] for v in ints]
    prog = _two_range_checks()
    x = random.Random(185).randrange(Q)
    for var in [None] + POKES:
        c = _composer(emu, prog, oracle)
        if var is not None:
            value = (oracle.to_ints(c.variables(var, 1))[0] + 3) % Q
            c.poke_variable(var, oracle.from_ints([value])[0])
        log_n = c.domain_log_size()
        t = c.quotient(*ch[:4])
        ev, out = c.prover_openings(t, *ch)
        pi_z = om.horner(oracle.to_ints(c.public_input_polynomial(form=COEFF)), ints[4])
        assert om.quotient_identity_holds(_ev_ints(oracle, ev), pi_z, ints[0], ints[1], ints[2], ints[4], 1 << log_n) == (var is None), var
        assert _openings_hold(oracle, c, t, ev, out, ints, ch, log_n, x), var


def test_emu_openings_errors(emu, oracle, golden):
    c = _composer(emu, golden["kat_range_check_0_ok"]["program"], oracle)
    k = c.domain_log_size()
    n = 1 << k
    ints = synth_wide(186, 7)
    ch = [oracle.from_ints([v])[0] for v in ints]
    t = c.quotient(*ch[:4])
    ev0, out0 = c.prover_openings(t, *ch)

    def code(fn):
        with pytest.raises(pg.EngineError) as e:
            fn()
        return e.value.code, str(e.value)

    for bad_log_n in (k - 1, 31, 33):
        tt = np.zeros((4, 1 << bad_log_n, 4), np.uint64) if bad_log_n < 31 else t
        assert code(lambda: c.prover_openings(tt, *ch, log_n=bad_log_n))[0] == -2, bad_log_n
    vp = lambda a: a.ctypes.data_as(pg.api.C.c_void_p)
    chs = np.ascontiguousarray(np.stack(ch))
    evbuf = np.zeros((17, 4), np.uint64)
    dst = np.zeros((3, n, 4), np.uint64)
    L = c._L
    for bad_log_n in (31, 33):                                  # the engine itself refuses before it writes anything
        assert L.pg_prover_openings(c._ctx, bad_log_n, vp(chs), vp(t), 0, vp(evbuf), vp(dst), 0) == -2
        assert "2^30" in L.pg_last_error(c._ctx).decode()
    for args in ((None, vp(t), vp(evbuf), vp(dst)), (vp(chs), None, vp(evbuf), vp(dst)), (vp(chs), vp(t), None, vp(dst)), (vp(chs), vp(t), vp(evbuf), None)):
        assert L.pg_prover_openings(c._ctx, k, args[0], args[1], 0, args[2], args[3], 0) == -2
        assert "null" in L.pg_last_error(c._ctx).decode()
    unreduced = np.array([0xFFFFFFFF00000001, 0x53BDA402FFFE5BFE, 0x3339D80809A1D805, 0x73EDA753299D7D48], dtype=np.uint64)   # q itself
    for i in range(7):
        bad = list(ch); bad[i] = unreduced
        cd, msg = code(lambda: c.prover_openings(t, *bad))
        assert cd == -2 and "reduced" in msg, i
    tb = t.copy(); tb[2, 5] = unreduced
    cd, msg = code(lambda: c.prover_openings(tb, *ch))
    assert cd == -2 and "of t not fully reduced" in msg and f"first at index {2 * n + 5}" in msg
    for z in (1, pm.group_gen(k), pow(pm.group_gen(k), 3, Q)):  # zeta^N = 1
        bad = list(ch); bad[4] = oracle.from_ints([z])[0]
        cd, msg = code(lambda: c.prover_openings(t, *bad))
        assert cd == -2 and "zeta^N = 1" in msg, z
    zero = oracle.from_ints([0])[0]                             # beta = gamma = 0: the zero variable's rows have a zero z denominator
    cd, msg = code(lambda: c.prover_openings(t, ch[0], zero, zero, *ch[3:]))
    assert cd == -2 and "zero denominator" in msg and "first at row 0" in msg
    ev, out = c.prover_openings(t, *ch)                         # afterwards the ctx still computes, and the same
    assert all(np.array_equal(ev[k], ev0[k]) for k in om.EVALUATIONS) and np.array_equal(out, out0)
