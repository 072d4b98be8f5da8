"""The openings' two test oracles against each other: the big-int model (tests/opening_model.py) and the C restatement
(tests/oracle_openings/openings.c) on a few programs, and the quotient identity on every golden program, which must hold exactly on
the ones whose constraints hold."""
import numpy as np
import pytest

from oracle import pymodel as pm
from oracle.gen_golden import run_pymodel_composer
from tests import opening_model as om
from tests import quotient_model as qm
from tests.programs import Q, synth_wide


@pytest.mark.parametrize("name", ["kat_range_check_0_ok", "kat_range_gate_8bits_ok", "batch_is_non_zero_maybe_equal", "kat_select_one_sel1"])
def test_model_matches_c_restatement(oracle, golden, name):
    ints = synth_wide(195, 7)
    m = run_pymodel_composer(golden[name]["program"])
    log_n = pm.domain_log_size(m.n)
    polys = qm.component_polynomials(m, log_n, ints[1], ints[2])
    t, _rem, _num = qm.quotient(m, log_n, *ints[:4])
    ev, r, wz, wzw, _rems = om.openings_from_polys(polys, t, log_n, *ints)
    mont = lambda cols: np.stack([oracle.from_ints(col) for col in cols])
    ev_c, out_c = om.open_oracle(oracle, mont(polys[:17]), mont(t), log_n, [oracle.from_ints([v])[0] for v in ints])
    assert oracle.to_ints(ev_c) == [ev[k] for k in om.EVALUATIONS]
    assert [oracle.to_ints(col) for col in out_c] == [wz, wzw, r]


def test_c_ruffini_and_evaluate(oracle):
    vals = synth_wide(196, 37)
    for p in (0, 1, Q - 1, synth_wide(197, 1)[0]):
        pm_ = oracle.from_ints([p])[0]
        assert oracle.to_ints(om.c_ruffini(oracle.from_ints(vals), pm_)) == om.ruffini(vals, p)
        assert oracle.to_ints(om.c_evaluate(oracle.from_ints(vals), pm_)[None]) == [om.horner(vals, p)]
    # f = (X - p) q + f(p)
    p = synth_wide(198, 1)[0]
    q = om.ruffini(vals, p)
    rebuilt = [(-p * q[0] + om.horner(vals, p)) % Q] + [(q[i - 1] - p * q[i]) % Q for i in range(1, len(vals))]
    assert rebuilt == vals


def test_quotient_identity_on_golden(golden):
    """The identity holds on every honest golden program and fails on every unsatisfied one (domains up to 2^12)."""
    ints = synth_wide(199, 7)
    seen = {True: 0, False: 0}
    for name, spec in sorted(golden.items()):
        if spec["expected"]["error"] or (1 << pm.domain_log_size(spec["expected"]["n_rows"])) > 1 << 12:
            continue
        m = run_pymodel_composer(spec["program"])
        log_n = pm.domain_log_size(m.n)
        ev, _r, _wz, _wzw, rems, _t, pi_z = om.openings(m, log_n, *ints)
        honest = not spec["expected"]["unsat"]
        assert om.quotient_identity_holds(ev, pi_z, ints[0], ints[1], ints[2], ints[4], 1 << log_n) == honest, name
        assert rems == om.aggregate_values(ev, ints[4], 1 << log_n, ints[5], ints[6]), name
        seen[honest] += 1
    assert seen[True] and seen[False]
