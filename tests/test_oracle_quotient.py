"""The recalled constants of the quotient polynomial, re-derived, and the big-int model (tests/quotient_model.py) against the C
restatement (tests/oracle_quotient/quotient.c) on a few programs."""
import numpy as np
import pytest

from oracle import pymodel as pm
from oracle.gen_golden import run_pymodel_composer
from tests import quotient_model as qm
from tests.programs import Q, run_oracle, synth_wide


def test_coset_generator_is_outside_every_domain():
    """7^(2^32) != 1: g^(4N) != 1 for every N <= 2^30, so g*<zeta> misses the 4N-th roots of unity -- x^N - 1 != 0 and x != 1 at every
    point of the coset."""
    assert pow(qm.GENERATOR, 1 << 32, Q) != 1
    assert qm.GENERATOR == pm.GENERATOR


@pytest.mark.parametrize("log_n", [2, 12, 25, 30])
def test_iota_is_a_primitive_fourth_root(log_n):
    zeta = pm.group_gen(log_n + 2)
    assert pow(zeta, 4, Q) == pm.group_gen(log_n)                # zeta^4 = w
    iota = pow(zeta, 1 << log_n, Q)
    assert pow(iota, 4, Q) == 1 and pow(iota, 2, Q) == Q - 1


@pytest.mark.parametrize("name", ["kat_range_check_0_ok", "kat_range_gate_8bits_ok", "batch_is_non_zero_maybe_equal", "kat_select_one_sel1"])
def test_model_matches_c_restatement(oracle, golden, name):
    al, be, ga, rh = synth_wide(172, 4)
    m = run_pymodel_composer(golden[name]["program"])
    _s, oc = run_oracle(golden[name]["program"], return_composer=True)
    log_n = pm.domain_log_size(m.n)
    t, _rem, _num = qm.quotient(m, log_n, al, be, ga, rh)
    got = qm.quot_oracle_t(oracle, oc, log_n, *(oracle.from_ints([v])[0] for v in (al, be, ga, rh)))
    assert [oracle.to_ints(col) for col in got] == t


def test_c_horner(oracle):
    vals = synth_wide(173, 37)
    x = synth_wide(174, 1)[0]
    got = qm.horner_mont(oracle.from_ints(vals), oracle.from_ints([x])[0])
    assert oracle.to_ints(got[None]) == [qm.horner(vals, x)]
    assert np.array_equal(qm.horner_mont(np.zeros((0, 4), np.uint64), oracle.from_ints([x])[0]), np.zeros(4, np.uint64))
