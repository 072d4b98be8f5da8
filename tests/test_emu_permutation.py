"""CPU tests of the permutation argument (pg_sigma_polynomials, pg_permutation_z, pg_permutation_z_rows, pg_fr_op 7) through
tests/emu: the engine's host logic and the bodies PermSigmaBody / PermRatioHook run on the loop backend and are compared with
the big-int loops of tests/permutation_model.py, the C restatement (tests/oracle_perm/permutation.c) and the digests of tests/golden/permutation.json.
The CUDA kernels (k_simple<PermSigmaBody>, k_batch_inv<PermRatioHook>, k_fr_scan_*) are checked on the B200 by tests/test_gpu_permutation.py."""
import json
import os

import numpy as np
import pytest

import plonk_gadgets_b200 as pg
from oracle.gen_golden import coeff_digest, run_pymodel_composer
from tests import permutation_model as perm
from tests.engine_runner import run_engine
from tests.programs import Q, run_oracle, synth_wide, unhx
from tests.test_emu_engine import emu  # noqa: F401  (fixture)

COEFF = pg.api.FORM_COEFFICIENTS


@pytest.fixture(scope="module")
def golden_perm():
    with open(os.path.join(os.path.dirname(__file__), "golden", "permutation.json")) as f:
        return json.load(f)


def _ok_programs(golden):
    return [name for name, spec in sorted(golden.items()) if not spec["expected"]["error"]]


def test_emu_permutation_golden(emu, oracle, golden, golden_perm):
    """Every non-error golden program: sigma and z in both forms equal the digests of the model, z equals the C oracle, closing = 1,
    and the rows path fed the materialised rows and pg_permutation gives the same z."""
    beta, gamma = (oracle.from_ints([unhx(golden_perm[k])]) for k in ("beta", "gamma"))
    names = _ok_programs(golden)
    assert sorted(golden_perm["programs"]) == names
    for name in names:
        exp = golden_perm["programs"][name]
        _snap, c = run_engine(golden[name]["program"], lambda: pg.StandardComposer(_cdll=emu), oracle, return_composer=True)
        log_n = c.domain_log_size()
        assert log_n == exp["log_n"], name
        ints = lambda a: [oracle.to_ints(col) for col in a]
        assert coeff_digest(ints(c.sigma_polynomials())) == exp["sigma_evaluations"], name
        assert coeff_digest(ints(c.sigma_polynomials(form=COEFF))) == exp["sigma_coefficients"], name
        z, closing = c.permutation_z(beta, gamma)
        assert oracle.to_ints(closing[None]) == [1], name
        assert coeff_digest([oracle.to_ints(z)]) == exp["z_evaluations"], name
        zc, closing2 = c.permutation_z(beta, gamma, form=COEFF)
        assert coeff_digest([oracle.to_ints(zc)]) == exp["z_coefficients"] and np.array_equal(closing2, closing), name
        _s, oc = run_oracle(golden[name]["program"], return_composer=True)
        osig, oz, oclosing = perm.perm_oracle_z(oracle, oc, log_n, beta, gamma)
        assert np.array_equal(z, oz) and np.array_equal(c.sigma_polynomials(), osig) and np.array_equal(closing, oclosing), name
        rows = c.rows(want=("w_val",))
        zr, cr = c.permutation_z_rows(rows["w_val"], c.permutation(), beta, gamma, log_n)
        assert np.array_equal(zr, z) and np.array_equal(cr, closing), name


@pytest.mark.parametrize("name", ["kat_range_check_0_ok", "batch_is_non_zero_maybe_equal", "kat_range_gate_8bits_ok", "kat_select_one_sel1"])
def test_emu_permutation_model(emu, oracle, golden, name):
    """Element by element against the defining loops of the model (its own variable map), at a larger domain than needed too."""
    beta, gamma = synth_wide(120, 2)
    m = run_pymodel_composer(golden[name]["program"])
    _snap, c = run_engine(golden[name]["program"], lambda: pg.StandardComposer(_cdll=emu), oracle, return_composer=True)
    for log_n in (c.domain_log_size(), c.domain_log_size() + 1):
        sig = perm.sigma_evaluations(m, log_n)
        assert [oracle.to_ints(col) for col in c.sigma_polynomials(log_n)] == sig
        assert [oracle.to_ints(col) for col in c.sigma_polynomials(log_n, form=COEFF)] == [perm.ifft(col) for col in sig]
        z, closing = perm.permutation_z(m, log_n, beta, gamma)
        got, got_closing = c.permutation_z(oracle.from_ints([beta]), oracle.from_ints([gamma]), log_n)
        assert oracle.to_ints(got) == z and oracle.to_ints(got_closing[None]) == [closing] == [1]
        got_c, _ = c.permutation_z(oracle.from_ints([beta]), oracle.from_ints([gamma]), log_n, form=COEFF)
        assert oracle.to_ints(got_c) == perm.ifft(z)


@pytest.mark.parametrize("n", [1, 2, 3, 31, 32, 33, 1023, 1024, 1025, 3000])
def test_emu_fr_op_prefix_product(emu, oracle, n):
    vals = synth_wide(130 + n, n)
    vals[n // 2] = 0 if n > 4 else vals[n // 2]                # a zero in the middle: every later prefix is 0
    c = pg.StandardComposer(_cdll=emu)
    out = oracle.to_ints(c.fr_op(7, oracle.from_ints(vals)))
    acc, exp = 1, []
    for v in vals:
        exp.append(acc)
        acc = acc * v % Q
    assert out == exp


def test_emu_permutation_errors(emu, oracle, golden):
    spec = golden["kat_range_check_0_ok"]
    _snap, c = run_engine(spec["program"], lambda: pg.StandardComposer(_cdll=emu), oracle, return_composer=True)
    k = c.domain_log_size()
    beta, gamma = oracle.from_ints(synth_wide(140, 2))
    for bad_log_n in (k - 1, 33):
        with pytest.raises(pg.EngineError) as e:
            c.permutation_z(beta, gamma, bad_log_n)
        assert e.value.code == -2
        with pytest.raises(pg.EngineError):
            c.sigma_polynomials(bad_log_n)
    zero = oracle.from_ints([0])[0]
    with pytest.raises(pg.EngineError) as e:                   # beta = gamma = 0: the zero variable's rows have den = 0
        c.permutation_z(zero, zero)
    assert e.value.code == -2 and "zero denominator" in str(e.value) and "first at row 0" in str(e.value)
    unreduced = np.array([0xFFFFFFFF00000001, 0x53BDA402FFFE5BFE, 0x3339D80809A1D805, 0x73EDA753299D7D48], dtype=np.uint64)   # q itself
    with pytest.raises(pg.EngineError) as e:
        c.permutation_z(unreduced, gamma)
    assert e.value.code == -2 and "reduced" in str(e.value)
    rows, sigma = c.rows(want=("w_val",))["w_val"], c.permutation()
    bad = sigma.copy(); bad[2, 5] = 4 << k                     # one position past the domain
    with pytest.raises(pg.EngineError) as e:
        c.permutation_z_rows(rows, bad, beta, gamma, k)
    assert e.value.code == -2 and "first at row 5" in str(e.value)
    w = rows.copy(); w[1, 3] = unreduced
    with pytest.raises(pg.EngineError) as e:
        c.permutation_z_rows(w, sigma, beta, gamma, k)
    assert "first at row 3" in str(e.value)
    with pytest.raises(pg.EngineError):
        c.permutation_z_rows(rows, sigma, beta, gamma, (c.circuit_size() - 1).bit_length() - 1)   # fewer points than rows
    # after the errors the ctx still computes (the row checks use per-call counters, not the composer's sticky ones)
    z, closing = c.permutation_z(beta, gamma)
    assert oracle.to_ints(closing[None]) == [1] and oracle.to_ints(z[:1]) == [1]


def test_emu_permutation_rows_broken_copy_constraint(emu, oracle, golden):
    """A wire value changed at a position in a cycle of length > 1: closing != 1, z equal up to that row and different after it."""
    spec = golden["batch_is_non_zero_maybe_equal"]
    _snap, c = run_engine(spec["program"], lambda: pg.StandardComposer(_cdll=emu), oracle, return_composer=True)
    k = c.domain_log_size()
    beta, gamma = oracle.from_ints(synth_wide(150, 2))
    w, sigma = c.rows(want=("w_val",))["w_val"], c.permutation()
    honest, _ = c.permutation_z_rows(w, sigma, beta, gamma, k)
    r = next(i for i in range(c.circuit_size() // 2, c.circuit_size()) if int(sigma[0, i]) != 4 * i)
    w2 = w.copy(); w2[0, r] = oracle.from_ints([oracle.to_ints(w[0, r:r + 1])[0] + 1])[0]
    z, closing = c.permutation_z_rows(w2, sigma, beta, gamma, k)
    assert oracle.to_ints(closing[None]) != [1]
    assert np.array_equal(z[: r + 1], honest[: r + 1]) and not np.array_equal(z[r + 1], honest[r + 1])
