"""Prover rounds 4 and 5 on the B200 (k_simple<OpenEvalBody / OpenSumBody / OpenCombineBody>, the Ruffini scan k_fr_ruffini_reduce /
k_fr_ruffini_apply): the golden digests, the big-int model, bit-exact parity with the C restatement (tests/oracle_openings/openings.c)
at domain 2^18 and on a circuit with PI and range gates, pg_fr_op 8 across scan levels, and at the headline size (2^16 range_check
instances, domain 2^25) the evaluations against C Horner, the opening identities at a random point, the quotient identity, and a
pairing-free verifier that knows the SRS secret tau ([f] = f(tau) G), honest, with an altered evaluation and on a poked composer.
Run with `pytest -m gpu`."""
import json
import os
import random

import numpy as np
import pytest

import plonk_gadgets_b200 as pg
from oracle import pymodel as pm
from oracle.gen_golden import coeff_digest, run_pymodel_composer
from tests import opening_model as om
from tests import quotient_model as qm
from tests.engine_runner import run_engine
from tests.programs import Q, SEED, run_oracle, synth_wide, unhx
from tests.test_emu_msm import to_oracle
from tests.test_gpu_quotient import _mixed_program, _range_check_program

pytestmark = pytest.mark.gpu
COEFF = pg.api.FORM_COEFFICIENTS


def gpu_composer(**kw):
    return pg.StandardComposer(device=0, **kw)


def _ev_ints(oracle, ev):
    return {k: oracle.to_ints(ev[k][None])[0] for k in om.EVALUATIONS}


def test_openings_golden_gpu(oracle, golden):
    with open(os.path.join(os.path.dirname(__file__), "golden", "openings.json")) as f:
        go = json.load(f)
    ints = [unhx(x) for x in go["challenges"]]
    ch = [oracle.from_ints([v])[0] for v in ints]
    for name, exp in sorted(go["programs"].items()):
        _snap, c = run_engine(golden[name]["program"], gpu_composer, oracle, return_composer=True)
        ev, out = c.prover_openings(c.quotient(*ch[:4]), *ch)
        evi = _ev_ints(oracle, ev)
        assert coeff_digest([[evi[k] for k in om.EVALUATIONS]]) == exp["evaluations"], name
        assert [coeff_digest([oracle.to_ints(out[i])]) for i in (0, 1, 2)] == [exp["w_z"], exp["w_zw"], exp["r"]], name
        c.close()


@pytest.mark.parametrize("name", ["kat_range_check_0_ok", "kat_range_gate_8bits_ok", "batch_mixed_circuit", "batch_is_non_zero_maybe_equal"])
def test_openings_model_gpu(oracle, golden, name):
    ints = synth_wide(187, 7)
    ch = [oracle.from_ints([v])[0] for v in ints]
    m = run_pymodel_composer(golden[name]["program"])
    _snap, c = run_engine(golden[name]["program"], gpu_composer, oracle, return_composer=True)
    for log_n in (c.domain_log_size(), c.domain_log_size() + 1):
        ev_m, r, wz, wzw, _rems, t, _pi = om.openings(m, log_n, *ints)
        ev, out = c.prover_openings(np.stack([oracle.from_ints(col) for col in t]), *ch, log_n=log_n)
        assert _ev_ints(oracle, ev) == ev_m
        assert [oracle.to_ints(col) for col in out] == [wz, wzw, r]
    c.close()


def _component_vectors(c, k, ch):
    """(17, N, 4): the engine's wire, z, sigma and selector coefficient vectors (each checked against the oracles by earlier tests)."""
    return np.concatenate([c.wire_polynomials(k), c.permutation_z(ch[1], ch[2], k, form=COEFF)[0][None],
                           c.sigma_polynomials(k, form=COEFF), c.selector_polynomials(k, form=COEFF)])


@pytest.mark.timeout(1500)
def test_openings_oracle_parity_gpu(oracle):
    """Bit-exact against the C restatement: 2^10 range_check instances (domain 2^18) and a mixed circuit with range gates and PI."""
    ch = [oracle.from_ints([v])[0] for v in synth_wide(188, 7)]
    prog = _range_check_program(1 << 10, 189, 32)
    c = gpu_composer()
    col = c.add_input(oracle.from_ints([unhx(x) for x in prog[0]["values"]]))
    pg.range_check(c, oracle.from_ints([0]), oracle.from_ints([1 << 32]), col)
    assert c.circuit_size() > 1 << 17
    for p, comp in ((prog, c), (_mixed_program(), None)):
        if comp is None:
            _snap, comp = run_engine(p, gpu_composer, oracle, return_composer=True)
        k = comp.domain_log_size()
        _s, oc = run_oracle(p, return_composer=True)
        t = qm.quot_oracle_t(oracle, oc, k, *ch[:4])
        ev, out = comp.prover_openings(t, *ch)
        ev_c, out_c = om.open_oracle(oracle, _component_vectors(comp, k, ch), t, k, ch)
        assert np.array_equal(np.stack([ev[name] for name in om.EVALUATIONS]), ev_c)
        assert np.array_equal(out, out_c)
        comp.close()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("n", [1, 2, 1023, 1024, 1025, (1 << 20) + 1, 1 << 22])
def test_fr_op_ruffini_gpu(oracle, n):
    """pg_fr_op 8 (one, two and three scan levels; in place on its staged copy) against the C restatement's Polynomial::ruffini and
    Polynomial::evaluate, for p in {0, 1, -1, w, random}."""
    c = gpu_composer()
    a = np.random.default_rng(190).integers(0, 1 << 64, size=(n, 4), dtype=np.uint64)
    a[:, 3] %= np.uint64(0x73EDA753299D7D48)                   # below q: any reduced value is a Montgomery scalar
    for p in (0, 1, Q - 1, pm.group_gen(22), synth_wide(191, 1)[0]):
        pm_ = oracle.from_ints([p])
        got = c.fr_op(8, a, pm_)
        assert np.array_equal(got[:n - 1], om.c_ruffini(a, pm_[0])[:n - 1]), p
        assert np.array_equal(got[n - 1], om.c_evaluate(a, pm_[0])), p
    c.close()


# ------------------------------------------------------------------------------------------------ headline size, verifier
def _headline(oracle, torch, poked):
    n = 1 << 16
    c = gpu_composer()
    wit = torch.empty((n, 4), dtype=torch.int64, device="cuda"); c.synth(SEED, 2, 2, 64, wit)
    w = c.add_input(wit)
    pg.range_check(c, oracle.from_ints([0]), oracle.from_ints([1 << 64]), w)
    if poked:                                                  # the pokes of test_quotient_headline_gpu
        for var in (5 + 32, 5 + 256, 5 + n + 653 * 255 + 1 + 256 + 3):
            c.poke_variable(var, oracle.from_ints([12345 + var])[0])
    return c


def _g1(oracle, pt):
    return oracle.g1_to_ints(to_oracle(pt))[0]


def _verify(ev, com, ints, tau, k):
    """The two KZG opening equations with the SRS secret known: (tau - p) [W_p] == [agg_p] - agg_p(p) G, [agg] formed from the
    commitments and the evaluations the way the verifier forms it (its [r] from the commitments of the selectors, z and sigma_4)."""
    al, be, ga, rh, z, v, vs = ints
    n = 1 << k
    zw = z * pm.group_gen(k) % Q
    G = pm.G1_GENERATOR

    def comb(pairs):
        acc = None
        for s, p in pairs:
            acc = pm.g1_add(acc, pm.g1_mul(s % Q, p))
        return acc
    wts = om.linearisation_weights(ev, al, be, ga, rh, z, n)
    r_com = comb([(wgt, com["poly", i]) for i, wgt in wts.items()])
    zn = pow(z, n, Q)
    agg_z = comb([(pow(zn, r, Q), com["t", r]) for r in range(4)] + [(v, r_com)] + [(pow(v, 2 + i, Q), com["poly", om.W + i]) for i in range(4)]
                 + [(pow(v, 6 + i, Q), com["poly", om.S + i]) for i in range(3)])
    agg_zw = comb([(1, com["poly", om.Z]), (vs, com["poly", om.W]), (vs * vs, com["poly", om.W + 1]), (vs ** 3, com["poly", om.W + 3])])
    bar_z, bar_zw = om.aggregate_values(ev, z, n, v, vs)
    ok_z = pm.g1_mul((tau - z) % Q, com["W", 0]) == pm.g1_add(agg_z, pm.g1_neg(pm.g1_mul(bar_z, G)))
    ok_zw = pm.g1_mul((tau - zw) % Q, com["W", 1]) == pm.g1_add(agg_zw, pm.g1_neg(pm.g1_mul(bar_zw, G)))
    return ok_z, ok_zw


@pytest.mark.timeout(3000)
def test_openings_headline_gpu(oracle):
    """2^16 range_check instances, 17.8 M rows, domain 2^25.  Honest: the evaluations equal C Horner of the engine's component vectors,
    the opening identities hold at a random x, the quotient identity holds, and the pairing-free verifier accepts both openings; with
    a_eval (a_next_eval) altered it rejects the opening at z (z*w).  Poked: the openings still verify, the quotient identity fails."""
    import torch
    ints = tuple(synth_wide(192, 7))
    ch = [oracle.from_ints([v])[0] for v in ints]
    x, tau = random.Random(193).randrange(Q), random.Random(194).randrange(Q)
    k = 25
    N = 1 << k
    z, zw = ints[4], ints[4] * pm.group_gen(k) % Q
    pts = [oracle.from_ints([p])[0] for p in (z, zw, x)]
    at = lambda vec: [oracle.to_ints(om.c_evaluate(vec, p)[None])[0] for p in pts]          # (at z, at z*w, at x)
    for poked in (False, True):
        c = _headline(oracle, torch, poked)
        assert c.domain_log_size() == k and c.circuit_size() > 17_000_000
        mono = torch.empty((N, 12), dtype=torch.int64, device="cuda")
        c.srs_powers(oracle.from_ints([tau])[0], N, out=mono)
        t_dev = torch.empty((4, N, 4), dtype=torch.int64, device="cuda")
        out_dev = torch.empty((3, N, 4), dtype=torch.int64, device="cuda")
        c.quotient(*ch[:4], log_n=k, out=t_dev)
        ev, _ = c.prover_openings(t_dev, *ch, log_n=k, out=out_dev); torch.cuda.synchronize()
        evi = _ev_ints(oracle, ev)
        com, vals = {}, {}
        for key, vec in ([(("t", r), t_dev[r]) for r in range(4)] + [(("W", i), out_dev[i]) for i in range(2)] + [(("r", 0), out_dev[2])]):
            com[key] = _g1(oracle, c.msm(mono, vec))
            vals[key] = at(vec.cpu().numpy().view(np.uint64))
        del t_dev
        buf = torch.empty((8, N, 4), dtype=torch.int64, device="cuda")
        fill = [(lambda: c.wire_polynomials(k, out=buf[:4]), range(0, 4)), (lambda: c.permutation_z(ch[1], ch[2], k, form=COEFF, out=buf[0]), range(4, 5)),
                (lambda: c.sigma_polynomials(k, form=COEFF, out=buf[:4]), range(5, 9)), (lambda: c.selector_polynomials(k, form=COEFF, out=buf), range(9, 17))]
        for make, idx in fill:
            make(); torch.cuda.synchronize()
            for j, i in enumerate(idx):
                com["poly", i] = _g1(oracle, c.msm(mono, buf[j]))
                vals["poly", i] = at(buf[j].cpu().numpy().view(np.uint64))
        pi_z = om.horner(oracle.to_ints(c.public_input_polynomial(k, form=COEFF)), z)
        del buf, mono
        c.close()
        # the evaluations against C Horner of the engine's vectors
        P = lambda i, j=0: vals["poly", i][j]
        zn = pow(z, N, Q)
        exp = dict(a_eval=P(0), b_eval=P(1), c_eval=P(2), d_eval=P(3), a_next_eval=P(0, 1), b_next_eval=P(1, 1), d_next_eval=P(3, 1),
                   q_arith_eval=P(om.QARITH), q_c_eval=P(om.QC), q_l_eval=P(om.QL), q_r_eval=P(om.QR), left_sigma_eval=P(5), right_sigma_eval=P(6),
                   out_sigma_eval=P(7), lin_poly_eval=vals["r", 0][0], perm_eval=P(4, 1),
                   quot_eval=sum(pow(zn, r, Q) * vals["t", r][0] for r in range(4)) % Q)
        assert evi == exp
        # r by its formula from the vectors' values at x, then the opening identities at x
        wts = om.linearisation_weights(evi, *ints[:4], z, N)
        assert vals["r", 0][2] == sum(wgt * P(i, 2) for i, wgt in wts.items()) % Q
        v, vs = ints[5], ints[6]
        quot_x = sum(pow(zn, r, Q) * vals["t", r][2] for r in range(4))
        agg_x = sum(pow(v, j, Q) * y for j, y in enumerate([quot_x, vals["r", 0][2], P(0, 2), P(1, 2), P(2, 2), P(3, 2), P(5, 2), P(6, 2), P(7, 2)])) % Q
        agg_xw = sum(pow(vs, j, Q) * y for j, y in enumerate([P(4, 2), P(0, 2), P(1, 2), P(3, 2)])) % Q
        bar_z, bar_zw = om.aggregate_values(evi, z, N, v, vs)
        assert (x - z) * vals["W", 0][2] % Q == (agg_x - bar_z) % Q
        assert (x - zw) * vals["W", 1][2] % Q == (agg_xw - bar_zw) % Q
        assert om.quotient_identity_holds(evi, pi_z, ints[0], ints[1], ints[2], z, N) != poked
        assert _verify(evi, com, ints, tau, k) == (True, True)
        if not poked:
            assert _verify(dict(evi, a_eval=(evi["a_eval"] + 1) % Q), com, ints, tau, k)[0] is False
            assert _verify(dict(evi, a_next_eval=(evi["a_next_eval"] + 1) % Q), com, ints, tau, k)[1] is False


def _sharded_rank(rank, world, uid, q):
    import torch
    torch.cuda.set_device(rank)
    c = pg.StandardComposer(device=rank)
    c.comm_init(uid, rank, world)
    one = np.array([1, 0, 0, 0], np.uint64)
    t = np.zeros((4, 1 << c.domain_log_size(), 4), np.uint64)
    try:
        c.prover_openings(t, one, one, one, one, np.array([5, 0, 0, 0], np.uint64), one, one); code = 0
    except pg.EngineError as e:
        code = e.code
    q.put((rank, code))
    c.comm_destroy()
    c.close()


@pytest.mark.timeout(600)
def test_openings_refused_on_sharded_composer_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs: the refusal is checked on a communicator of two ranks")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    uid = pg.comm_unique_id()
    procs = [ctx.Process(target=_sharded_rank, args=(r, 2, uid, q)) for r in range(2)]
    for p in procs: p.start()
    got = [q.get(timeout=300) for _ in range(2)]
    for p in procs: p.join(timeout=120)
    assert all(p.exitcode == 0 for p in procs)
    assert all(code == -6 for _rank, code in got)
