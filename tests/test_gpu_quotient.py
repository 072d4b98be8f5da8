"""The quotient polynomial on the B200 (k_ntt_coset_pass, k_simple<QuotientBody>, k_simple<QuotientSplitBody>): selectors, PI and t_1 .. t_4
against the golden digests, the big-int model and the C restatement (tests/oracle_quotient/quotient.c, one 4N coset transform), the
headline size (2^16 range_check instances, domain 2^25) with its degree bound and the identity t(x) Z_H(x) = N(x) at a random point,
pokes, and the refusal on a sharded composer.  Run with `pytest -m gpu`."""
import json
import os
import random

import numpy as np
import pytest

import plonk_gadgets_b200 as pg
from oracle import pymodel as pm
from oracle.gen_golden import coeff_digest, run_pymodel_composer
from tests import permutation_model as perm
from tests import quotient_model as qm
from tests.engine_runner import run_engine
from tests.programs import Q, SEED, hx, run_oracle, synth_wide, unhx

pytestmark = pytest.mark.gpu
COEFF = pg.api.FORM_COEFFICIENTS


def gpu_composer(**kw):
    return pg.StandardComposer(device=0, **kw)


def _ints(oracle, a):
    return [oracle.to_ints(col) for col in a]


def test_quotient_golden_gpu(oracle, golden):
    with open(os.path.join(os.path.dirname(__file__), "golden", "quotient.json")) as f:
        gq = json.load(f)
    ch = [oracle.from_ints([unhx(gq[k])])[0] for k in ("alpha", "beta", "gamma", "range_challenge")]
    for name, exp in sorted(gq["programs"].items()):
        _snap, c = run_engine(golden[name]["program"], gpu_composer, oracle, return_composer=True)
        assert coeff_digest(_ints(oracle, c.selector_polynomials())) == exp["selector_evaluations"], name
        assert coeff_digest(_ints(oracle, c.selector_polynomials(form=COEFF))) == exp["selector_coefficients"], name
        assert coeff_digest([oracle.to_ints(c.public_input_polynomial())]) == exp["pi_evaluations"], name
        assert coeff_digest([oracle.to_ints(c.public_input_polynomial(form=COEFF))]) == exp["pi_coefficients"], name
        t = c.quotient(*ch)
        assert coeff_digest(_ints(oracle, t)) == exp["t"], name
        assert (not t[3, -4:].any()) == (not golden[name]["expected"]["unsat"]), name
        c.close()


@pytest.mark.parametrize("name", ["kat_range_check_0_ok", "kat_range_gate_8bits_ok", "batch_mixed_circuit", "batch_is_non_zero_maybe_equal"])
def test_quotient_model_gpu(oracle, golden, name):
    al, be, ga, rh = synth_wide(166, 4)
    ch = [oracle.from_ints([v])[0] for v in (al, be, ga, rh)]
    m = run_pymodel_composer(golden[name]["program"])
    _snap, c = run_engine(golden[name]["program"], gpu_composer, oracle, return_composer=True)
    for log_n in (c.domain_log_size(), c.domain_log_size() + 1):
        assert _ints(oracle, c.selector_polynomials(log_n)) == qm.selector_evaluations(m, log_n)
        assert oracle.to_ints(c.public_input_polynomial(log_n, form=COEFF)) == perm.ifft(qm.public_input_evaluations(m, log_n))
        t, _rem, _num = qm.quotient(m, log_n, al, be, ga, rh)
        assert _ints(oracle, c.quotient(*ch, log_n=log_n)) == t


def _range_check_program(n, stream, bits):
    vals = [v & ((1 << bits) - 1) for v in synth_wide(stream, n)]
    return [dict(op="add_input", values=[hx(v) for v in vals]), dict(op="range_check", min=hx(0), max=hx(1 << bits), witness=0)]


def _mixed_program():
    v = [x & ((1 << 60) - 1) for x in synth_wide(167, 60)]
    return [dict(op="add_input", values=[hx(x) for x in v]),
            dict(op="range_gate", witness=0, num_bits=64),
            dict(op="is_non_zero", var=0, assigned=[hx(x) for x in v]),
            dict(op="constrain_to_constant", a=0, constant=[hx(x * 4 % Q) for x in v], pi=[hx(x * 3 % Q) for x in v]),   # a - 4a + 3a = 0
            dict(op="range_check", min=hx(0), max=hx(1 << 62), witness=0),
            dict(op="constrain_to_constant", a=4, constant=hx(1))]


@pytest.mark.timeout(1500)
def test_quotient_oracle_parity_gpu(oracle):
    """Bit-exact against the C restatement: 2^10 range_check instances (domain 2^18) and a mixed circuit with range gates and PI."""
    ch = [oracle.from_ints([v])[0] for v in synth_wide(168, 4)]
    prog = _range_check_program(1 << 10, 169, 32)
    c = gpu_composer()                                         # (built directly: run_engine's big-int snapshot is slow at this size)
    col = c.add_input(oracle.from_ints([unhx(x) for x in prog[0]["values"]]))
    pg.range_check(c, oracle.from_ints([0]), oracle.from_ints([1 << 32]), col)
    assert c.circuit_size() > 1 << 17 and c.check_circuit_satisfied() == (0, None)
    for p, comp in ((prog, c), (_mixed_program(), None)):
        if comp is None:
            _snap, comp = run_engine(p, gpu_composer, oracle, return_composer=True)
            assert comp.public_input_polynomial().any() and comp.selector_polynomials()[7].any()
        _s, oc = run_oracle(p, return_composer=True)
        t = comp.quotient(*ch)
        assert np.array_equal(t, qm.quot_oracle_t(oracle, oc, comp.domain_log_size(), *ch))
        assert not t[3, -4:].any()


def _numerator_at(c, oracle, torch, k, x, chal):
    """N(x) from the engine's component polynomials (each already checked against the oracles at smaller sizes), evaluated by the C Horner
    at x and x*w, and the big-int numerator formula of tests/quotient_model.py."""
    N = 1 << k
    xw = x * pm.group_gen(k) % Q
    xm, xwm = oracle.from_ints([x])[0], oracle.from_ints([xw])[0]
    buf4 = torch.empty((4, N, 4), dtype=torch.int64, device="cuda")
    buf8 = torch.empty((8, N, 4), dtype=torch.int64, device="cuda")
    buf1 = torch.empty((N, 4), dtype=torch.int64, device="cuda")
    at = lambda t, pt: oracle.to_ints(qm.horner_mont(t.cpu().numpy().view(np.uint64), pt)[None])[0]
    al, be, ga, rh = chal
    bm, gm = oracle.from_ints([be])[0], oracle.from_ints([ga])[0]
    c.wire_polynomials(k, out=buf4); torch.cuda.synchronize()
    wires = [at(buf4[w], xm) for w in range(4)]
    d_next = at(buf4[3], xwm)
    c.permutation_z(bm, gm, k, form=COEFF, out=buf1); torch.cuda.synchronize()
    z, z_next = at(buf1, xm), at(buf1, xwm)
    c.sigma_polynomials(k, form=COEFF, out=buf4); torch.cuda.synchronize()
    sig = [at(buf4[w], xm) for w in range(4)]
    c.selector_polynomials(k, form=COEFF, out=buf8); torch.cuda.synchronize()
    sel = [at(buf8[s], xm) for s in range(8)]
    c.public_input_polynomial(k, form=COEFF, out=buf1); torch.cuda.synchronize()
    pi = at(buf1, xm)
    xn = pow(x, N, Q)
    l1 = (xn - 1) * pow(N * (x - 1), Q - 2, Q) % Q
    return qm.numerator_at(wires + [z] + sig + sel + [pi], x, [0, 0, 0, d_next, z_next], l1, al, be, ga, rh)


def _identity_holds(oracle, t, k, x, n_x):
    xn = pow(x, 1 << k, Q)
    xm = oracle.from_ints([x])[0]
    parts = [oracle.to_ints(qm.horner_mont(t[r], xm)[None])[0] for r in range(4)]
    return sum(p * pow(xn, r, Q) for r, p in enumerate(parts)) * (xn - 1) % Q == n_x


@pytest.mark.timeout(2400)
def test_quotient_headline_gpu(oracle):
    """2^16 range_check instances, 17.8 M rows, domain 2^25: degree bound and identity, honest and after pokes at warp and block
    boundaries (the add_input witnesses of instances 32 and 256, and an accumulator of instance 255)."""
    import torch
    chal = tuple(synth_wide(170, 4))
    ch = [oracle.from_ints([v])[0] for v in chal]
    x = random.Random(171).randrange(Q)
    n = 1 << 16
    for poked in (False, True):
        c = gpu_composer()
        wit = torch.empty((n, 4), dtype=torch.int64, device="cuda"); c.synth(SEED, 2, 2, 64, wit)
        w = c.add_input(wit)
        pg.range_check(c, oracle.from_ints([0]), oracle.from_ints([1 << 64]), w)
        k = c.domain_log_size()
        assert k == 25 and c.circuit_size() > 17_000_000
        if poked:
            for var in (5 + 32, 5 + 256, 5 + n + 653 * 255 + 1 + 256 + 3):
                c.poke_variable(var, oracle.from_ints([12345 + var])[0])
        t_dev = torch.empty((4, 1 << k, 4), dtype=torch.int64, device="cuda")
        c.quotient(*ch, log_n=k, out=t_dev); torch.cuda.synchronize()
        t = t_dev.cpu().numpy().view(np.uint64)
        del t_dev
        assert t[3, -4:].any() == poked
        assert _identity_holds(oracle, t, k, x, _numerator_at(c, oracle, torch, k, x, chal)) != poked
        c.close()
        del t


def _sharded_rank(rank, world, uid, q):
    import torch
    torch.cuda.set_device(rank)
    c = pg.StandardComposer(device=rank)
    c.comm_init(uid, rank, world)
    one = np.array([1, 0, 0, 0], np.uint64)
    codes = []
    for call in (lambda: c.quotient(one, one, one, one), lambda: c.selector_polynomials(), lambda: c.public_input_polynomial()):
        try:
            call(); codes.append(0)
        except pg.EngineError as e:
            codes.append(e.code)
    q.put((rank, codes))
    c.comm_destroy()
    c.close()


@pytest.mark.timeout(600)
def test_quotient_refused_on_sharded_composer_gpu():
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
    assert all(codes == [-6, -6, -6] for _rank, codes in got)
