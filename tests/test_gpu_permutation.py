"""The permutation argument on the B200 (k_simple<PermSigmaBody>, k_batch_inv<PermRatioHook>, k_fr_scan_reduce / k_fr_scan_apply): sigma and
z(X) against the golden digests, the big-int model and the C restatement (tests/oracle_perm/permutation.c), the scan at awkward sizes, the
headline size (2^16 range_check instances, domain 2^25), soundness through caller-supplied rows, pokes, commitments, and the
refusal on a sharded composer.  Run with `pytest -m gpu`."""
import json
import os
import random

import numpy as np
import pytest

import plonk_gadgets_b200 as pg
from oracle import pymodel as pm
from oracle.gen_golden import coeff_digest, run_pymodel_composer
from tests import permutation_model as perm
from tests.engine_runner import run_engine
from tests.programs import Q, SEED, hx, run_oracle, synth_wide, unhx

pytestmark = pytest.mark.gpu
COEFF = pg.api.FORM_COEFFICIENTS


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch


def gpu_composer(**kw):
    return pg.StandardComposer(device=0, **kw)


def _u64(t):
    return t.cpu().numpy().view(np.uint64)


def test_permutation_golden_gpu(oracle, golden):
    with open(os.path.join(os.path.dirname(__file__), "golden", "permutation.json")) as f:
        gp = json.load(f)
    beta, gamma = (oracle.from_ints([unhx(gp[k])]) for k in ("beta", "gamma"))
    for name, exp in sorted(gp["programs"].items()):
        _snap, c = run_engine(golden[name]["program"], gpu_composer, oracle, return_composer=True)
        ints = lambda a: [oracle.to_ints(col) for col in a]
        assert coeff_digest(ints(c.sigma_polynomials())) == exp["sigma_evaluations"], name
        assert coeff_digest(ints(c.sigma_polynomials(form=COEFF))) == exp["sigma_coefficients"], name
        z, closing = c.permutation_z(beta, gamma)
        zc, _ = c.permutation_z(beta, gamma, form=COEFF)
        assert oracle.to_ints(closing[None]) == [1], name
        assert coeff_digest([oracle.to_ints(z)]) == exp["z_evaluations"] and coeff_digest([oracle.to_ints(zc)]) == exp["z_coefficients"], name
        c.close()


def test_permutation_model_gpu(oracle, golden):
    name = "batch_is_non_zero_maybe_equal"
    beta, gamma = synth_wide(160, 2)
    m = run_pymodel_composer(golden[name]["program"])
    _snap, c = run_engine(golden[name]["program"], gpu_composer, oracle, return_composer=True)
    log_n = c.domain_log_size() + 1
    assert [oracle.to_ints(col) for col in c.sigma_polynomials(log_n)] == perm.sigma_evaluations(m, log_n)
    z, closing = perm.permutation_z(m, log_n, beta, gamma)
    got, got_closing = c.permutation_z(oracle.from_ints([beta]), oracle.from_ints([gamma]), log_n)
    assert oracle.to_ints(got) == z and oracle.to_ints(got_closing[None]) == [closing] == [1]


SCAN_TILE = 1024


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, SCAN_TILE - 1, SCAN_TILE, SCAN_TILE + 1, SCAN_TILE * (SCAN_TILE + 1), (1 << 20) + 3])
def test_scan_edge_sizes_gpu(oracle, n):
    """fr_op 7 (the grand-product scan) against the serial big-int product; SCAN_TILE * (SCAN_TILE + 1) and 2^20 + 3 have more tile
    totals than one block scans, so they go through the second level."""
    rng = random.Random(n)
    vals = [rng.randrange(1, Q) for _ in range(n)]
    if n > 40:
        vals[n // 3] = 1
    c = gpu_composer()
    got = oracle.to_ints(c.fr_op(7, oracle.from_ints(vals)))
    acc, exp = 1, []
    for v in vals:
        exp.append(acc)
        acc = acc * v % Q
    assert got == exp


def _range_check_program(n, stream):
    vals = [v & ((1 << 64) - 1) for v in synth_wide(stream, n)]
    return [dict(op="add_input", values=[hx(v) for v in vals]), dict(op="range_check", min=hx(0), max=hx(1 << 64), witness=0)]


def _mixed_program():
    v = [x & ((1 << 60) - 1) for x in synth_wide(170, 60)]
    return [dict(op="add_input", values=[hx(x) for x in v]),
            dict(op="range_gate", witness=0, num_bits=64),
            dict(op="is_non_zero", var=0, assigned=[hx(x) for x in v]),
            dict(op="constrain_to_constant", a=0, constant=[hx(x) for x in v]),
            dict(op="range_check", min=hx(0), max=hx(1 << 62), witness=0),
            dict(op="constrain_to_constant", a=4, constant=hx(1))]


def _oracle_parity(oracle, program, c, beta, gamma):
    _s, oc = run_oracle(program, return_composer=True)
    k = c.domain_log_size()
    osig, oz, oclosing = perm.perm_oracle_z(oracle, oc, k, beta, gamma)
    assert oracle.to_ints(oclosing[None]) == [1]
    z, closing = c.permutation_z(beta, gamma)
    assert np.array_equal(z, oz) and np.array_equal(closing, oclosing)
    zc, _ = c.permutation_z(beta, gamma, form=COEFF)
    assert np.array_equal(zc, oracle.fft(oz, inverse=True))
    assert np.array_equal(c.sigma_polynomials(), osig)
    sc = c.sigma_polynomials(form=COEFF)
    assert all(np.array_equal(sc[w], oracle.fft(osig[w], inverse=True)) for w in range(4))


@pytest.mark.timeout(1200)
def test_permutation_oracle_parity_gpu(oracle):
    beta, gamma = oracle.from_ints(synth_wide(171, 2))
    prog = _range_check_program(1 << 10, 172)
    c = gpu_composer()                                         # (built directly: run_engine's big-int snapshot of 2^18 rows is slow)
    col = c.add_input(oracle.from_ints([unhx(x) for x in prog[0]["values"]]))
    pg.range_check(c, oracle.from_ints([0]), oracle.from_ints([1 << 64]), col)
    assert c.circuit_size() > 1 << 17 and c.check_circuit_satisfied() == (0, None)
    _oracle_parity(oracle, prog, c, beta, gamma)
    prog = _mixed_program()
    _snap, c = run_engine(prog, gpu_composer, oracle, return_composer=True)
    _oracle_parity(oracle, prog, c, beta, gamma)


def test_permutation_is_non_zero_layouts_gpu(oracle):
    """is_non_zero through pg_is_non_zero_batch_flags in both layouts: without a zero value both append what the reference appends."""
    beta, gamma = oracle.from_ints(synth_wide(173, 2))
    v = synth_wide(174, 500)
    prog = [dict(op="add_input", values=[hx(x) for x in v]), dict(op="is_non_zero", var=0, assigned=[hx(x) for x in v])]
    for layout in (pg.NZ_UNIFORM, pg.NZ_REFERENCE):
        c = gpu_composer()
        col = c.add_input(oracle.from_ints(v))
        flags = pg.is_non_zero_flags(c, col, oracle.from_ints(v), layout=layout)
        assert not flags.any()
        _oracle_parity(oracle, prog, c, beta, gamma)


@pytest.mark.timeout(1800)
def test_permutation_headline_gpu(oracle, torch_cuda):
    """2^16 range_check instances, 17.8 M rows, domain 2^25."""
    torch = torch_cuda
    c = gpu_composer()
    n = 1 << 16
    wit = torch.empty((n, 4), dtype=torch.int64, device="cuda"); c.synth(SEED, 2, 2, 64, wit)
    w = c.add_input(wit)
    pg.range_check(c, oracle.from_ints([0]), oracle.from_ints([1 << 64]), w)
    k = c.domain_log_size(); rows = c.circuit_size()
    assert k == 25 and rows > 17_000_000
    bi, gi = synth_wide(175, 2)
    beta, gamma = oracle.from_ints([bi]), oracle.from_ints([gi])
    N = 1 << k
    z = torch.empty((N, 4), dtype=torch.int64, device="cuda")
    _, closing = c.permutation_z(beta, gamma, out=z)
    assert oracle.to_ints(closing[None]) == [1]
    zh = _u64(z)
    assert oracle.to_ints(zh[:1]) == [1]
    # the rows path on the materialised rows and the map gives the same z
    wv = torch.empty((4, rows, 4), dtype=torch.int64, device="cuda")
    c._ok(c._L.pg_materialize_rows(c._ctx, 0, rows, None, pg.api.C.c_void_p(wv.data_ptr()), None, None, 1), "pg_materialize_rows")
    sig = torch.empty((4, rows), dtype=torch.int64, device="cuda")
    c._ok(c._L.pg_permutation(c._ctx, 0, rows, pg.api.C.c_void_p(sig.data_ptr()), 1), "pg_permutation")
    z2 = torch.empty_like(z)
    _, closing2 = c.permutation_z_rows(wv, sig, beta, gamma, k, out=z2)
    assert torch.equal(z, z2) and np.array_equal(closing, closing2)
    # the recurrence z_{i+1} * den_i = z_i * num_i in big ints at seeded rows, the last row and the first padding row
    rng = random.Random(176)
    picks = sorted(set(rng.randrange(N - 1) for _ in range(4096)) | {rows - 1, rows})
    wvh, sigh = _u64(wv), _u64(sig)
    g = pm.group_gen(k)
    zi = oracle.to_ints(zh[picks]); zn = oracle.to_ints(zh[[i + 1 for i in picks]])
    in_rows = [i for i in picks if i < rows]
    vals = {w_: dict(zip(in_rows, oracle.to_ints(wvh[w_, in_rows]))) for w_ in range(4)}
    for t, i in enumerate(picks):
        num = den = 1
        for w_ in range(4):
            v = vals[w_].get(i, 0)
            s = int(sigh[w_, i]) if i < rows else 4 * i + w_
            num = num * (v + bi * perm.PERM_K[w_] * pow(g, i, Q) + gi) % Q
            den = den * (v + bi * perm.PERM_K[s & 3] * pow(g, s >> 2, Q) + gi) % Q
        assert zn[t] * den % Q == zi[t] * num % Q, i
    del wv, sig, z2
    # coefficient form equals pg_fft's inverse transform of the evaluations
    zc = torch.empty_like(z)
    c.permutation_z(beta, gamma, form=COEFF, out=zc)
    c.fft(z, inverse=True)
    torch.cuda.synchronize()
    assert torch.equal(z, zc)


def test_permutation_soundness_gpu(oracle):
    """A changed wire value at a position in a cycle of length > 1: closing != 1; z equals the honest z up to and including that row."""
    prog = _range_check_program(200, 177)
    _snap, c = run_engine(prog, gpu_composer, oracle, return_composer=True)
    k = c.domain_log_size()
    beta, gamma = oracle.from_ints(synth_wide(178, 2))
    w, sigma = c.rows(want=("w_val",))["w_val"], c.permutation()
    honest, hc = c.permutation_z_rows(w, sigma, beta, gamma, k)
    assert oracle.to_ints(hc[None]) == [1]
    for r in (c.circuit_size() // 3, c.circuit_size() - 2):
        r = next(i for i in range(r, c.circuit_size()) if int(sigma[1, i]) != 4 * i + 1)
        w2 = w.copy(); w2[1, r] = oracle.from_ints([oracle.to_ints(w[1, r:r + 1])[0] + 5])[0]
        z, closing = c.permutation_z_rows(w2, sigma, beta, gamma, k)
        assert oracle.to_ints(closing[None]) != [1]
        assert np.array_equal(z[: r + 1], honest[: r + 1]) and not np.array_equal(z[r + 1], honest[r + 1]), r


def test_permutation_after_poke_gpu(oracle, golden):
    name = "kat_range_check_0_ok"
    _snap, c = run_engine(golden[name]["program"], gpu_composer, oracle, return_composer=True)
    m = run_pymodel_composer(golden[name]["program"])
    k = c.domain_log_size()
    bi, gi = synth_wide(179, 2)
    beta, gamma = oracle.from_ints([bi]), oracle.from_ints([gi])
    before, _ = c.permutation_z(beta, gamma)
    var = 5                                                    # the witness of add_input: used on several rows
    c.poke_variable(var, oracle.from_ints([123456789])[0])
    m.variables[var] = 123456789
    z, closing = c.permutation_z(beta, gamma)
    mz, mclosing = perm.permutation_z(m, k, bi, gi)
    assert oracle.to_ints(z) == mz and oracle.to_ints(closing[None]) == [mclosing] == [1]
    assert not np.array_equal(z, before)


@pytest.mark.timeout(1200)
def test_permutation_commitment_gpu(oracle, torch_cuda):
    """Domain 2^20: msm(lagrange, z evaluations) == msm(powers_of_g, z coefficients)."""
    torch = torch_cuda
    c = gpu_composer()
    n = 2500
    wit = torch.empty((n, 4), dtype=torch.int64, device="cuda"); c.synth(SEED, 3, 2, 64, wit)
    w = c.add_input(wit)
    pg.range_check(c, oracle.from_ints([0]), oracle.from_ints([1 << 64]), w)
    k = c.domain_log_size(); assert k == 20
    beta, gamma = oracle.from_ints(synth_wide(180, 2))
    ze = torch.empty((1 << k, 4), dtype=torch.int64, device="cuda"); zc = torch.empty_like(ze)
    c.permutation_z(beta, gamma, out=ze); c.permutation_z(beta, gamma, form=COEFF, out=zc)
    tau = oracle.from_ints([0x2b3c4d5e6f708192a3b4c5d6e7f8091a2b3c4d5e6f708192a3b4c5d6e7f80 % Q])[0]
    mono = torch.empty((1 << k, 12), dtype=torch.int64, device="cuda"); lag = torch.empty_like(mono); torch.cuda.synchronize()
    c.srs_powers(tau, 1 << k, out=mono); c.srs_lagrange(tau, k, out=lag)
    a, b = c.msm(lag, ze), c.msm(mono, zc)
    assert np.array_equal(a, b) and a.any()


def _sharded_rank(rank, world, uid, q):
    import torch
    torch.cuda.set_device(rank)
    c = pg.StandardComposer(device=rank)
    c.comm_init(uid, rank, world)
    codes = []
    for call in (lambda: c.permutation_z(np.zeros(4, np.uint64), np.zeros(4, np.uint64)), lambda: c.sigma_polynomials()):
        try:
            call(); codes.append(0)
        except pg.EngineError as e:
            codes.append(e.code)
    q.put((rank, codes))
    c.comm_destroy()
    c.close()


@pytest.mark.timeout(600)
def test_permutation_refused_on_sharded_composer_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    uid = pg.comm_unique_id()
    procs = [ctx.Process(target=_sharded_rank, args=(r, 2, uid, q)) for r in range(2)]
    for p in procs: p.start()
    got = [q.get(timeout=300) for _ in range(2)]
    for p in procs: p.join(timeout=120)
    assert all(p.exitcode == 0 for p in procs)
    assert all(codes == [-6, -6] for _rank, codes in got)
