"""pg_srs_lagrange_from_powers on the B200 (k_simple<G1FftIngestBody / G1FftStageBody / G1BatchAffineBody>): bit-exact parity with
the C restatement tests/oracle_lagrange/group_fft.c at 2^12, equality with pg_srs_lagrange up to 2^20 (host and device buffers,
tau = 0 included), with fixed_base_mul(ifft(k)) at 2^20 -- the late stages, where the lanes of a warp hold different twiddles --
and at the headline domain 2^25 with pg_srs_lagrange and with the monomial wire commitments of 2^16 range_check instances.
Run with `pytest -m gpu`."""
import random

import numpy as np
import pytest

import plonk_gadgets_b200 as pg
from tests import lagrange_model as lm
from tests.programs import Q, SEED
from tests.test_emu_msm import to_oracle

pytestmark = pytest.mark.gpu
TAU = 0x3a7c5e1f9b2d4c6e8a0f1e3d5c7b9a8f6e4d2c0b1a3f5e7d9c8b6a4f2e0d1c3b % Q


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch


def gpu_composer():
    return pg.StandardComposer(device=0)


def test_from_powers_matches_c_restatement_gpu(oracle, torch_cuda):
    """2^12 random points (infinity and an opposite pair among them) against the textbook serial inverse FFT in C."""
    log_n, n = 12, 1 << 12
    c = gpu_composer()
    rnd = random.Random(12)
    ks = [rnd.randrange(Q) for _ in range(n)]
    ks[7] = 0; ks[100] = 0; ks[200] = Q - ks[201]
    pts = c.g1_fixed_base_mul(oracle.from_ints(ks))
    got = c.srs_lagrange_from_powers(pts, log_n)
    assert np.array_equal(to_oracle(got), lm.group_ifft(to_oracle(pts), log_n))


@pytest.mark.parametrize("log_n", [1, 5, 11, 17, 20])
def test_from_powers_equals_srs_lagrange_gpu(oracle, torch_cuda, log_n):
    torch = torch_cuda
    n = 1 << log_n
    c = gpu_composer()
    tau = oracle.from_ints([TAU])[0]
    want = c.srs_lagrange(tau, log_n)
    powers = c.srs_powers(tau, n + 3)                                    # three powers more than the domain: not read
    assert np.array_equal(c.srs_lagrange_from_powers(powers, log_n), want)
    mono = torch.empty((n, 12), dtype=torch.int64, device="cuda"); lag = torch.empty_like(mono); torch.cuda.synchronize()
    c.srs_powers(tau, n, out=mono)
    c.srs_lagrange_from_powers(mono, log_n, out=lag); torch.cuda.synchronize()
    assert np.array_equal(lag.cpu().numpy().view(np.uint64), want)
    assert np.array_equal(c.srs_lagrange_from_powers(mono, log_n), want)         # device powers, host output


def test_from_powers_tau_zero_gpu(oracle, torch_cuda):
    """tau = 0: powers G, O, O, ...; every intermediate value is G or O, every output G/n."""
    c = gpu_composer()
    zero = oracle.from_ints([0])[0]
    got = c.srs_lagrange_from_powers(c.srs_powers(zero, 1 << 11), 11)
    assert np.array_equal(got, c.srs_lagrange(zero, 11))
    assert (got == got[0]).all() and got[0].any()


@pytest.mark.timeout(1200)
def test_from_powers_random_points_2p20_gpu(oracle, torch_cuda):
    """P_j = k_j G for random k: the output is (ifft k)_i G (pg_fft inverse, pg_g1_fixed_base_mul)."""
    torch = torch_cuda
    log_n, n = 20, 1 << 20
    c = gpu_composer()
    ks = torch.empty((n, 4), dtype=torch.int64, device="cuda"); c.synth(SEED, 9, 0, 0, ks); torch.cuda.synchronize()
    k_host = ks.cpu().numpy().view(np.uint64).copy()
    k_host[3] = 0                                                                  # a point at infinity
    pts = c.g1_fixed_base_mul(k_host)
    want = c.g1_fixed_base_mul(c.fft(k_host, inverse=True))
    assert np.array_equal(c.srs_lagrange_from_powers(pts, log_n), want)


@pytest.mark.timeout(3000)
def test_from_powers_headline_gpu(oracle, torch_cuda):
    """Domain 2^25: the derived form equals pg_srs_lagrange(tau), and the wire commitments of 2^16 range_check instances (17.8 M
    rows) taken from the values against it equal the monomial ones."""
    torch = torch_cuda
    k, N = 25, 1 << 25
    c = gpu_composer()
    wit = torch.empty((1 << 16, 4), dtype=torch.int64, device="cuda"); c.synth(SEED, 2, 2, 64, wit)
    w = c.add_input(wit)
    pg.range_check(c, oracle.from_ints([0]), oracle.from_ints([1 << 64]), w)
    assert c.domain_log_size() == k and c.circuit_size() > 17_000_000
    tau = oracle.from_ints([TAU])[0]
    mono = torch.empty((N, 12), dtype=torch.int64, device="cuda"); lag = torch.empty_like(mono); ref = torch.empty_like(mono)
    torch.cuda.synchronize()
    c.srs_powers(tau, N, out=mono)
    c.srs_lagrange_from_powers(mono, k, out=lag)
    c.srs_lagrange(tau, k, out=ref); torch.cuda.synchronize()
    assert torch.equal(lag, ref)
    del ref
    a, b = c.commit_wire_evaluations(lag), c.commit_wire_polynomials(mono)
    assert np.array_equal(a, b) and a.any()
