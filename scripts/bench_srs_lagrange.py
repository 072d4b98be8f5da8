"""Cost of deriving the Lagrange-basis SRS from the monomial powers (pg_srs_lagrange_from_powers, the group inverse FFT of g1fft.cuh)
at domains 2^16, 2^20, 2^22 and 2^25, powers and output on the device; then, at the headline circuit (2^16 range_check instances,
17.8 M rows, domain 2^25), the wire and z commitments through the derived form against the monomial MSMs.  One JSON line.

Per size: a first call (the warm-up; the growth of the ctx's buffer pool over it is the device memory the call needs), then two
calls timed with CUDA events on the engine's stream.  The work is counted from the schedule kept in g1fft.cuh: a butterfly with a
non-trivial twiddle does one scalar multiplication (G1FFT_MUL_FP_MULS = 3341 Fp multiplications) and two additions (2 x 14), a
twiddle-1 butterfly only the two additions, and the 1/n scaling is one more scalar multiplication per point.  A torch.profiler pass
at 2^20 splits the time between the scaling (G1FftIngestBody), the stages (G1FftStageBody) and the normalisation (G1BatchAffineBody).
The card's name and power limit are read in the same run."""
from __future__ import annotations

import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import plonk_gadgets_b200 as pg

SEED = 0x706C6F6E6B5F6732
MUL_FP, ADD_FP = 9 + 13 * 14 + 63 * (4 * 9 + 14), 14          # g1fft.cuh: g1x_mul_fixed; g1.cuh: g1x_add
dev = torch.device("cuda", 0)
stream = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(stream)
R2 = np.array([[0xc999e990f3f29c6d, 0x2b6cedcb87925c23, 0x05d314967254398f, 0x0748d9d99f59ff11]], dtype=np.uint64)


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for _ in range(reps):
        torch.cuda.synchronize(dev); e0.record(stream)
        fn()
        e1.record(stream); torch.cuda.synchronize(dev)
        out.append(e0.elapsed_time(e1))
    return out


def counts(log_n):
    n = 1 << log_n
    nontrivial = (n // 2) * log_n - (n - 1)
    fp = nontrivial * (MUL_FP + 2 * ADD_FP) + (n - 1) * 2 * ADD_FP + n * MUL_FP
    return n, nontrivial, fp


def main():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out = {"op": "pg_srs_lagrange_from_powers: Lagrange-basis SRS from the monomial powers (group inverse FFT over G1), device buffers",
           "gpu": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(dev),
           "fp_muls_per_scalar_mul": MUL_FP, "fp_muls_per_nontrivial_butterfly": MUL_FP + 2 * ADD_FP, "sizes": {}}
    c = pg.StandardComposer(device=0, stream=stream.cuda_stream)
    mk = lambda raw: c.fr_op(0, np.array([raw], dtype=np.uint64), R2)[0]
    tau = mk([0x5eed, 0x7a0, 0x1234, 0])
    for log_n in (16, 20, 22, 25):
        n, nontrivial, fp = counts(log_n)
        mono = torch.empty((n, 12), dtype=torch.int64, device=dev); lag = torch.empty_like(mono)
        c.srs_powers(tau, n, out=mono); torch.cuda.synchronize(dev)
        free0 = torch.cuda.mem_get_info(dev)[0]
        warm = timed(lambda: c.srs_lagrange_from_powers(mono, log_n, out=lag), 1)[0]
        free1 = torch.cuda.mem_get_info(dev)[0]
        runs = timed(lambda: c.srs_lagrange_from_powers(mono, log_n, out=lag), 2)
        best = min(runs) * 1e-3
        out["sizes"][log_n] = {"ms_warmup": warm, "ms_runs": runs, "nontrivial_butterflies": nontrivial, "scaling_muls": n,
                               "scalar_muls_per_s": (nontrivial + n) / best, "fp_muls": fp, "fp_muls_per_s": fp / best,
                               "pool_growth_gib": (free0 - free1) / 2 ** 30}
        print(json.dumps({"log_n": log_n, **out["sizes"][log_n]}), file=sys.stderr, flush=True)
        del mono, lag
    # kernel split at 2^20
    from torch.profiler import ProfilerActivity, profile
    mono = torch.empty((1 << 20, 12), dtype=torch.int64, device=dev); lag = torch.empty_like(mono)
    c.srs_powers(tau, 1 << 20, out=mono); torch.cuda.synchronize(dev)
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        c.srs_lagrange_from_powers(mono, 20, out=lag); torch.cuda.synchronize(dev)
    kern = {}
    for e in p.key_averages():
        tm = (getattr(e, "self_device_time_total", None) or getattr(e, "self_cuda_time_total", 0)) / 1e3
        if tm > 0:
            tag = next((g for g in ("G1FftIngestBody", "G1FftStageBody", "G1BatchAffineBody") if g in e.key), "other")
            kern[tag] = kern.get(tag, 0.0) + tm
    out["kernel_ms_2p20"] = kern
    del mono, lag
    # end to end at the headline circuit: commitments through the derived Lagrange form against the monomial MSMs
    wit = torch.empty((1 << 16, 4), dtype=torch.int64, device=dev); c.synth(SEED, 2, 2, 64, wit)
    w = c.add_input(wit); pg.range_check(c, mk([0, 0, 0, 0])[None], mk([0, 1, 0, 0])[None], w)
    k = c.domain_log_size(); N = 1 << k
    mono = torch.empty((N, 12), dtype=torch.int64, device=dev); lag = torch.empty_like(mono)
    c.srs_powers(tau, N, out=mono)
    derive_ms = timed(lambda: c.srs_lagrange_from_powers(mono, k, out=lag), 1)[0]
    beta, gamma = mk([0x1234567, 0x89abcdef, 0x42, 0]), mk([0x7654321, 0xfedcba98, 0x24, 0])
    zc = torch.empty((N, 4), dtype=torch.int64, device=dev); ze = torch.empty_like(zc)
    c.permutation_z(beta, gamma, k, form=pg.api.FORM_COEFFICIENTS, out=zc); c.permutation_z(beta, gamma, k, out=ze)
    res = {}
    wire_mono_ms = timed(lambda: res.__setitem__("wm", c.commit_wire_polynomials(mono, k)), 2)
    wire_lag_ms = timed(lambda: res.__setitem__("wl", c.commit_wire_evaluations(lag, k)), 2)
    z_mono_ms = timed(lambda: res.__setitem__("zm", c.msm(mono, zc)), 2)
    z_lag_ms = timed(lambda: res.__setitem__("zl", c.msm(lag, ze)), 2)
    assert np.array_equal(res["wm"], res["wl"]) and np.array_equal(res["zm"], res["zl"]) and res["wm"].any(), "commitments differ"
    saved = min(wire_mono_ms) + min(z_mono_ms) - min(wire_lag_ms) - min(z_lag_ms)
    out["headline"] = {"rows": c.circuit_size(), "log_domain": k, "derive_ms": derive_ms,
                       "wire_commitments_monomial_ms": wire_mono_ms, "wire_commitments_lagrange_ms": wire_lag_ms,
                       "z_commitment_monomial_ms": z_mono_ms, "z_commitment_lagrange_ms": z_lag_ms, "commitments_equal": True,
                       "saved_per_proof_ms": saved, "proofs_to_pay_back": derive_ms / saved if saved > 0 else None}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
