"""Throughput of the permutation argument (pg_sigma_polynomials, pg_permutation_z) on the circuit of `bench_msm.py --round1`:
2^16 range_check instances, 17.8 M rows, domain 2^25.  CUDA events on the engine's stream after a warm-up; one JSON line.

For the z-evaluation kernels it derives, from counts kept here and times measured in the same run:
  - Fr multiplications per row over the time, against pg_microbench mode 6 (Montgomery multiplications per second on all SMs);
  - the scan's bytes over its time, against a device-to-device copy of the same size.
The kernel times of the parts (k_batch_inv<PermRatioHook>, k_fr_scan_*, k_simple<PermSigmaBody>) come from a torch.profiler pass over one
call of each, after the timed passes; `--trace-dir DIR` also writes its kernel table there."""
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
COEFF = pg.api.FORM_COEFFICIENTS
dev = torch.device("cuda", 0)
stream = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(stream)
R2 = np.array([[0xc999e990f3f29c6d, 0x2b6cedcb87925c23, 0x05d314967254398f, 0x0748d9d99f59ff11]], dtype=np.uint64)

# Fr multiplications per row of the z-evaluation kernels (bodies.cuh PermRatioHook, kernels.cuh k_batch_inv, scan.cuh):
#   num: 4 x (beta*k_w * w^i) + 3 products; den: 4 x (beta*k_w' * w^r') + 3 products          -> 14
#   batch inversion: 1 running product + 2 on the way back; post: num * den^-1                 -> 4
#   scan, per thread of 4 elements: k_fr_scan_reduce 4 + 5 (warp butterfly); k_fr_scan_apply 3 (the thread's product) + ~4 (shfl_up
#   scan, lanes below the distance idle) + 2 (warp and tile prefixes) + 4 (the walk) -> 22 / 4 = 5.5 per element
MULS_RATIO, MULS_SCAN = 18, 5.5


def timed(fn, reps=3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()                                                                # warm-up
    torch.cuda.synchronize(dev); e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream); torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def main():
    trace_dir = sys.argv[sys.argv.index("--trace-dir") + 1] if "--trace-dir" in sys.argv else None
    c = pg.StandardComposer(device=0, stream=stream.cuda_stream)
    mk = lambda raw: c.fr_op(0, np.array([raw], dtype=np.uint64), R2)[0]
    beta, gamma = mk([0x1234567, 0x89abcdef, 0x42, 0]), mk([0x7654321, 0xfedcba98, 0x24, 0])
    tau = mk([0x2468ace, 0x13579bdf, 0x77, 0])
    mn, mx = mk([0, 0, 0, 0]), mk([0, 1, 0, 0])
    n = 1 << 16
    wit = torch.empty((n, 4), dtype=torch.int64, device=dev); c.synth(SEED, 2, 2, 64, wit)
    w = c.add_input(wit); pg.range_check(c, mn[None], mx[None], w)
    assert c.check_circuit_satisfied() == (0, None)
    k = c.domain_log_size(); N = 1 << k; rows = c.circuit_size()
    sig = torch.empty((4, N, 4), dtype=torch.int64, device=dev)
    z = torch.empty((N, 4), dtype=torch.int64, device=dev); zc = torch.empty_like(z)
    polys = torch.empty((4, N, 4), dtype=torch.int64, device=dev)
    calls = {
        "sigma_evaluations_ms": lambda: c.sigma_polynomials(k, out=sig),
        "sigma_coefficients_ms": lambda: c.sigma_polynomials(k, form=COEFF, out=sig),
        "z_evaluations_ms": lambda: c.permutation_z(beta, gamma, k, out=z),
        "z_coefficients_ms": lambda: c.permutation_z(beta, gamma, k, form=COEFF, out=zc),
        "wire_polynomials_ms": lambda: c.wire_polynomials(k, out=polys),
    }
    out = {"op": "permutation argument: 2^16 range_check instances -> sigma polynomials, z(X), z commitment", "rows": rows, "log_domain": k}
    for name, fn in calls.items():
        out[name] = timed(fn)
    _, closing = c.permutation_z(beta, gamma, k, out=z)
    c.permutation_z(beta, gamma, k, form=COEFF, out=zc)
    assert (closing == c.fr_op(0, np.array([[1, 0, 0, 0]], dtype=np.uint64), R2)[0]).all()
    # kernel breakdown of one z evaluation and one sigma evaluation (profiler pass after the timed ones)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        calls["z_evaluations_ms"](); calls["sigma_evaluations_ms"](); torch.cuda.synchronize(dev)
    kern = {}
    for e in p.key_averages():
        t = getattr(e, "self_device_time_total", None) or getattr(e, "self_cuda_time_total", 0)
        for tag in ("k_batch_inv<pg::PermRatioHook>", "k_fr_scan_reduce", "k_fr_scan_apply", "PermSigmaBody", "k_materialize_tiled", "PermBody"):
            if tag in e.key:
                kern[tag] = kern.get(tag, 0.0) + t / 1e3
    out["kernel_ms"] = kern
    if trace_dir:
        os.makedirs(trace_dir, exist_ok=True)
        with open(os.path.join(trace_dir, "bench_permutation_kernels.txt"), "w") as f:
            f.write(p.key_averages().table(sort_by="cuda_time_total", row_limit=40))
    copy_src = torch.empty((N, 4), dtype=torch.int64, device=dev); copy_dst = torch.empty_like(copy_src)
    out["d2d_copy_of_z_ms"] = timed(lambda: copy_dst.copy_(copy_src))
    mul_rate = c.microbench(6)
    out["fr_mul_per_s_microbench"] = mul_rate
    ratio_ms = kern.get("k_batch_inv<pg::PermRatioHook>", 0.0)
    scan_ms = kern.get("k_fr_scan_reduce", 0.0) + kern.get("k_fr_scan_apply", 0.0)
    out["ratio_kernel_fr_mul_rate"] = N * MULS_RATIO / (ratio_ms * 1e-3) if ratio_ms else None
    out["ratio_kernel_share_of_fr_mul_peak"] = out["ratio_kernel_fr_mul_rate"] / mul_rate if ratio_ms else None
    out["z_evaluations_fr_mul_rate"] = N * (MULS_RATIO + MULS_SCAN) / (out["z_evaluations_ms"] * 1e-3)
    out["z_evaluations_share_of_fr_mul_peak"] = out["z_evaluations_fr_mul_rate"] / mul_rate
    # scan traffic: reduce reads N x 32 B, apply reads and writes N x 32 B; a copy of z reads and writes N x 32 B
    out["scan_bytes"] = 3 * N * 32
    out["scan_bytes_per_s"] = out["scan_bytes"] / (scan_ms * 1e-3) if scan_ms else None
    out["scan_fr_mul_rate"] = N * MULS_SCAN / (scan_ms * 1e-3) if scan_ms else None
    out["scan_share_of_fr_mul_peak"] = out["scan_fr_mul_rate"] / mul_rate if scan_ms else None
    out["d2d_copy_bytes_per_s"] = 2 * N * 32 / (out["d2d_copy_of_z_ms"] * 1e-3)
    # commitment of z: Lagrange SRS x evaluations == monomial SRS x coefficients
    mono = torch.empty((N, 12), dtype=torch.int64, device=dev); lag = torch.empty_like(mono)
    c.srs_powers(tau, N, out=mono); c.srs_lagrange(tau, k, out=lag)
    out["z_commit_lagrange_ms"] = timed(lambda: c.msm(lag, z), reps=2)
    out["z_commit_monomial_ms"] = timed(lambda: c.msm(mono, zc), reps=2)
    a, b = c.msm(lag, z), c.msm(mono, zc)
    assert (a == b).all() and a.any()
    out["z_commit_equal"] = True
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out["gpu"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(dev)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
