"""Throughput of prover round 3 (pg_quotient) on the circuit of `bench_permutation.py`: 2^16 range_check instances, 17.8 M rows,
domain 2^25.  CUDA events on the engine's stream after a warm-up; one JSON line.

The kernel split (transforms k_ntt_pass / k_ntt_coset_pass, the pointwise k_simple<QuotientBody>, the split k_simple<QuotientSplitBody>,
the rest) comes from a torch.profiler pass over one call after the timed ones; `--trace-dir DIR` also writes its kernel table there.
From counts kept here and times measured in the same run it derives the pointwise kernel's Fr multiplications per second against
pg_microbench mode 6, and its bytes per second against a device-to-device copy.  The device memory the call needs is the growth of
the ctx's buffer pool over a first call (the pool keeps every buffer it allocated, so this is the peak of the call)."""
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
dev = torch.device("cuda", 0)
stream = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(stream)
R2 = np.array([[0xc999e990f3f29c6d, 0x2b6cedcb87925c23, 0x05d314967254398f, 0x0748d9d99f59ff11]], dtype=np.uint64)

# QuotientBody per point (bodies.cuh) for a composer without range-widget rows and without PI (this circuit): arithmetic widget 7,
# permutation 18, the division by Z_H 1 -> 26 Montgomery multiplications.  Bytes: 17 evaluation vectors read (4 wires, z, 4 sigma,
# 7 selectors, alpha^2 L_1; z(xw) is the neighbour's entry, mostly from L1), one written, and the twiddle w^k (up to one more read).
MULS_POINT, BYTES_POINT = 26, (17 + 1 + 1) * 32


def timed(fn, reps=3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize(dev); e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream); torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def main():
    trace_dir = sys.argv[sys.argv.index("--trace-dir") + 1] if "--trace-dir" in sys.argv else None
    c = pg.StandardComposer(device=0, stream=stream.cuda_stream)
    mk = lambda raw: c.fr_op(0, np.array([raw], dtype=np.uint64), R2)[0]
    alpha, beta, gamma, rho = (mk([0x1234567 + i, 0x89abcdef, 0x42 + i, 0]) for i in range(4))
    mn, mx = mk([0, 0, 0, 0]), mk([0, 1, 0, 0])
    n = 1 << 16
    wit = torch.empty((n, 4), dtype=torch.int64, device=dev); c.synth(SEED, 2, 2, 64, wit)
    w = c.add_input(wit); pg.range_check(c, mn[None], mx[None], w)
    assert c.check_circuit_satisfied() == (0, None)
    k = c.domain_log_size(); N = 1 << k; rows = c.circuit_size()
    t = torch.empty((4, N, 4), dtype=torch.int64, device=dev)
    torch.cuda.synchronize(dev)
    free0 = torch.cuda.mem_get_info(dev)[0]
    c.quotient(alpha, beta, gamma, rho, k, out=t); torch.cuda.synchronize(dev)
    free1 = torch.cuda.mem_get_info(dev)[0]
    out = {"op": "quotient t(X): 2^16 range_check instances -> t_1..t_4 (domain 2^25)", "rows": rows, "log_domain": k,
           "pool_growth_gib": (free0 - free1) / 2 ** 30, "output_gib": 4 * N * 32 / 2 ** 30}
    top = t[3, -4:].cpu()
    assert not top.any(), "degree bound"
    out["quotient_ms"] = timed(lambda: c.quotient(alpha, beta, gamma, rho, k, out=t), reps=2)
    out["single_transform_ms"] = timed(lambda: c.fft(t[0], inverse=False), reps=4)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        c.quotient(alpha, beta, gamma, rho, k, out=t); torch.cuda.synchronize(dev)
    kern, launches, total = {}, {}, 0.0
    for e in p.key_averages():
        tm = (getattr(e, "self_device_time_total", None) or getattr(e, "self_cuda_time_total", 0)) / 1e3
        if tm <= 0:
            continue
        total += tm
        tag = next((g for g in ("k_ntt_coset_pass", "k_ntt_pass", "QuotientSplitBody", "QuotientBody") if g in e.key), "other")
        kern[tag] = kern.get(tag, 0.0) + tm
        launches[tag] = launches.get(tag, 0) + e.count
    out["kernel_ms"] = kern; out["kernel_launches"] = launches; out["kernel_total_ms"] = total
    if trace_dir:
        os.makedirs(trace_dir, exist_ok=True)
        with open(os.path.join(trace_dir, "bench_quotient_kernels.txt"), "w") as f:
            f.write(p.key_averages().table(sort_by="cuda_time_total", row_limit=40))
    copy_src = torch.empty((N, 4), dtype=torch.int64, device=dev); copy_dst = torch.empty_like(copy_src)
    out["d2d_copy_of_vector_ms"] = timed(lambda: copy_dst.copy_(copy_src))
    out["d2d_copy_bytes_per_s"] = 2 * N * 32 / (out["d2d_copy_of_vector_ms"] * 1e-3)
    mul_rate = c.microbench(6)
    out["fr_mul_per_s_microbench"] = mul_rate
    qb = kern.get("QuotientBody", 0.0)
    if qb:
        out["pointwise_fr_mul_rate"] = 4 * N * MULS_POINT / (qb * 1e-3)
        out["pointwise_share_of_fr_mul_peak"] = out["pointwise_fr_mul_rate"] / mul_rate
        out["pointwise_bytes_per_s"] = 4 * N * BYTES_POINT / (qb * 1e-3)
        out["pointwise_share_of_copy_rate"] = out["pointwise_bytes_per_s"] / out["d2d_copy_bytes_per_s"]
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out["gpu"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(dev)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
