"""Throughput of prover rounds 4 and 5 (pg_prover_openings) on the circuit of `bench_quotient.py`: 2^16 range_check instances,
17.8 M rows, domain 2^25, t resident on the device.  CUDA events on the engine's stream after a warm-up; one JSON line.

The kernel split (the evaluation pass k_simple<OpenEvalBody> + its sums k_simple<OpenSumBody>, the combination pass
k_simple<OpenCombineBody>, the two Ruffini scans k_fr_ruffini_reduce / k_fr_ruffini_apply, and everything else, which is the rebuild of
the wire, z, sigma and selector coefficient vectors) comes from a torch.profiler pass over one call after the timed ones; `--trace-dir
DIR` also writes its kernel table there.  From counts kept here and times measured in the same run it derives the passes' Fr
multiplications per second against pg_microbench mode 6 and their bytes per second against a device-to-device copy.  The device memory
the call needs is the growth of the ctx's buffer pool over a first call.  Last, rounds 1-5 without the transcript: the wire
commitments, pg_quotient, the z and t_1 .. t_4 commitments, pg_prover_openings and the W_z / W_zw commitments, each timed."""
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

# Evaluation pass (bodies.cuh OpenEvalBody): one Montgomery multiplication per coefficient and pair, 21 pairs at zeta and 4 at
# zeta*w; it reads the 17 coefficient vectors and t_1 .. t_4 once.  Combination pass (OpenCombineBody): 23 multiplications per
# coefficient; it reads 20 vectors (q_arith is not in r) and writes 3.
EVAL_MULS, EVAL_VECTORS = 25, 21
COMB_MULS, COMB_VECTORS = 23, 20 + 3


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
    ch = [mk([0x1234567 + i, 0x89abcdef, 0x42 + i, 0]) for i in range(7)]
    mn, mx = mk([0, 0, 0, 0]), mk([0, 1, 0, 0])
    n = 1 << 16
    wit = torch.empty((n, 4), dtype=torch.int64, device=dev); c.synth(SEED, 2, 2, 64, wit)
    w = c.add_input(wit); pg.range_check(c, mn[None], mx[None], w)
    assert c.check_circuit_satisfied() == (0, None)
    k = c.domain_log_size(); N = 1 << k; rows = c.circuit_size()
    t = torch.empty((4, N, 4), dtype=torch.int64, device=dev)
    o = torch.empty((3, N, 4), dtype=torch.int64, device=dev)
    c.quotient(*ch[:4], k, out=t)
    torch.cuda.synchronize(dev)
    free0 = torch.cuda.mem_get_info(dev)[0]
    c.prover_openings(t, *ch, log_n=k, out=o); torch.cuda.synchronize(dev)
    free1 = torch.cuda.mem_get_info(dev)[0]
    out = {"op": "prover openings (rounds 4, 5): 2^16 range_check instances -> evaluations, W_z, W_zw, r (domain 2^25)", "rows": rows,
           "log_domain": k, "pool_growth_gib": (free0 - free1) / 2 ** 30, "output_gib": 3 * N * 32 / 2 ** 30}
    out["openings_ms"] = timed(lambda: c.prover_openings(t, *ch, log_n=k, out=o), reps=2)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        c.prover_openings(t, *ch, log_n=k, out=o); torch.cuda.synchronize(dev)
    kern, launches, total = {}, {}, 0.0
    for e in p.key_averages():
        tm = (getattr(e, "self_device_time_total", None) or getattr(e, "self_cuda_time_total", 0)) / 1e3
        if tm <= 0:
            continue
        total += tm
        tag = next((g for g in ("OpenEvalBody", "OpenSumBody", "OpenCombineBody", "k_fr_ruffini_reduce", "k_fr_ruffini_apply") if g in e.key),
                   "rebuild_and_other")
        kern[tag] = kern.get(tag, 0.0) + tm
        launches[tag] = launches.get(tag, 0) + e.count
    out["kernel_ms"] = kern; out["kernel_launches"] = launches; out["kernel_total_ms"] = total
    out["ruffini_scan_ms_each"] = (kern.get("k_fr_ruffini_reduce", 0.0) + kern.get("k_fr_ruffini_apply", 0.0)) / 2
    if trace_dir:
        os.makedirs(trace_dir, exist_ok=True)
        with open(os.path.join(trace_dir, "bench_openings_kernels.txt"), "w") as f:
            f.write(p.key_averages().table(sort_by="cuda_time_total", row_limit=40))
    copy_src = torch.empty((N, 4), dtype=torch.int64, device=dev); copy_dst = torch.empty_like(copy_src)
    out["d2d_copy_of_vector_ms"] = timed(lambda: copy_dst.copy_(copy_src))
    out["d2d_copy_bytes_per_s"] = 2 * N * 32 / (out["d2d_copy_of_vector_ms"] * 1e-3)
    mul_rate = c.microbench(6)
    out["fr_mul_per_s_microbench"] = mul_rate
    for name, tag, muls, vecs in (("eval", "OpenEvalBody", EVAL_MULS, EVAL_VECTORS), ("combine", "OpenCombineBody", COMB_MULS, COMB_VECTORS)):
        tm = kern.get(tag, 0.0)
        if tm:
            out[f"{name}_fr_mul_rate"] = N * muls / (tm * 1e-3)
            out[f"{name}_share_of_fr_mul_peak"] = out[f"{name}_fr_mul_rate"] / mul_rate
            out[f"{name}_bytes_per_s"] = N * vecs * 32 / (tm * 1e-3)
            out[f"{name}_share_of_copy_rate"] = out[f"{name}_bytes_per_s"] / out["d2d_copy_bytes_per_s"]
    # rounds 1-5 without the transcript, against a monomial SRS of 2^25 points
    mono = torch.empty((N, 12), dtype=torch.int64, device=dev)
    c.srs_powers(mk([0x5eed, 0x7a0, 0, 0]), N, out=mono)
    z = torch.empty((N, 4), dtype=torch.int64, device=dev)
    c.permutation_z(ch[1], ch[2], k, form=pg.api.FORM_COEFFICIENTS, out=z)
    r15 = {"wire_commitments_ms": timed(lambda: c.commit_wire_polynomials(mono, k), reps=1),
           "z_commitment_ms": timed(lambda: c.msm(mono, z), reps=1),
           "quotient_ms": timed(lambda: c.quotient(*ch[:4], k, out=t), reps=1),
           "t_commitments_ms": timed(lambda: [c.msm(mono, t[r]) for r in range(4)], reps=1),
           "openings_ms": timed(lambda: c.prover_openings(t, *ch, log_n=k, out=o), reps=1),
           "w_commitments_ms": timed(lambda: [c.msm(mono, o[i]) for i in range(2)], reps=1)}
    r15["total_ms"] = sum(r15.values())
    out["rounds_1_to_5_without_transcript"] = r15
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out["gpu"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(dev)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
