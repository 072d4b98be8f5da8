#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path: Fr gate evals/sec, range_check batch 2^24 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--log2n 24] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic witnesses:
    fresh composer -> add_input(2^log2n witnesses) -> range_check(0, 2^64) [witness generation: 271 rows / 653 variables
    per instance, written to HBM as the packed variable table] -> gate check of every row (generic evaluation of
    q_m*a*b + q_l*a + q_r*b + q_o*c + q_4*d + q_c + PI, no selector value inspected) -> verdict.
`value`  : rows generated and evaluated per second with the witnesses already resident in HBM (CUDA events, max over ranks).
`e2e`    : the same step through the C ABI with HOST buffers: pinned-host witnesses copied in, per-instance results
           (32 B each) and the verdict copied out, inside the timed region.
Multi-GPU: one process per GPU (torchrun), instances sharded by pg_shard_plan (weak scaling: 2^log2n per GPU; `--scaling strong`:
2^log2n in total), the only collective of the step is the all-reduce of the verdict (pg_check_sharded: NCCL through the C ABI),
executed inside every timed step.  `--impl reference` times the restated reference CPU path (oracle/, faithful cost
structure: per-bit 256-step pow, hash-map variable store, per-row column pushes) on all host cores, rank 0 only.
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last timed step computed as .npy files (dump_outputs below), so
that two builds can be compared output for output: the synthetic witnesses depend only on the arguments.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (it may be read-only)

METRIC = "Fr gate evals/sec, range_check batch 2^24"
UNIT = "gate-evals/s"
ROWS_PER_INSTANCE = 271          # 4k+11, k = 65 (SURVEY.md section 3.1)
VARS_PER_INSTANCE = 653
IMAD_PER_ROW_DEFINITION = 816    # 6 Fr mul x 136 32x32->64 multiply-accumulates (SURVEY.md 8(d)): the DEFINITIONAL cost of a generic gate evaluation
EXECUTED_WIDE_PER_ROW = 420      # wide-class IMADs a row of k_check<GENERIC> executes (SASS): one Montgomery multiplication (64 + 48), a 4-term dot product with one
                                 # shared reduction (256 + 48) and 4 of address arithmetic; the "0 mod q" test compares with a shared-memory table of k*q since
                                 # run r05e (8 more products before); profiles/r05_sass_mix.txt
PACKED_BYTES_PER_INSTANCE = 141 * 32 + 2 * 32   # variable table written by witness generation (141 Fr slots + 2 bit planes)


def ncu_traffic(log2n: int, check_mode: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from a committed `ncu --set full` capture of this
    command (profiles/k_check_traffic.json: one entry per check mode, with the capture's file name and the git revision it was taken
    at).  Returns (bytes or None, provenance)."""
    try:
        with open(os.path.join(ROOT, "profiles", "k_check_traffic.json")) as f:
            t = json.load(f)
        e = t.get(check_mode)
        if e and e.get("log2n") == log2n:
            return e["bytes_per_launch"], f"{e.get('source')} @ {e.get('git')}"
    except Exception:
        pass
    return None, None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_run(log2n_sample: int | None, threads: int, budget_s: float = 15.0):
    """The restated reference CPU path on `threads` host cores over a bounded sample of the same workload."""
    import numpy as np
    from oracle import binding as ob
    ob.build()
    Q = ob.Q
    from tests.programs import synth_wide
    # calibrate on 2 instances per thread, then size the sample for ~budget_s of wall time
    def make(n):
        vals = synth_wide(2, n)
        return ob.from_ints([v if i % 2 else v % 2 ** 64 for i, v in enumerate(vals)])
    mn, mx = ob.from_ints([0]), ob.from_ints([2 ** 64])
    cal_n = 2 * threads
    cal = ob.bench_range(0, make(cal_n), mn, mx, threads, ob.FAITHFUL, 64)
    per_inst = cal["seconds"] / 2.0                              # each thread did 2 instances
    n = int(max(threads, min(1 << 16, budget_s / max(per_inst, 1e-6) * threads)))
    if log2n_sample is not None:
        n = 1 << log2n_sample
    n -= n % threads
    r = ob.bench_range(0, make(n), mn, mx, threads, ob.FAITHFUL, 64)
    assert r["unsat"] == 0 and r["rows"] == n * ROWS_PER_INSTANCE
    fast = ob.bench_range(0, make(n), mn, mx, threads, ob.FAST, 64)
    return {"value": r["rows"] / r["seconds"], "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n} range_check instances (k=65; even index uniform u64, odd uniform Fr), witness generation through the "
                      f"restated composer + gate check, {r['seconds']:.2f} s on {threads} threads",
            "seconds": r["seconds"], "instances": n,
            "optimised_cpu_value": fast["rows"] / fast["seconds"],
            "optimised_cpu_note": "same port with a 2^i table instead of the reference's per-bit 256-step pow"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    vals, secs = [], []
    info = None
    for s in range(args.warmup + args.steps):
        budget = float(os.environ.get("PG_BENCH_CPU_BUDGET_S", max(2.0, 40.0 / max(1, args.warmup + args.steps))))
        info = cpu_reference_run(None, threads, budget_s=budget)
        if s >= args.warmup:
            vals.append(info["value"]); secs.append(info["seconds"])
    v = sum(vals) / len(vals)
    line = {"metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * sum(secs) / len(secs), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32x8 (Fr Montgomery, 4xu64 on CPU)", "data": "synthetic", "impl": "reference",
            "config": {"workload": f"range_check batch 2^{args.log2n}, bounds [0, 2^64) (k=65), bounded sample per step", "timing": "CPU wall clock"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": info["sample"]},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "the Rust reference cannot be built here (no cargo, dusk-plonk not vendored): this is the C restatement "
                    "oracle/ with the reference's cost structure, all host cores, one composer per thread"}
    _emit(line)
    return 0


def bind_to_gpu_numa_node(index: int):
    """One process per GPU: run this process (and first-touch its pinned host buffers) on the CPUs NVML reports as local to GPU `index`,
    so that eight ranks do not stream their host<->device copies through one socket's memory.  Returns the CPU count bound to, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1 and 64 * w + b < n_cpu}
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


DUMP_SEED = 0x64756D70           # the sampled instances depend only on the batch size: the same files on every run
DUMP_RESULTS = 1 << 18           # instances whose range_check result is written (16 MiB)
DUMP_BLOCKS = 256                # instances whose whole variable block (VARS_PER_INSTANCE Fr each) is written (10.7 MB)
DUMP_MAX_BYTES = 64 << 20


def fr_words(a):
    """(..., 4) uint64 Fr limbs as the C ABI returns them (Montgomery form) -> (..., 8) float64 of their little-endian 32-bit words,
    which float64 holds exactly."""
    import numpy as np
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a.view(np.uint32).reshape(a.shape[:-1] + (8,)).astype(np.float64)


def dump_outputs(out_dir: str, c, res, n: int, bad: int, first):
    """What the last timed step handed its caller, as float64 .npy files in out_dir:
      range_check_results[_index]    the result column y (res: all n results of this rank, on the device) at a seeded sample of instances
      variables[_index]              the witness generation's variable block of a smaller seeded sample of instances: (m, 653, 8)
      verdict                        [unsatisfied rows, first unsatisfied row or -1] of the whole batch"""
    import numpy as np
    import torch
    rng = np.random.default_rng(DUMP_SEED)
    idx = np.sort(rng.choice(n, min(n, DUMP_RESULTS), replace=False))
    blk = np.sort(rng.choice(n, min(n, DUMP_BLOCKS), replace=False))
    results = res[torch.from_numpy(idx).to(res.device)].cpu().numpy().view(np.uint64)
    base = c.num_variables() - VARS_PER_INSTANCE * n                 # range_check allocates one block of VARS_PER_INSTANCE per instance, last
    blocks = np.stack([c.variables(base + VARS_PER_INSTANCE * int(i), VARS_PER_INSTANCE) for i in blk])
    arrays = {"range_check_results": fr_words(results), "range_check_results_index": idx.astype(np.float64),
              "variables": fr_words(blocks), "variables_index": blk.astype(np.float64),
              "verdict": np.array([bad, -1 if first is None else first], dtype=np.float64)}
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


_JSON_FD = None


def _claim_stdout():
    """stdout must carry exactly ONE JSON line: keep the real stdout for it and send everything libraries print to fd 1
    (NCCL's version banner, for one) to stderr."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line: dict):
    sys.stdout.flush()
    os.write(_JSON_FD if _JSON_FD is not None else 1, (json.dumps(line) + "\n").encode())


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--log2n", type=int, default=24, help="instances per GPU = 2^log2n (24 = the BASELINE metric configuration)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--check-mode", default="generic", choices=["generic", "sparse", "fused"],
                    help="generic: the headline (no selector inspected); sparse: structure-aware row program; fused: sparse + PG_F_FUSED_CHECK "
                         "(rows evaluated inside witness generation, the table is never re-read)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--check-shape", type=int, default=0, help="launch shape of the gate-check kernel (tuning knob)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: 2^log2n instances per GPU; strong: 2^log2n in total")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (rank 0's instances) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs: not with --impl reference")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    import plonk_gadgets_b200 as pg

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: plonk_gadgets_b200 has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None      # pinned host buffers next to the GPU they feed (end-to-end leg)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    warm = max(args.warmup, 3)
    # one non-default torch stream shared with the engine: torch.cuda.Event and the engine's kernels see the same stream
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    mode = pg.CHECK_GENERIC if args.check_mode == "generic" else pg.CHECK_SPARSE
    c = pg.StandardComposer(device=local, check_mode=mode, timing=True, stream=stream.cuda_stream, check_shape=args.check_shape,
                            fused_check=args.check_mode == "fused")
    assert stream.cuda_stream != 0
    # sharding: the batch of n_total instances is cut by the C ABI's plan; this rank runs [inst_lo, inst_hi) and numbers its rows as
    # the sequential composer of the whole batch does
    n_total = (1 << args.log2n) * (world if args.scaling == "weak" else 1)
    plan = pg.shard_plan([(pg.OP_ADD_INPUT, 0, n_total, 0), (pg.OP_RANGE_CHECK, 65, n_total, 0)], world, pg.SHARD_EVEN)
    mine = plan[rank]
    n = mine[0].inst_hi - mine[0].inst_lo
    if world > 1:
        uid = torch.zeros(pg.api.COMM_ID_BYTES, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid = torch.frombuffer(bytearray(pg.comm_unique_id()), dtype=torch.uint8).to(dev)
        dist.broadcast(uid, 0)
        c.comm_init(bytes(uid.cpu().numpy()), rank, world)          # the engine's own NCCL communicator (verdict all-reduce, gathers)

    # synthetic witnesses: even index uniform u64 (in range), odd index uniform Fr (out of range); per-rank stream id
    wit = torch.empty((n, 4), dtype=torch.int64, device=dev)
    c.synth(0x706C6F6E6B5F6732, 2 + 1000 * rank, 2, 64, wit)
    c.sync()
    from_u64 = lambda v: np.array([[v & (2 ** 64 - 1), v >> 64, 0, 0]], dtype=np.uint64)
    # bounds in Montgomery form via the engine itself: 0 and 2^64 (device kernels; no oracle in the product path)
    raw = np.zeros((2, 4), dtype=np.uint64); raw[1, 1] = 1                 # canonical 0 and 2^64
    r2 = np.array([[0xc999e990f3f29c6d, 0x2b6cedcb87925c23, 0x05d314967254398f, 0x0748d9d99f59ff11]] * 2, dtype=np.uint64)
    bounds = c.fr_op(0, raw, r2)                                           # mont_mul(raw, R^2) = raw * R
    mn, mx = bounds[0:1].copy(), bounds[1:2].copy()
    one_limbs = c.fr_op(0, np.array([[1, 0, 0, 0]], dtype=np.uint64), r2[:1])[0]

    def step_device():
        c.reset()
        w = c.add_input(wit)
        y = pg.range_check(c, mn, mx, w)
        bad, first, _ = c.check_sharded(mine, 0)                            # local gate check + NCCL all-reduce of the verdict
        return y, bad, first

    host_in = torch.empty((n, 4), dtype=torch.int64).pin_memory()
    host_in.copy_(wit.cpu())
    host_out = torch.empty((n, 4), dtype=torch.int64).pin_memory()

    def step_e2e():
        c.reset()
        w = c.add_input(host_in)                                           # cudaMemcpyAsync from pinned host memory
        y = pg.range_check(c, mn, mx, w)
        c.read_column_into(y, host_out, asynchronous=True)                 # per-instance results -> pinned host, on the copy stream
        bad, first, _ = c.check_sharded(mine, 0)                           # verdict of the whole batch (all-reduce; device -> host, 32 B); overlaps with the copy
        c.sync()                                                           # results have arrived
        return bad

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(warm):
        y, bad, first = step_device()
        assert bad == 0, (bad, first)
    c.timing(reset=True)
    sampler = ClockSampler(local); sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    tot_bad = 0
    for _ in range(args.steps):
        y, bad, first = step_device()
        tot_bad += bad
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    tim = c.timing(reset=True)
    # result pattern check on the last step (outside the timed region)
    res = torch.empty((n, 4), dtype=torch.int64, device=dev)
    c.read_column_into(y, res); c.sync()
    one_t = torch.from_numpy(one_limbs.view(np.int64)).to(dev)
    assert bool((res[0::2] == one_t).all()) and bool((res[1::2] == 0).all()) and tot_bad == 0, "result pattern / verdict"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, c, res, n, bad, first)

    # e2e (host buffers, copies inside the timed region)
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3

    # max over ranks (the verdict all-reduce already ran inside every step: `bad` is the whole batch's count)
    t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0]), float(t[1])
    g_bad, g_err = tot_bad, 0
    rows_step_total = n_total * ROWS_PER_INSTANCE
    value = rows_step_total * args.steps / (ms * 1e-3)
    e2e_value = rows_step_total * args.steps / (e2e_ms * 1e-3)

    if rank == 0:
        hbm_peak, hbm_src = peaks()
        wide_peak = c.microbench(1)          # IMAD.WIDE.U32 32x32->64 products per second (product only: the multiplier-pipe ceiling)
        chain_peak = c.microbench(4)         # the same products issued as the multiplier's mad.lo.cc/madc.hi.cc carry chains
        lo_peak = c.microbench(0)
        fr_mul_peak = c.microbench(6)
        # two gate-check launches per step on rank 0 (3-row preamble segment + the range_check segment): report per step
        check_ms = tim["check_ms"] / args.steps
        rows_per_launch = tim["check_rows"] / args.steps
        wit_ms = tim["witness_ms"] / args.steps
        traffic, traffic_src = ncu_traffic(args.log2n if args.scaling == "weak" or world == 1 else -1, args.check_mode)
        table_bytes = n * PACKED_BYTES_PER_INSTANCE
        hbm_obj = lambda kernel, ms_: {"kernel": kernel, "achieved": table_bytes / (ms_ * 1e-3) / 1e9 if ms_ else None, "peak": hbm_peak, "unit": "GB/s",
                                       "peak_source": hbm_src, "frac": (table_bytes / (ms_ * 1e-3) / 1e9 / hbm_peak) if ms_ else None, "ms_per_launch": ms_,
                                       "algorithmic_bytes_per_launch": table_bytes}
        if args.check_mode == "generic":
            executed = rows_per_launch * EXECUTED_WIDE_PER_ROW / (check_ms * 1e-3)
            roofline = {"bound": "imad", "kernel": "k_check<GENERIC>", "achieved": executed / 1e12, "peak": wide_peak / 1e12,
                        "unit": f"T 32x32->64 products/s EXECUTED ({EXECUTED_WIDE_PER_ROW} IMAD.WIDE per gate evaluation)",
                        "frac": executed / wide_peak if wide_peak else None,
                        "peak_source": "measured in this run: IMAD.WIDE.U32 products on all SMs (pg_microbench mode 1)",
                        "frac_of_carry_chain_peak": executed / chain_peak if chain_peak else None,
                        "carry_chain_peak": chain_peak / 1e12, "imad_lo_peak": lo_peak / 1e12, "isolated_fr_mul_per_s": fr_mul_peak,
                        "definitional_816": {"note": "SURVEY.md 8d counts a generic gate evaluation as 6 separate Montgomery multiplications = 816 "
                                                     "multiply-accumulates; the kernel evaluates the factored polynomial with one shared reduction, so this "
                                                     "figure is a rate of DEFINED work, not a pipe utilisation, and may exceed the peak",
                                             "T_mac_per_s": rows_per_launch * IMAD_PER_ROW_DEFINITION / (check_ms * 1e-3) / 1e12},
                        "traffic": traffic, "traffic_source": traffic_src, "ms_per_launch": check_ms,
                        "hbm": hbm_obj("RangePre + k_batch_inv + RangePost (witness generation, 3 launches)", wit_ms)}
        elif args.check_mode == "sparse":
            r = hbm_obj("k_check_prog (structure-aware row program: reads the packed variable table once)", check_ms)
            roofline = {"bound": "hbm", **r, "traffic": traffic, "traffic_source": traffic_src,
                        "hbm_witness": hbm_obj("RangePre + k_batch_inv + RangePost (witness generation, 3 launches)", wit_ms)}
        else:
            r = hbm_obj("RangePre<FUSED> + k_batch_inv + RangePost<FUSED>: witness generation that also evaluates its rows (table written once, "
                        "never re-read for the verdict)", wit_ms)
            roofline = {"bound": "hbm", **r, "traffic": traffic, "traffic_source": traffic_src}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "u32x8 (Fr Montgomery)", "data": "synthetic",
            "config": {"workload": f"range_check batch 2^{args.log2n} {'per GPU' if args.scaling == 'weak' else 'in total'}, bounds [0, 2^64) (k=65): 271 rows / 653 variables per instance",
                       "check_mode": args.check_mode, "l2": "inputs larger than L2 (512 MiB of witnesses, ~77 GB variable table per step)",
                       "timed_region": "composer reset + add_input + witness generation + gate check + verdict all-reduce + verdict read",
                       "instances_per_gpu": n, "instances_total": n_total,
                       "host_numa_binding": f"rank bound to the {numa} CPUs local to its GPU" if numa else "none"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * 32, "d2h_bytes_per_step": n * 32 + 64, "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(tim["check_launches"] + tim["witness_launches"] + tim["other_launches"]),
            "roofline": roofline,
            "kernel_ms": {"check": tim["check_ms"] / args.steps, "witness": tim["witness_ms"] / args.steps, "other": tim["other_ms"] / args.steps},
            "verdict": {"n_unsat": g_bad, "n_err": g_err,
                        "collective": "ncclAllReduce(sum, min) inside every step (pg_check_sharded)" if world > 1 else "world of one rank"},
        }
        if not args.no_cpu_baseline and world == 1:               # the CPU baseline is a single-GPU-run item (rank 0 at N = 1)
            line["cpu_baseline"] = cpu_reference_run(None, os.cpu_count() or 1)
        _emit(line)
    if world > 1:
        dist.barrier()
        c.comm_destroy()
        dist.destroy_process_group()
    c.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
