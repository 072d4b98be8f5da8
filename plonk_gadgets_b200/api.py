"""Host-side mirror of plonk_gadgets' public interface over the C ABI (include/pg_b200.h), batched.

Names, argument order and error behaviour follow the reference crate (/root/reference/src/lib.rs:37-45):

    reference (one instance)                                   here (n instances per call)
    -----------------------------------------------------------------------------------------------------------------
    AllocatedScalar::allocate(composer, scalar)                AllocatedScalar.allocate(composer, scalars)
    range_check(composer, min_range, max_range, witness)       range_check(composer, min_range, max_range, witness)
    max_bound(composer, max_range, witness) -> (Variable,u64)  max_bound(composer, max_range, witness) -> (Variables, k)
    maybe_equal(composer, a, b)                                maybe_equal(composer, a, b)
    is_non_zero(composer, var, value_assigned) -> Result       is_non_zero(composer, var, value_assigned)  raises NonExistingInverse
    conditionally_select_zero(composer, x, select)             conditionally_select_zero(composer, x, select)
    conditionally_select_one(composer, y, selector)            conditionally_select_one(composer, y, selector)

A ``Variables`` object is a column of n composer variables (one per instance); scalars are numpy arrays of dtype uint64
and shape (n, 4) holding raw ``BlsScalar`` limbs (Montgomery form), or CUDA tensors/pointers of the same layout.
Every call is equal to the sequential loop ``for i in range(n): gadget(composer, .., operand_i)`` on the reference composer.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

from . import _lib

CHECK_GENERIC, CHECK_SPARSE = 0, 1
F_TIMING = 1
F_FUSED_CHECK = 2
FORM_EVALUATIONS, FORM_COEFFICIENTS = 0, 1
# pg_proof_evaluations: dusk-plonk 0.8 ProofEvaluations' fields in order, then the quotient's evaluation at the challenge
OPENING_EVALUATIONS = ("a_eval", "b_eval", "c_eval", "d_eval", "a_next_eval", "b_next_eval", "d_next_eval", "q_arith_eval", "q_c_eval",
                       "q_l_eval", "q_r_eval", "left_sigma_eval", "right_sigma_eval", "out_sigma_eval", "lin_poly_eval", "perm_eval", "quot_eval")
UINT64_MAX = 2 ** 64 - 1


COMM_ID_BYTES = 128
OP_ADD_INPUT, OP_RANGE_CHECK, OP_MAX_BOUND, OP_MAYBE_EQUAL, OP_IS_NON_ZERO, OP_SELECT_ZERO, OP_SELECT_ONE, OP_CONSTRAIN, OP_RANGE_GATE = range(9)
SHARD_EVEN, SHARD_ROWS = 0, 1


def comm_unique_id() -> bytes:
    """ncclGetUniqueId through the C ABI (rank 0 calls it and hands the 128 bytes to the other ranks)."""
    L = _lib.load()
    buf = (C.c_uint8 * COMM_ID_BYTES)()
    if L.pg_comm_unique_id(buf) != 0:
        raise RuntimeError("pg_comm_unique_id failed (NCCL not loadable?)")
    return bytes(buf)


def op_shape(gadget: int, num_bits: int = 0):
    """(rows, variables) one instance of the gadget appends."""
    L = _lib.load()
    r, v = C.c_uint64(), C.c_uint64()
    if L.pg_op_shape(gadget, num_bits, C.byref(r), C.byref(v)) != 0:
        raise ValueError("unknown gadget / num_bits")
    return r.value, v.value


def template_get(gadget: int, num_bits: int = 0, a=None, b=None, _cdll=None):
    """Rows one instance of a gadget appends (pg_template_get): (w_ref (4, rows) int64, sel (6, rows, 4) uint64, gate (rows,) uint32,
    n_vars).  a / b: the call's public scalars ((4,) uint64 Montgomery limbs): range_check (min, max), max_bound (None, max),
    constrain_to_constant (pi or None, constant)."""
    L = _cdll if _cdll is not None else _lib.load()
    ptr = lambda x: None if x is None else np.ascontiguousarray(x, dtype=np.uint64).reshape(4).ctypes.data_as(C.c_void_p)
    keep = [None if x is None else np.ascontiguousarray(x, dtype=np.uint64).reshape(4) for x in (a, b)]
    pa, pb = (None if k is None else k.ctypes.data_as(C.c_void_p) for k in keep)
    rows, nv = C.c_uint64(), C.c_uint64()
    if L.pg_template_get(gadget, num_bits, pa, pb, C.byref(rows), C.byref(nv), None, None, None) != 0:
        raise ValueError("pg_template_get: bad gadget / bounds / num_bits")
    w = np.zeros((4, rows.value), dtype=np.int64); sel = np.zeros((6, rows.value, 4), dtype=np.uint64); gate = np.zeros(rows.value, dtype=np.uint32)
    rc = L.pg_template_get(gadget, num_bits, pa, pb, C.byref(rows), C.byref(nv), w.ctypes.data_as(C.c_void_p), sel.ctypes.data_as(C.c_void_p),
                           gate.ctypes.data_as(C.c_void_p))
    assert rc == 0
    return w, sel, gate, nv.value


def shard_plan(ops, world: int, policy: int = SHARD_EVEN, _cdll=None):
    """ops: list of (gadget, num_bits, n, group).  Returns plan[rank][k] = pg_op_shard(inst_lo, inst_hi, row_base, var_base): what
    `rank` runs of call k and where it sits in the sequential composer (pure host code, no GPU needed)."""
    L = _cdll if _cdll is not None else _lib.load()
    n = len(ops)
    arr = (_lib.pg_op * n)(*[_lib.pg_op(g, k, cnt, grp, 0) for (g, k, cnt, grp) in ops])
    out = (_lib.pg_op_shard * (n * world))()
    rc = L.pg_shard_plan(arr, n, world, policy, out)
    if rc != 0:
        raise ValueError(f"pg_shard_plan: {L.pg_strerror(rc).decode()}")
    return [[out[r * n + k] for k in range(n)] for r in range(world)]


class Error(Exception):
    """Gadget errors (/root/reference/src/errors.rs:13-18)."""


class NonExistingInverse(Error):
    """Error::NonExistingInverse (/root/reference/src/errors.rs:17, returned at /root/reference/src/scalar.rs:79)."""

    def __init__(self, n_err: int, first_err: int):
        super().__init__(f"value_assigned is zero for {n_err} instance(s), first at index {first_err}")
        self.n_err, self.first_err = n_err, first_err


class EngineError(RuntimeError):
    """Negative return codes of the C ABI (CUDA failure, bad argument, out of memory, ...)."""

    def __init__(self, code: int, what: str, detail: str):
        super().__init__(f"{what} (code {code}): {detail}")
        self.code = code


class DevicePtr:
    """n scalars living in device memory (32 bytes each, 16-byte aligned)."""

    def __init__(self, ptr: int, n: int, owner=None):
        self.ptr, self.n, self.owner = int(ptr), int(n), owner


def _scalars(x):
    """-> (pointer, on_device, n, keepalive)"""
    if isinstance(x, DevicePtr):
        return C.c_void_p(x.ptr), 1, x.n, x
    if hasattr(x, "data_ptr") and hasattr(x, "is_cuda"):          # torch tensor, without importing torch here
        if not x.is_contiguous():
            raise ValueError("scalar tensors must be contiguous")
        n = x.numel() * x.element_size() // 32
        if x.is_cuda:
            return C.c_void_p(x.data_ptr()), 1, n, x
        return C.c_void_p(x.data_ptr()), 0, n, x
    a = np.ascontiguousarray(x, dtype=np.uint64)
    if a.ndim == 1 and a.shape[0] == 4:
        a = a.reshape(1, 4)
    if a.ndim != 2 or a.shape[1] != 4:
        raise ValueError("scalars must have shape (n, 4) uint64")
    return a.ctypes.data_as(C.c_void_p), 0, a.shape[0], a


@dataclass(frozen=True)
class Variables:
    """A column of n `Variable`s: element i is the variable instance i of the producing call allocated."""
    composer: "StandardComposer"
    col: int
    n: int

    def ids(self) -> np.ndarray:
        """The reference's Variable indices (first + i*stride)."""
        first, stride = self.composer._col_geometry(self.col)
        return first + stride * np.arange(self.n, dtype=np.uint64)

    def values(self, i0: int = 0, cnt: int | None = None) -> np.ndarray:
        """composer.variables[var] for the column, as (cnt, 4) uint64."""
        return self.composer.read_column(self, i0, cnt)


@dataclass(frozen=True)
class AllocatedScalar:
    """/root/reference/src/allocated_scalar.rs:17-31 -- here `var` is a column and `scalar` its values (read on demand)."""
    var: Variables

    @property
    def scalar(self) -> np.ndarray:
        return self.var.values()

    @staticmethod
    def allocate(composer: "StandardComposer", scalar) -> "AllocatedScalar":
        return AllocatedScalar(composer.add_input(scalar))


class StandardComposer:
    """Device-resident batched composer (dusk-plonk StandardComposer, arithmetic-row subset).  Fresh state: 3 rows, 5 variables."""

    def __init__(self, device: int = 0, check_mode: int = CHECK_GENERIC, timing: bool = False, stream: int | None = None, check_shape: int = 0,
                 fused_check: bool = False, _cdll=None):
        self._L = _cdll if _cdll is not None else _lib.load()
        cfg = _lib.pg_cfg(device=device, check_mode=check_mode, flags=(F_TIMING if timing else 0) | (F_FUSED_CHECK if fused_check else 0), check_shape=check_shape, stream=stream)
        ctx = C.c_void_p()
        rc = self._L.pg_ctx_create(C.byref(cfg), C.byref(ctx))
        if rc != 0:
            raise EngineError(rc, "pg_ctx_create", self._L.pg_strerror(rc).decode())
        self._ctx = ctx
        self._keep = []

    def close(self):
        if getattr(self, "_ctx", None):
            self._L.pg_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing
    def _ok(self, rc: int, what: str):
        if rc < 0:
            raise EngineError(rc, what, self._L.pg_last_error(self._ctx).decode())
        return rc

    def _col_geometry(self, col: int):
        n, first, stride = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._ok(self._L.pg_col_info(self._ctx, col, C.byref(n), C.byref(first), C.byref(stride)), "pg_col_info")
        return first.value, stride.value

    def reset(self):
        self._ok(self._L.pg_composer_reset(self._ctx), "pg_composer_reset")
        self._keep.clear()

    def sync(self):
        self._ok(self._L.pg_sync(self._ctx), "pg_sync")
        self._keep.clear()

    # -- composer surface used by the gadgets and the reference's tests
    def add_input(self, scalars) -> Variables:
        p, dev, n, keep = _scalars(scalars)
        self._keep.append(keep)
        out = C.c_uint64()
        self._ok(self._L.pg_add_input_batch(self._ctx, n, p, dev, C.byref(out)), "pg_add_input_batch")
        return Variables(self, out.value, n)

    def constrain_to_constant(self, a: Variables, constant, pi=None):
        pc, dev, nc, k1 = _scalars(constant)
        pp, npi, k2 = None, 0, None
        if pi is not None:
            pp, dev2, npi, k2 = _scalars(pi)
            if dev2 != dev:
                raise ValueError("constant and pi must both be host or both be device scalars")
        self._keep += [k1, k2]
        self._ok(self._L.pg_constrain_to_constant_batch(self._ctx, a.col, pc, nc, pp, npi, dev), "pg_constrain_to_constant_batch")

    def range_gate(self, witness: Variables, num_bits: int):
        """composer.range_gate(witness, num_bits) for every variable of the column [dusk-plonk StandardComposer::range_gate, the native
        quad-accumulator gate /root/reference/src/range.rs:9-12 recommends for power-of-two bounds]; num_bits even, 2..256."""
        self._ok(self._L.pg_range_gate_batch(self._ctx, witness.col, int(num_bits)), "pg_range_gate_batch")

    def circuit_size(self) -> int:
        r, v = C.c_uint64(), C.c_uint64()
        self._ok(self._L.pg_counts(self._ctx, C.byref(r), C.byref(v)), "pg_counts")
        return r.value

    def num_variables(self) -> int:
        r, v = C.c_uint64(), C.c_uint64()
        self._ok(self._L.pg_counts(self._ctx, C.byref(r), C.byref(v)), "pg_counts")
        return v.value

    def check_circuit_satisfied(self):
        """(number of unsatisfied rows, first unsatisfied row or None): the arithmetic gate equation on every row."""
        bad, first = C.c_uint64(), C.c_uint64()
        self._ok(self._L.pg_check(self._ctx, C.byref(bad), C.byref(first)), "pg_check")
        return bad.value, (None if first.value == UINT64_MAX else first.value)

    def export(self, path: str, chunk_rows: int = 0, sigma: bool = False):
        """pg_export_composer: the whole composer (calls, Variable values as to_bytes, wire ids, selector columns, dense PI, optionally
        the permutation) in one chunked file -- the import adapter's input (read it back with plonk_gadgets_b200.export_format)."""
        self._ok(self._L.pg_export_composer(self._ctx, os.fsencode(path), chunk_rows, 1 if sigma else 0), "pg_export_composer")

    # -- multi-GPU: communicator, sharded verdict, gathers (include/pg_b200.h "multi-GPU"; SURVEY.md 8e)
    def comm_init(self, unique_id: bytes, rank: int, world: int):
        """Joins the communicator of the box's ranks (collective).  unique_id: comm_unique_id() of rank 0, handed over out of band."""
        if len(unique_id) != COMM_ID_BYTES:
            raise ValueError("unique_id must be COMM_ID_BYTES long")
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(unique_id)
        self._ok(self._L.pg_comm_init(self._ctx, buf, rank, world), "pg_comm_init")

    def comm_destroy(self):
        self._ok(self._L.pg_comm_destroy(self._ctx), "pg_comm_destroy")

    def check_sharded(self, mine=None, n_err: int = 0):
        """pg_check of this rank's shard + all-reduce: (n_unsat, first bad row in the sequential composer's numbering or None, n_err)
        of the WHOLE circuit.  mine: this rank's row of shard_plan(...) (list of pg_op_shard) or None."""
        bad, first, err = C.c_uint64(), C.c_uint64(), C.c_uint64(n_err)
        arr, n_ops = None, 0
        if mine is not None:
            n_ops = len(mine)
            arr = (_lib.pg_op_shard * n_ops)(*mine)
        self._ok(self._L.pg_check_sharded(self._ctx, arr, n_ops, C.byref(bad), C.byref(first), C.byref(err)), "pg_check_sharded")
        return bad.value, (None if first.value == UINT64_MAX else first.value), err.value

    def gather_column(self, v: "Variables", out):
        """All-gather of a column (per-instance results of a call): fills `out` (host array or device tensor sized for the shards of
        all ranks) in rank order = instance order of the whole batch.  Returns (total, [count of rank 0, count of rank 1, ...])."""
        counts = (C.c_uint64 * 64)()
        total = C.c_uint64()
        p, dev, n, keep = _scalars(out)
        self._ok(self._L.pg_gather_column(self._ctx, v.col, p, n, dev, counts, C.byref(total)), "pg_gather_column")
        return total.value, [int(x) for x in counts]

    def gather_variables(self, call: int, out):
        """Gather of witness shards: the Variables of call `call` from all ranks, in the sequential composer's order.  Returns the total."""
        total = C.c_uint64()
        p, dev, n, keep = _scalars(out)
        self._ok(self._L.pg_gather_variables(self._ctx, call, p, n, dev, C.byref(total)), "pg_gather_variables")
        return total.value

    # -- read-back in the reference's representation
    def read_column(self, v: Variables, i0: int = 0, cnt: int | None = None) -> np.ndarray:
        cnt = v.n - i0 if cnt is None else cnt
        out = np.empty((cnt, 4), dtype=np.uint64)
        self._ok(self._L.pg_col_read(self._ctx, v.col, i0, cnt, out.ctypes.data_as(C.c_void_p), 0), "pg_col_read")
        return out

    def read_column_into(self, v: Variables, dst, i0: int = 0, cnt: int | None = None, asynchronous: bool = False):
        """Device (or host) destination variant of read_column.  asynchronous=True (pinned host tensors only): the copy runs on
        the engine's copy stream, overlaps with whatever is enqueued next, and is complete after sync()."""
        cnt = v.n - i0 if cnt is None else cnt
        p, dev, n, keep = _scalars(dst)
        if n < cnt:
            raise ValueError("destination too small")
        if asynchronous:
            if dev or not (hasattr(dst, "is_pinned") and dst.is_pinned()):
                raise ValueError("asynchronous reads need a pinned host tensor")
            self._keep.append(keep)
            dev = 2
        self._ok(self._L.pg_col_read(self._ctx, v.col, i0, cnt, p, dev), "pg_col_read")

    def variables(self, var0: int = 0, cnt: int | None = None) -> np.ndarray:
        cnt = self.num_variables() - var0 if cnt is None else cnt
        out = np.empty((cnt, 4), dtype=np.uint64)
        self._ok(self._L.pg_read_variables(self._ctx, var0, cnt, out.ctypes.data_as(C.c_void_p), 0), "pg_read_variables")
        return out

    def rows(self, row0: int = 0, cnt: int | None = None, want=("w_idx", "w_val", "sel", "pi")) -> dict:
        """Materialised rows: w_idx (4,cnt) uint64, w_val (4,cnt,4), sel (6,cnt,4) in q_m q_l q_r q_o q_4 q_c order, pi (cnt,4)."""
        cnt = self.circuit_size() - row0 if cnt is None else cnt
        out = {}
        if "w_idx" in want: out["w_idx"] = np.empty((4, cnt), dtype=np.uint64)
        if "w_val" in want: out["w_val"] = np.empty((4, cnt, 4), dtype=np.uint64)
        if "sel" in want: out["sel"] = np.empty((6, cnt, 4), dtype=np.uint64)
        if "pi" in want: out["pi"] = np.empty((cnt, 4), dtype=np.uint64)
        ptr = lambda k: out[k].ctypes.data_as(C.c_void_p) if k in out else None
        self._ok(self._L.pg_materialize_rows(self._ctx, row0, cnt, ptr("w_idx"), ptr("w_val"), ptr("sel"), ptr("pi"), 0), "pg_materialize_rows")
        return out

    def poke_variable(self, var: int, value) -> None:
        """Fault injection: composer.variables[var] = value ((4,) uint64 Montgomery limbs); rows are left as they are."""
        v = np.ascontiguousarray(value, dtype=np.uint64).reshape(4)
        self._ok(self._L.pg_poke_variable(self._ctx, int(var), v.ctypes.data_as(C.c_void_p)), "pg_poke_variable")

    def gate_selectors(self, row0: int = 0, cnt: int | None = None):
        """(q_arith, q_range), each (cnt,4): 1 / 0 on arithmetic rows, 0 / 1 on the rows of range_gate (0 / 0 on its closing gate)."""
        cnt = self.circuit_size() - row0 if cnt is None else cnt
        qa = np.empty((cnt, 4), dtype=np.uint64); qr = np.empty((cnt, 4), dtype=np.uint64)
        self._ok(self._L.pg_materialize_gate_selectors(self._ctx, row0, cnt, qa.ctypes.data_as(C.c_void_p), qr.ctypes.data_as(C.c_void_p), 0),
                 "pg_materialize_gate_selectors")
        return qa, qr

    def check_rows(self, w_val, sel, pi=None, q_arith=None, q_range=None):
        """Gate equation over caller-supplied materialised rows (host arrays).  With q_arith / q_range (cnt,4) the range widget's
        term is included (pg_check_rows_ex); without them the arithmetic widget alone."""
        w = np.ascontiguousarray(w_val, dtype=np.uint64); s = np.ascontiguousarray(sel, dtype=np.uint64)
        n = w.shape[1]
        p = np.ascontiguousarray(pi, dtype=np.uint64) if pi is not None else None
        bad, first = C.c_uint64(), C.c_uint64()
        if q_arith is not None or q_range is not None:
            qa = np.ascontiguousarray(q_arith, dtype=np.uint64) if q_arith is not None else None
            qr = np.ascontiguousarray(q_range, dtype=np.uint64) if q_range is not None else None
            vp = lambda x: x.ctypes.data_as(C.c_void_p) if x is not None else None
            self._ok(self._L.pg_check_rows_ex(self._ctx, n, vp(w), vp(s), vp(p), vp(qa), vp(qr), 0, C.byref(bad), C.byref(first)), "pg_check_rows_ex")
            return bad.value, (None if first.value == UINT64_MAX else first.value)
        self._ok(self._L.pg_check_rows(self._ctx, n, w.ctypes.data_as(C.c_void_p), s.ctypes.data_as(C.c_void_p),
                                       p.ctypes.data_as(C.c_void_p) if p is not None else None, 0, C.byref(bad), C.byref(first)), "pg_check_rows")
        return bad.value, (None if first.value == UINT64_MAX else first.value)

    def permutation(self, row0: int = 0, cnt: int | None = None) -> np.ndarray:
        """(4, cnt) uint64: cycle successor (row*4 + wire) of every wire position -- the copy-constraint map of the composer."""
        cnt = self.circuit_size() - row0 if cnt is None else cnt
        out = np.empty((4, cnt), dtype=np.uint64)
        self._ok(self._L.pg_permutation(self._ctx, row0, cnt, out.ctypes.data_as(C.c_void_p), 0), "pg_permutation")
        return out

    # -- evaluation domain: EvaluationDomain::fft / ifft and the wire polynomials of Prover::prove ([DEP] dusk-plonk 0.8)
    def fft(self, scalars, inverse: bool = False, out=None):
        """FFT / inverse FFT of 2^k scalars over dusk-plonk's evaluation domain (natural order in and out).
        Host: (n, 4) uint64 array in, new array out.  Device: anything with data_ptr() (in place unless `out` is given)."""
        if hasattr(scalars, "data_ptr"):
            n = scalars.shape[0]
            dst = scalars if out is None else out
            src_p, dst_p, on_dev = C.c_void_p(scalars.data_ptr()), C.c_void_p(dst.data_ptr()), 1
        else:
            a = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)
            n = a.shape[0]
            dst = np.empty_like(a)
            src_p, dst_p, on_dev = a.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p), 0
        if n == 0 or n & (n - 1):
            raise ValueError("fft: the number of scalars must be a power of two")
        self._ok(self._L.pg_fft(self._ctx, n.bit_length() - 1, 1 if inverse else 0, src_p, dst_p, on_dev), "pg_fft")
        return dst

    def domain_log_size(self) -> int:
        """log2 of EvaluationDomain::new(circuit_size).size()."""
        return max(self.circuit_size() - 1, 0).bit_length()

    def wire_polynomials(self, log_n: int | None = None, out=None):
        """Coefficients of w_l, w_r, w_o, w_4: (4, 2^log_n, 4) uint64 (host array, or written to the device tensor `out`)."""
        log_n = self.domain_log_size() if log_n is None else log_n
        if not 0 <= log_n <= 32 or (1 << log_n) < self.circuit_size():
            raise EngineError(-2, "pg_wire_polynomials", f"a domain of 2^{log_n} cannot hold {self.circuit_size()} rows (or exceeds 2^32)")
        if out is not None:
            self._ok(self._L.pg_wire_polynomials(self._ctx, log_n, C.c_void_p(out.data_ptr()), 1), "pg_wire_polynomials")
            return out
        dst = np.empty((4, 1 << log_n, 4), dtype=np.uint64)
        self._ok(self._L.pg_wire_polynomials(self._ctx, log_n, dst.ctypes.data_as(C.c_void_p), 0), "pg_wire_polynomials")
        return dst

    # -- permutation argument: preprocessing's sigma polynomials and prover round 2's z(X) ([DEP] dusk-plonk 0.8 permutation.rs)
    def _domain(self, log_n):
        log_n = self.domain_log_size() if log_n is None else log_n
        if not 0 <= log_n <= 32:
            raise EngineError(-2, "permutation argument", f"log_n = {log_n} is outside 0..32")
        return log_n

    def sigma_polynomials(self, log_n: int | None = None, form: int = FORM_EVALUATIONS, out=None):
        """sigma_w over the domain 2^log_n: (4, 2^log_n, 4) uint64 evaluations or coefficients (host array, or written to the
        device tensor `out`)."""
        log_n = self._domain(log_n)
        if out is not None:
            self._ok(self._L.pg_sigma_polynomials(self._ctx, log_n, form, C.c_void_p(out.data_ptr()), 1), "pg_sigma_polynomials")
            return out
        dst = np.empty((4, 1 << log_n, 4), dtype=np.uint64)
        self._ok(self._L.pg_sigma_polynomials(self._ctx, log_n, form, dst.ctypes.data_as(C.c_void_p), 0), "pg_sigma_polynomials")
        return dst

    def _z_call(self, fn, what, log_n, head, beta, gamma, form, out):
        b = np.ascontiguousarray(beta, dtype=np.uint64).reshape(4); g = np.ascontiguousarray(gamma, dtype=np.uint64).reshape(4)
        closing = np.zeros(4, dtype=np.uint64)
        vp = lambda x: x.ctypes.data_as(C.c_void_p)
        if out is not None:
            self._ok(fn(self._ctx, log_n, *head, vp(b), vp(g), form, C.c_void_p(out.data_ptr()), 1, vp(closing)), what)
            return out, closing
        dst = np.empty((1 << log_n, 4), dtype=np.uint64)
        self._ok(fn(self._ctx, log_n, *head, vp(b), vp(g), form, vp(dst), 0, vp(closing)), what)
        return dst, closing

    def permutation_z(self, beta, gamma, log_n: int | None = None, form: int = FORM_EVALUATIONS, out=None):
        """(z, closing): the grand-product polynomial over the domain 2^log_n ((2^log_n, 4) uint64, or the device tensor `out`)
        and the product of all 2^log_n ratios ((4,) uint64; one on every honestly wired composer)."""
        return self._z_call(self._L.pg_permutation_z, "pg_permutation_z", self._domain(log_n), (), beta, gamma, form, out)

    def permutation_z_rows(self, w_val, sigma, beta, gamma, log_n: int, form: int = FORM_EVALUATIONS, out=None):
        """permutation_z over caller-supplied rows: w_val (4, n, 4) wire values and sigma (4, n) positions (row*4 + wire), both host
        arrays or both device tensors; rows n .. 2^log_n are padding."""
        if hasattr(w_val, "data_ptr"):
            n = w_val.shape[1]
            head = (n, C.c_void_p(w_val.data_ptr()), C.c_void_p(sigma.data_ptr()), 1)
        else:
            w = np.ascontiguousarray(w_val, dtype=np.uint64); s = np.ascontiguousarray(sigma, dtype=np.uint64)
            n = w.shape[1]
            if s.shape != (4, n):
                raise ValueError("permutation_z_rows: sigma must be (4, n) for w_val (4, n, 4)")
            head = (n, w.ctypes.data_as(C.c_void_p), s.ctypes.data_as(C.c_void_p), 0)
        return self._z_call(self._L.pg_permutation_z_rows, "pg_permutation_z_rows", log_n, head, beta, gamma, form, out)

    # -- quotient polynomial: preprocessing's selector / public-input polynomials and prover round 3's t(X) ([DEP] quotient_poly.rs)
    def _columns(self, fn, what, cols, log_n, form, out):
        log_n = self._domain(log_n)
        if out is not None:
            self._ok(fn(self._ctx, log_n, form, C.c_void_p(out.data_ptr()), 1), what)
            return out
        dst = np.empty((cols, 1 << log_n, 4), dtype=np.uint64)
        self._ok(fn(self._ctx, log_n, form, dst.ctypes.data_as(C.c_void_p), 0), what)
        return dst

    def selector_polynomials(self, log_n: int | None = None, form: int = FORM_EVALUATIONS, out=None):
        """q_m q_l q_r q_o q_4 q_c q_arith q_range over the domain 2^log_n (padding rows zero): (8, 2^log_n, 4) uint64 evaluations
        or coefficients (host array, or written to the device tensor `out`)."""
        return self._columns(self._L.pg_selector_polynomials, "pg_selector_polynomials", 8, log_n, form, out)

    def public_input_polynomial(self, log_n: int | None = None, form: int = FORM_EVALUATIONS, out=None):
        """The dense public-input vector padded to 2^log_n, or PI(X)'s coefficients: (2^log_n, 4) uint64 (or the device tensor `out`)."""
        r = self._columns(self._L.pg_public_input_polynomial, "pg_public_input_polynomial", 1, log_n, form, out)
        return r if out is not None else r[0]

    def quotient(self, alpha, beta, gamma, range_challenge, log_n: int | None = None, out=None):
        """Prover round 3: t_1 .. t_4, (4, 2^log_n, 4) uint64 coefficients (or written to the device tensor `out`); the challenges
        are one Montgomery scalar each.  log_n <= 30."""
        log_n = self._domain(log_n)
        if log_n > 30:
            raise EngineError(-2, "pg_quotient", f"log_n = {log_n}: the 4N coset needs 2-adicity log_n + 2 <= 32")
        ch = [np.ascontiguousarray(x, dtype=np.uint64).reshape(4) for x in (alpha, beta, gamma, range_challenge)]
        vp = lambda x: x.ctypes.data_as(C.c_void_p)
        if out is not None:
            self._ok(self._L.pg_quotient(self._ctx, log_n, *map(vp, ch), C.c_void_p(out.data_ptr()), 1), "pg_quotient")
            return out
        dst = np.empty((4, 1 << log_n, 4), dtype=np.uint64)
        self._ok(self._L.pg_quotient(self._ctx, log_n, *map(vp, ch), vp(dst), 0), "pg_quotient")
        return dst

    # -- openings: prover rounds 4 and 5 ([DEP] Prover::prove, linearisation_poly::compute, Polynomial::ruffini)
    def prover_openings(self, t, alpha, beta, gamma, range_challenge, z, v, v_shifted, log_n: int | None = None, out=None):
        """Prover rounds 4 and 5 for pg_quotient's t_1 .. t_4 (a (4, 2^log_n, 4) host array or device tensor) and the challenges (one
        Montgomery scalar each; z is the evaluation challenge, v / v_shifted aggregate the openings at z and z*w): (evaluations, openings).
        evaluations: dict name -> (4,) uint64 in ProofEvaluations' order plus quot_eval (OPENING_EVALUATIONS); openings: [W_z, W_zw, r],
        (3, 2^log_n, 4) uint64 coefficients (or written to the device tensor `out`).  log_n <= 30."""
        log_n = self._domain(log_n)
        if log_n > 30:
            raise EngineError(-2, "pg_prover_openings", f"log_n = {log_n}: the quotient's domain bound is 2^30")
        ch = np.ascontiguousarray(np.stack([np.ascontiguousarray(x, dtype=np.uint64).reshape(4)
                                            for x in (alpha, beta, gamma, range_challenge, z, v, v_shifted)]))
        vp = lambda x: x.ctypes.data_as(C.c_void_p)
        ev = np.zeros((len(OPENING_EVALUATIONS), 4), dtype=np.uint64)
        if isinstance(t, np.ndarray):
            t = np.ascontiguousarray(t, dtype=np.uint64)
            if t.shape != (4, 1 << log_n, 4):
                raise EngineError(-2, "pg_prover_openings", f"t has shape {t.shape}, expected {(4, 1 << log_n, 4)}")
            t_ptr, t_dev = vp(t), 0
        else:
            if tuple(t.shape) != (4, 1 << log_n, 4) or not t.is_contiguous():
                raise EngineError(-2, "pg_prover_openings", f"t must be a contiguous (4, 2^{log_n}, 4) tensor")
            t_ptr, t_dev = C.c_void_p(t.data_ptr()), 1
        if out is not None:
            self._ok(self._L.pg_prover_openings(self._ctx, log_n, vp(ch), t_ptr, t_dev, vp(ev), C.c_void_p(out.data_ptr()), 1), "pg_prover_openings")
            dst = out
        else:
            dst = np.empty((3, 1 << log_n, 4), dtype=np.uint64)
            self._ok(self._L.pg_prover_openings(self._ctx, log_n, vp(ch), t_ptr, t_dev, vp(ev), vp(dst), 0), "pg_prover_openings")
        return dict(zip(OPENING_EVALUATIONS, ev)), dst

    # -- commitments: G1 multi-scalar multiplication, SRS powers, wire-polynomial commitments ([DEP] dusk-plonk 0.8 / dusk-bls12_381)
    @staticmethod
    def _points(x):
        """(pointer, on_device, n, keep-alive): points are (n, 12) uint64 = n x {x: Fp, y: Fp} Montgomery limbs; all-zero = infinity."""
        if hasattr(x, "data_ptr"):
            return C.c_void_p(x.data_ptr()), 1, x.shape[0], x
        a = np.ascontiguousarray(x, dtype=np.uint64).reshape(-1, 12)
        return a.ctypes.data_as(C.c_void_p), 0, a.shape[0], a

    def msm(self, points, scalars) -> np.ndarray:
        """sum_i scalars[i] * points[i] -> (12,) uint64 affine point (msm_variable_base)."""
        pp, pdev, n, _k1 = self._points(points)
        if hasattr(scalars, "data_ptr"):
            sp, sdev, sn, _k2 = C.c_void_p(scalars.data_ptr()), 1, scalars.shape[0], scalars
        else:
            _k2 = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)
            sp, sdev, sn = _k2.ctypes.data_as(C.c_void_p), 0, _k2.shape[0]
        if n != sn or pdev != sdev:
            raise ValueError("msm: points and scalars must have the same length and live on the same side")
        out = np.zeros(12, dtype=np.uint64)
        self._ok(self._L.pg_msm(self._ctx, n, pp, sp, out.ctypes.data_as(C.c_void_p), pdev), "pg_msm")
        return out

    def srs_powers(self, beta, n: int, base=None, out=None):
        """powers_of_g[i] = beta^i * base (default base: the G1 generator) -- PublicParameters::setup."""
        b = np.ascontiguousarray(beta, dtype=np.uint64).reshape(4)
        bp = None if base is None else np.ascontiguousarray(base, dtype=np.uint64).reshape(12)
        bptr = None if bp is None else bp.ctypes.data_as(C.c_void_p)
        if out is not None:
            self._ok(self._L.pg_srs_powers(self._ctx, b.ctypes.data_as(C.c_void_p), bptr, n, C.c_void_p(out.data_ptr()), 1), "pg_srs_powers")
            return out
        res = np.zeros((n, 12), dtype=np.uint64)
        self._ok(self._L.pg_srs_powers(self._ctx, b.ctypes.data_as(C.c_void_p), bptr, n, res.ctypes.data_as(C.c_void_p), 0), "pg_srs_powers")
        return res

    def g1_fixed_base_mul(self, scalars, base=None) -> np.ndarray:
        a = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)
        bp = None if base is None else np.ascontiguousarray(base, dtype=np.uint64).reshape(12)
        res = np.zeros((a.shape[0], 12), dtype=np.uint64)
        self._ok(self._L.pg_g1_fixed_base_mul(self._ctx, a.shape[0], None if bp is None else bp.ctypes.data_as(C.c_void_p),
                                              a.ctypes.data_as(C.c_void_p), res.ctypes.data_as(C.c_void_p), 0), "pg_g1_fixed_base_mul")
        return res

    def commit_wire_polynomials(self, powers_of_g, log_n: int | None = None) -> np.ndarray:
        """(4, 12) uint64: commitments to w_l, w_r, w_o, w_4 against powers_of_g[0 .. 2^log_n)."""
        log_n = self.domain_log_size() if log_n is None else log_n
        pp, pdev, n, _keep = self._points(powers_of_g)
        out = np.zeros((4, 12), dtype=np.uint64)
        self._ok(self._L.pg_commit_wire_polynomials(self._ctx, log_n, pp, n, pdev, out.ctypes.data_as(C.c_void_p)), "pg_commit_wire_polynomials")
        return out

    def srs_lagrange(self, beta, log_n: int, base=None, out=None):
        """Lagrange-basis SRS of the domain 2^log_n: out[i] = L_i(beta) * base (local setups that know beta)."""
        b = np.ascontiguousarray(beta, dtype=np.uint64).reshape(4)
        bp = None if base is None else np.ascontiguousarray(base, dtype=np.uint64).reshape(12)
        bptr = None if bp is None else bp.ctypes.data_as(C.c_void_p)
        if out is not None:
            self._ok(self._L.pg_srs_lagrange(self._ctx, b.ctypes.data_as(C.c_void_p), bptr, log_n, C.c_void_p(out.data_ptr()), 1), "pg_srs_lagrange")
            return out
        res = np.zeros((1 << log_n, 12), dtype=np.uint64)
        self._ok(self._L.pg_srs_lagrange(self._ctx, b.ctypes.data_as(C.c_void_p), bptr, log_n, res.ctypes.data_as(C.c_void_p), 0), "pg_srs_lagrange")
        return res

    def srs_lagrange_from_powers(self, powers, log_n: int, out=None):
        """Lagrange-basis SRS of the domain 2^log_n from the monomial powers alone: out[i] = (1/n) sum_j w^(-ij) powers[j] over the
        first n = 2^log_n powers (a group inverse FFT; equals srs_lagrange(beta, log_n) when powers[j] = beta^j * G).  powers: (m, 12)
        uint64 on the host or a device tensor; out: a device tensor to fill, else a new (n, 12) host array is returned."""
        pp, pdev, m, _keep = self._points(powers)
        if out is not None:
            self._ok(self._L.pg_srs_lagrange_from_powers(self._ctx, log_n, pp, m, pdev, C.c_void_p(out.data_ptr()), 1), "pg_srs_lagrange_from_powers")
            return out
        res = np.zeros((1 << log_n, 12), dtype=np.uint64)
        self._ok(self._L.pg_srs_lagrange_from_powers(self._ctx, log_n, pp, m, pdev, res.ctypes.data_as(C.c_void_p), 0), "pg_srs_lagrange_from_powers")
        return res

    def commit_wire_evaluations(self, lagrange, log_n: int | None = None) -> np.ndarray:
        """(4, 12) uint64: the commitments of commit_wire_polynomials, computed from the wire values against a Lagrange-basis SRS."""
        log_n = self.domain_log_size() if log_n is None else log_n
        pp, pdev, n, _keep = self._points(lagrange)
        out = np.zeros((4, 12), dtype=np.uint64)
        self._ok(self._L.pg_commit_wire_evaluations(self._ctx, log_n, pp, n, pdev, out.ctypes.data_as(C.c_void_p)), "pg_commit_wire_evaluations")
        return out

    def g1_op(self, op: int, a, b=None) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 12)
        b = np.ascontiguousarray(b, dtype=np.uint64).reshape(-1, 12) if b is not None else None
        out = np.zeros_like(a)
        self._ok(self._L.pg_g1_op(self._ctx, op, a.shape[0], a.ctypes.data_as(C.c_void_p),
                                  b.ctypes.data_as(C.c_void_p) if b is not None else None, out.ctypes.data_as(C.c_void_p)), "pg_g1_op")
        return out

    # -- wire format: canonical little-endian bytes <-> Montgomery limbs (BlsScalar::to_bytes / from_bytes)
    def to_bytes(self, scalars) -> np.ndarray:
        a = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)
        out = np.empty((a.shape[0], 32), dtype=np.uint8)
        self._ok(self._L.pg_fr_to_bytes(self._ctx, a.shape[0], a.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), 0), "pg_fr_to_bytes")
        return out

    def from_bytes(self, raw):
        """(n,32) uint8 -> ((n,4) uint64 Montgomery limbs, number of rejected encodings >= q, index of the first one or None)."""
        r = np.ascontiguousarray(raw, dtype=np.uint8).reshape(-1, 32)
        out = np.empty((r.shape[0], 4), dtype=np.uint64)
        bad, first = C.c_uint64(), C.c_uint64()
        self._ok(self._L.pg_fr_from_bytes(self._ctx, r.shape[0], r.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), 0,
                                          C.byref(bad), C.byref(first)), "pg_fr_from_bytes")
        return out, bad.value, (None if first.value == UINT64_MAX else first.value)

    # -- measurement helpers
    def synth(self, seed: int, stream: int, kind: int, bits: int, dst) -> None:
        p, dev, n, _ = _scalars(dst)
        if not dev:
            raise ValueError("synth writes to device memory")
        self._ok(self._L.pg_synth(self._ctx, seed, stream, n, kind, bits, p), "pg_synth")

    def timing(self, reset: bool = True) -> dict:
        t = _lib.pg_timing()
        self._ok(self._L.pg_get_timing(self._ctx, C.byref(t), int(reset)), "pg_get_timing")
        return {k: getattr(t, k) for k, _ in _lib.pg_timing._fields_}

    CHECK_KINDS = ("instance_generic", "instance_terms", "program", "rowpar", "gates", "fused")

    def check_stats(self, reset: bool = True) -> dict:
        """{kind: (launches, rows)} of the gate-check kernels since the last reset (pg_get_check_stats)."""
        st = _lib.pg_check_stats()
        self._ok(self._L.pg_get_check_stats(self._ctx, C.byref(st), int(reset)), "pg_get_check_stats")
        return {k: (int(st.launches[i]), int(st.rows[i])) for i, k in enumerate(self.CHECK_KINDS)}

    def measure_imad_peak(self):
        w, l = C.c_double(), C.c_double()
        self._ok(self._L.pg_measure_imad_peak(self._ctx, C.byref(w), C.byref(l)), "pg_measure_imad_peak")
        return w.value, l.value

    MICROBENCH_MODES = ("imad_lo", "imad_wide_mul", "imad_wide_acc", "imad_hi", "carry_chain_product", "iadd3", "fr_mul", "fr_mul_cios", "fr_add", "dfma", "imad_wide_plus_dfma_interleaved")

    def microbench(self, mode: int) -> float:
        v = C.c_double()
        self._ok(self._L.pg_microbench(self._ctx, mode, C.byref(v)), "pg_microbench")
        return v.value

    def fr_op(self, op: int, a, b=None) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint64)
        b = np.ascontiguousarray(b, dtype=np.uint64) if b is not None else None
        out = np.empty_like(a)
        self._ok(self._L.pg_fr_op(self._ctx, op, a.shape[0], a.ctypes.data_as(C.c_void_p),
                                  b.ctypes.data_as(C.c_void_p) if b is not None else None, out.ctypes.data_as(C.c_void_p)), "pg_fr_op")
        return out


# ---------------------------------------------------------------------------------------------------- RangeGadgets
def _var(x) -> Variables:
    return x.var if isinstance(x, AllocatedScalar) else x


def range_check(composer: StandardComposer, min_range, max_range, witness) -> Variables:
    """/root/reference/src/range.rs:27-43.  Bounds: one scalar (uniform) or n scalars of one bit width."""
    w = _var(witness)
    pmn, dev, n1, k1 = _scalars(min_range)
    pmx, dev2, n2, k2 = _scalars(max_range)
    if dev != dev2 or n1 != n2:
        raise ValueError("min_range and max_range must have the same length and residency")
    composer._keep += [k1, k2]
    out, k = C.c_uint64(), C.c_uint64()
    composer._ok(composer._L.pg_range_check_batch(composer._ctx, pmn, pmx, n1, dev, w.col, C.byref(out), C.byref(k)), "pg_range_check_batch")
    return Variables(composer, out.value, w.n)


def max_bound(composer: StandardComposer, max_range, witness):
    """/root/reference/src/range.rs:82-113 -> (Variables, num_bits)."""
    w = _var(witness)
    pmx, dev, n1, k1 = _scalars(max_range)
    composer._keep.append(k1)
    out, k = C.c_uint64(), C.c_uint64()
    composer._ok(composer._L.pg_max_bound_batch(composer._ctx, pmx, n1, dev, w.col, C.byref(out), C.byref(k)), "pg_max_bound_batch")
    return Variables(composer, out.value, w.n), k.value


# ---------------------------------------------------------------------------------------------------- ScalarGadgets
def conditionally_select_zero(composer: StandardComposer, x: Variables, select: Variables) -> Variables:
    """/root/reference/src/scalar.rs:21-27."""
    out = C.c_uint64()
    composer._ok(composer._L.pg_select_zero_batch(composer._ctx, _var(x).col, _var(select).col, C.byref(out)), "pg_select_zero_batch")
    return Variables(composer, out.value, _var(x).n)


def conditionally_select_one(composer: StandardComposer, y: Variables, selector: Variables) -> Variables:
    """/root/reference/src/scalar.rs:36-59."""
    out = C.c_uint64()
    composer._ok(composer._L.pg_select_one_batch(composer._ctx, _var(y).col, _var(selector).col, C.byref(out)), "pg_select_one_batch")
    return Variables(composer, out.value, _var(y).n)


def is_non_zero(composer: StandardComposer, var: Variables, value_assigned) -> None:
    """/root/reference/src/scalar.rs:63-97.  Raises NonExistingInverse like `is_non_zero(..)?` in a loop would."""
    p, dev, n, keep = _scalars(value_assigned)
    if n != _var(var).n:
        raise ValueError("value_assigned must have one scalar per variable")
    composer._keep.append(keep)
    n_err, first = C.c_uint64(), C.c_uint64()
    rc = composer._ok(composer._L.pg_is_non_zero_batch(composer._ctx, _var(var).col, p, dev, C.byref(n_err), C.byref(first)), "pg_is_non_zero_batch")
    if rc == 1:
        raise NonExistingInverse(n_err.value, first.value)


NZ_UNIFORM, NZ_REFERENCE = 0, 1


def is_non_zero_flags(composer: StandardComposer, var: Variables, value_assigned, layout: int = NZ_UNIFORM, flags_out=None) -> np.ndarray:
    """``[is_non_zero(composer, var_i, value_assigned_i).is_err() for i in range(n)]`` -- /root/reference/src/scalar.rs:63-97 with
    every Result kept: the batch does not stop at a zero.  Returns the (n,) uint8 error flags (or fills the CUDA tensor `flags_out`
    when value_assigned lives on the device).  layout NZ_UNIFORM: 3 variables + 3 rows for every instance (errored ones hold
    inv = 0 and fail their last row); NZ_REFERENCE: errored instances leave 1 variable + 1 row like the reference call does."""
    p, dev, n, keep = _scalars(value_assigned)
    if n != _var(var).n:
        raise ValueError("value_assigned must have one scalar per variable")
    composer._keep.append(keep)
    n_err = C.c_uint64()
    if dev:
        fp = C.c_void_p(flags_out.data_ptr()) if flags_out is not None else None
        flags = flags_out
    else:
        flags = np.zeros(n, dtype=np.uint8)
        fp = flags.ctypes.data_as(C.c_void_p)
    composer._ok(composer._L.pg_is_non_zero_batch_flags(composer._ctx, _var(var).col, p, dev, fp, int(layout), C.byref(n_err)), "pg_is_non_zero_batch_flags")
    composer.last_n_err = n_err.value
    return flags


def maybe_equal(composer: StandardComposer, a, b) -> Variables:
    """/root/reference/src/scalar.rs:105-140."""
    out = C.c_uint64()
    composer._ok(composer._L.pg_maybe_equal_batch(composer._ctx, _var(a).col, _var(b).col, C.byref(out)), "pg_maybe_equal_batch")
    return Variables(composer, out.value, _var(a).n)
