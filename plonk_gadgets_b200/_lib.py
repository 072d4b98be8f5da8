"""Loader/builder of the CUDA shared library behind the C ABI (include/pg_b200.h).

There is no CPU fallback: if ``libpg_b200.so`` is missing or cannot be loaded this module raises, and every entry point
of the library itself fails with PG_ERR_NO_DEVICE when no sm_100a GPU is present.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpg_b200.so")
CSRC = os.path.join(_HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


class pg_fr(C.Structure):
    _fields_ = [("l", C.c_uint64 * 4)]


class pg_cfg(C.Structure):
    _fields_ = [("device", C.c_int32), ("check_mode", C.c_int32), ("flags", C.c_uint32), ("check_shape", C.c_uint32),
                ("stream", C.c_void_p)]


class pg_timing(C.Structure):
    _fields_ = [("check_ms", C.c_double), ("witness_ms", C.c_double), ("other_ms", C.c_double),
                ("check_launches", C.c_uint64), ("witness_launches", C.c_uint64), ("other_launches", C.c_uint64),
                ("check_rows", C.c_uint64)]


class pg_op(C.Structure):
    _fields_ = [("gadget", C.c_uint32), ("num_bits", C.c_uint32), ("n", C.c_uint64), ("group", C.c_uint32), ("reserved", C.c_uint32)]


class pg_op_shard(C.Structure):
    _fields_ = [("inst_lo", C.c_uint64), ("inst_hi", C.c_uint64), ("row_base", C.c_uint64), ("var_base", C.c_uint64)]


class pg_check_stats(C.Structure):
    _fields_ = [("launches", C.c_uint64 * 8), ("rows", C.c_uint64 * 8)]


ABI_VERSION = 7

# every symbol include/pg_b200.h declares: name -> (restype, argtypes)
_vp, _u64, _i32, _u32 = C.c_void_p, C.c_uint64, C.c_int, C.c_uint32
_pu64 = C.POINTER(C.c_uint64)
SIGNATURES = {
    "pg_abi_version": (_i32, []),
    "pg_strerror": (C.c_char_p, [_i32]),
    "pg_last_error": (C.c_char_p, [_vp]),
    "pg_ctx_create": (_i32, [C.POINTER(pg_cfg), C.POINTER(_vp)]),
    "pg_ctx_destroy": (None, [_vp]),
    "pg_composer_reset": (_i32, [_vp]),
    "pg_sync": (_i32, [_vp]),
    "pg_add_input_batch": (_i32, [_vp, _u64, _vp, _i32, _pu64]),
    "pg_range_check_batch": (_i32, [_vp, _vp, _vp, _u64, _i32, _u64, _pu64, _pu64]),
    "pg_max_bound_batch": (_i32, [_vp, _vp, _u64, _i32, _u64, _pu64, _pu64]),
    "pg_maybe_equal_batch": (_i32, [_vp, _u64, _u64, _pu64]),
    "pg_is_non_zero_batch": (_i32, [_vp, _u64, _vp, _i32, _pu64, _pu64]),
    "pg_is_non_zero_batch_flags": (_i32, [_vp, _u64, _vp, _i32, _vp, _i32, _pu64]),
    "pg_select_zero_batch": (_i32, [_vp, _u64, _u64, _pu64]),
    "pg_select_one_batch": (_i32, [_vp, _u64, _u64, _pu64]),
    "pg_constrain_to_constant_batch": (_i32, [_vp, _u64, _vp, _u64, _vp, _u64, _i32]),
    "pg_range_gate_batch": (_i32, [_vp, _u64, _u32]),
    "pg_check": (_i32, [_vp, _pu64, _pu64]),
    "pg_check_rows": (_i32, [_vp, _u64, _vp, _vp, _vp, _i32, _pu64, _pu64]),
    "pg_check_rows_ex": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp, _vp, _i32, _pu64, _pu64]),
    "pg_template_get": (_i32, [_u32, _u32, _vp, _vp, _pu64, _pu64, _vp, _vp, _vp]),
    "pg_op_shape": (_i32, [_u32, _u32, _pu64, _pu64]),
    "pg_shard_plan": (_i32, [C.POINTER(pg_op), _u64, _u32, _i32, C.POINTER(pg_op_shard)]),
    "pg_comm_unique_id": (_i32, [_vp]),
    "pg_comm_init": (_i32, [_vp, _vp, _u32, _u32]),
    "pg_comm_destroy": (_i32, [_vp]),
    "pg_check_sharded": (_i32, [_vp, C.POINTER(pg_op_shard), _u64, _pu64, _pu64, _pu64]),
    "pg_gather_column": (_i32, [_vp, _u64, _vp, _u64, _i32, _pu64, _pu64]),
    "pg_gather_variables": (_i32, [_vp, _u64, _vp, _u64, _i32, _pu64]),
    "pg_poke_variable": (_i32, [_vp, _u64, _vp]),
    "pg_counts": (_i32, [_vp, _pu64, _pu64]),
    "pg_col_info": (_i32, [_vp, _u64, _pu64, _pu64, _pu64]),
    "pg_col_read": (_i32, [_vp, _u64, _u64, _u64, _vp, _i32]),
    "pg_read_variables": (_i32, [_vp, _u64, _u64, _vp, _i32]),
    "pg_materialize_rows": (_i32, [_vp, _u64, _u64, _vp, _vp, _vp, _vp, _i32]),
    "pg_materialize_gate_selectors": (_i32, [_vp, _u64, _u64, _vp, _vp, _i32]),
    "pg_permutation": (_i32, [_vp, _u64, _u64, _vp, _i32]),
    "pg_export_composer": (_i32, [_vp, C.c_char_p, _u64, _u32]),
    "pg_fft": (_i32, [_vp, _u32, _i32, _vp, _vp, _i32]),
    "pg_wire_polynomials": (_i32, [_vp, _u32, _vp, _i32]),
    "pg_sigma_polynomials": (_i32, [_vp, _u32, _i32, _vp, _i32]),
    "pg_permutation_z": (_i32, [_vp, _u32, _vp, _vp, _i32, _vp, _i32, _vp]),
    "pg_permutation_z_rows": (_i32, [_vp, _u32, _u64, _vp, _vp, _i32, _vp, _vp, _i32, _vp, _i32, _vp]),
    "pg_selector_polynomials": (_i32, [_vp, _u32, _i32, _vp, _i32]),
    "pg_public_input_polynomial": (_i32, [_vp, _u32, _i32, _vp, _i32]),
    "pg_quotient": (_i32, [_vp, _u32, _vp, _vp, _vp, _vp, _vp, _i32]),
    "pg_prover_openings": (_i32, [_vp, _u32, _vp, _vp, _i32, _vp, _vp, _i32]),
    "pg_msm": (_i32, [_vp, _u64, _vp, _vp, _vp, _i32]),
    "pg_srs_powers": (_i32, [_vp, _vp, _vp, _u64, _vp, _i32]),
    "pg_g1_fixed_base_mul": (_i32, [_vp, _u64, _vp, _vp, _vp, _i32]),
    "pg_commit_wire_polynomials": (_i32, [_vp, _u32, _vp, _u64, _i32, _vp]),
    "pg_srs_lagrange": (_i32, [_vp, _vp, _vp, _u32, _vp, _i32]),
    "pg_srs_lagrange_from_powers": (_i32, [_vp, _u32, _vp, _u64, _i32, _vp, _i32]),
    "pg_commit_wire_evaluations": (_i32, [_vp, _u32, _vp, _u64, _i32, _vp]),
    "pg_g1_op": (_i32, [_vp, _i32, _u64, _vp, _vp, _vp]),
    "pg_fr_to_bytes": (_i32, [_vp, _u64, _vp, _vp, _i32]),
    "pg_fr_from_bytes": (_i32, [_vp, _u64, _vp, _vp, _i32, _pu64, _pu64]),
    "pg_synth": (_i32, [_vp, _u64, _u64, _u64, _i32, _u32, _vp]),
    "pg_get_timing": (_i32, [_vp, C.POINTER(pg_timing), _i32]),
    "pg_get_check_stats": (_i32, [_vp, C.POINTER(pg_check_stats), _i32]),
    "pg_measure_imad_peak": (_i32, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "pg_microbench": (_i32, [_vp, _i32, C.POINTER(C.c_double)]),
    "pg_fr_op": (_i32, [_vp, _i32, _u64, _vp, _vp, _vp]),
}


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile plonk_gadgets_b200/csrc/engine.cu for sm_100a into libpg_b200.so (in-tree).  nvcc cross-compiles without a GPU."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "pg_b200.h")]
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in srcs):
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libpg_b200.so")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH, os.path.join(CSRC, "engine.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


def bind(cdll):
    """Attach the header's signatures to a loaded library; raises AttributeError if a declared symbol is missing."""
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(cdll, name)
        fn.restype, fn.argtypes = res, args
    return cdll


_cdll = None


def load():
    """The CUDA library.  Raises if it has not been built -- there is nothing to fall back to."""
    global _cdll
    if _cdll is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(plonk_gadgets_b200 has no CPU fallback)")
        _cdll = bind(C.CDLL(LIB_PATH))
        if _cdll.pg_abi_version() != ABI_VERSION:
            raise RuntimeError("libpg_b200.so ABI version mismatch")
    return _cdll
