"""The Lagrange-basis SRS's test oracles (TEST INFRASTRUCTURE ONLY), for pg_srs_lagrange_from_powers:

  * group_ifft: the C restatement tests/oracle_lagrange/group_fft.c (the textbook serial radix-2 inverse FFT over Jacobian G1 with
    jac_mul twiddles and a final 1/n), built into tests/oracle_lagrange/_build;
  * definition_sum: the big-int definition (1/n) sum_j w^(-ij) P_j over the affine points of oracle/pymodel.py;
  * scalar_ifft: the same transform of scalars -- for P_j = k_j G the result is (ifft k)_i G.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from oracle import pymodel as pm
from tests.programs import Q

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_SRC = os.path.join(HERE, "oracle_lagrange", "group_fft.c")
_SO = os.path.join(HERE, "oracle_lagrange", "_build", "liblagrange_oracle.so")
_lib = None


def _clib():
    global _lib
    if _lib is None:
        deps = [_SRC, os.path.join(ROOT, "oracle", "fr.h"), os.path.join(ROOT, "oracle", "g1.c")]
        if not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
            os.makedirs(os.path.dirname(_SO), exist_ok=True)
            subprocess.run(["gcc", "-O3", "-march=x86-64-v3", "-madx", "-fPIC", "-shared", "-std=gnu11", "-o", _SO, _SRC], check=True)
        _lib = C.CDLL(_SO)
        _lib.lag_group_ifft.restype = None
        _lib.lag_group_ifft.argtypes = [C.c_void_p, C.c_uint, C.c_void_p]
    return _lib


def group_ifft(points13, log_n: int) -> np.ndarray:
    """(2^log_n, 13) oracle points -> (2^log_n, 13): the C restatement over the first 2^log_n points."""
    p = np.ascontiguousarray(points13, dtype=np.uint64).reshape(-1, 13)[: 1 << log_n].copy()
    assert p.shape[0] == 1 << log_n
    out = np.zeros_like(p)
    _clib().lag_group_ifft(p.ctypes.data_as(C.c_void_p), log_n, out.ctypes.data_as(C.c_void_p))
    return out


def _weights(log_n: int):
    n = 1 << log_n
    w_inv, n_inv = pow(pm.group_gen(log_n), -1, Q), pow(n, -1, Q)
    return n, w_inv, n_inv


def scalar_ifft(ks, log_n: int) -> list:
    """(1/n) sum_j w^(-ij) k_j, i < n, over integers mod q."""
    n, w_inv, n_inv = _weights(log_n)
    return [n_inv * sum(k * pow(w_inv, i * j, Q) for j, k in enumerate(ks[:n])) % Q for i in range(n)]


def definition_sum(points, log_n: int) -> list:
    """(1/n) sum_j w^(-ij) P_j, i < n, for affine integer points ((x, y) or None), one scalar multiplication per term."""
    n, w_inv, n_inv = _weights(log_n)
    out = []
    for i in range(n):
        acc = None
        for j, pt in enumerate(points[:n]):
            acc = pm.g1_add(acc, pm.g1_mul(n_inv * pow(w_inv, i * j, Q), pt))
        out.append(acc)
    return out
