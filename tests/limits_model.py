"""TEST INFRASTRUCTURE ONLY: scalar replay of the placement search with per-type platform limits
(sls_multi_kernel<false, false, true>, timberborn_support_solver_b200/csrc/sls_multi.cu) for the tests.  tests/limits_model.cpp
includes the oracle's model of the placement search and restates its step loop with the class counters; it is compiled on first
use into a per-user temporary directory (the repository tree is never written)."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "limits_model.cpp")
_ORACLE = os.path.join(_HERE, "..", "oracle", "slsm_model.cpp")
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for src in (_SRC, _ORACLE):
            with open(src, "rb") as f:
                h.update(f.read())
        out_dir = os.path.join(tempfile.gettempdir(), f"tss_limits_model_{os.getuid()}")
        so = os.path.join(out_dir, f"limits_model_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            os.makedirs(out_dir, exist_ok=True)
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-Wall", "-shared", "-o", tmp, _SRC])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def _p(a, t=C.c_int):
    return a.ctypes.data_as(C.POINTER(t))


def limits_model(grid, key_dims, costs, key_mask, class_limit, n_chains, epochs, seed=0, chain_offset=0, noise_pct=20, share_bound=True,
                 count_flips=False):
    """oracle.slsm_model with per-type limits: key_mask[k] = classes of key k (bit j = class j), class_limit[j] = at most that
    many platforms in class j.  -> the same dict as oracle.slsm_model (flips_total with count_flips)."""
    g = np.ascontiguousarray(grid, dtype=np.uint8)
    kd = np.ascontiguousarray(key_dims, np.int32).reshape(-1, 2)
    cs = np.ascontiguousarray(costs, np.int32)
    mk = np.ascontiguousarray(key_mask, np.int32).reshape(-1)
    lm = np.ascontiguousarray(class_limit, np.int32).reshape(-1)
    assert len(mk) == len(cs)
    ep = np.ascontiguousarray(epochs, dtype=np.int64).reshape(-1, 3)
    items = np.zeros((n_chains, 1024), np.uint16)
    best_items = np.zeros((n_chains, 1024), np.uint16)
    k, best_k, best = np.zeros(n_chains, np.int32), np.zeros(n_chains, np.int32), np.zeros(n_chains, np.int32)
    step = np.zeros(n_chains, np.uint32)
    totals = np.zeros(3, np.uint64)
    rc = lib().limits_model(_p(g, C.c_uint8), g.shape[1], g.shape[0], _p(kd), _p(cs), len(cs), _p(mk), _p(lm), len(lm), n_chains, C.c_uint32(chain_offset),
                            C.c_uint64(seed), noise_pct, _p(ep, C.c_longlong), len(ep), int(share_bound), _p(items, C.c_uint16), _p(k),
                            _p(best_items, C.c_uint16), _p(best_k), _p(best), _p(step, C.c_uint32), _p(totals, C.c_uint64))
    assert rc == 0
    out = dict(items=items, k=k, best_items=best_items, best_k=best_k, best=best, step=step, scored_total=int(totals[0]), steps_total=int(totals[1]))
    if count_flips:
        out["flips_total"] = int(totals[2])
    return out
