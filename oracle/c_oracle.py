"""ORACLE / TEST INFRASTRUCTURE ONLY.  ctypes binding of oracle/schur_pairs.c (plain-C restatement of the sparse Schur
assembly, /root/reference/src/makeBBBB.jl:39-64,139-213) -- built by `make -C oracle` (also run by __graft_entry__.build())."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def build():
    """path of liboracle.so compiled on this host: oracle/_build/, or, when the checkout is read-only, a private directory
    of this process (tempfile.mkdtemp: mode 0700, unpredictable name, removed at exit)"""
    # -march=native code must be rebuilt on the machine that runs it (the build machine may have another CPU than the GPU host)
    host = os.uname().nodename + ":" + (open("/proc/cpuinfo").read().split("model name")[1].split("\n")[0] if os.path.exists("/proc/cpuinfo") else "")
    d = os.path.join(_HERE, "_build")
    so, stamp = os.path.join(d, "liboracle.so"), os.path.join(d, "host")
    if os.path.exists(so) and os.path.exists(stamp) and open(stamp).read() == host and \
            os.path.getmtime(so) >= os.path.getmtime(os.path.join(_HERE, "schur_pairs.c")):
        return so
    if not os.access(d if os.path.isdir(d) else _HERE, os.W_OK):
        d = tempfile.mkdtemp(prefix="liboracle_")
        atexit.register(shutil.rmtree, d, True)
        so, stamp = os.path.join(d, "liboracle.so"), os.path.join(d, "host")
    subprocess.run(["make", "-C", _HERE, "-B", f"O={d}", so], check=True, capture_output=True)
    with open(stamp, "w") as f:
        f.write(host)
    return so


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.lrn_oracle_schur_pairs.restype = None
        L.lrn_oracle_schur_pairs.argtypes = [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64]
        L.lrn_oracle_max_threads.restype = C.c_int32
        _lib = L
    return _lib


def entry_lists(AAi, m):
    """constraint-major entry lists of AA_i (n_var x m^2 scipy sparse, row k = vec(calA_k)): rowptr, p, q, v"""
    A = AAi.tocsr()
    A.sort_indices()
    rowptr = A.indptr.astype(np.int64)
    ep = (A.indices % m).astype(np.int32)
    eq = (A.indices // m).astype(np.int32)
    ev = np.ascontiguousarray(A.data, dtype=np.float64)
    return rowptr, ep, eq, ev


def schur_pairs_lower(AAi, m, W, H=None, accumulate=False, nthreads=0, cols=None):
    """lower triangle of H_i[j,k] = tr(calA_j W calA_k W) into the Fortran-ordered n x n array H (allocated if None);
    cols = (k0, k1): only that column panel, returned as an n x (k1 - k0) array (entries above the diagonal stay zero)"""
    n = AAi.shape[0]
    rowptr, ep, eq, ev = entry_lists(AAi, m)
    Wf = np.asfortranarray(W, dtype=np.float64)
    k0, k1 = (0, 0) if cols is None else (int(cols[0]), int(cols[1]))
    if H is None:
        H = np.zeros((n, n if cols is None else k1 - k0), order="F")
    assert H.flags.f_contiguous and H.dtype == np.float64
    lib().lrn_oracle_schur_pairs(n, m, rowptr.ctypes.data, ep.ctypes.data, eq.ctypes.data, ev.ctypes.data, Wf.ctypes.data,
                                 H.ctypes.data, H.shape[0], 1 if accumulate else 0, int(nthreads), k0, k1)
    return H


def max_threads():
    return int(lib().lrn_oracle_max_threads())
