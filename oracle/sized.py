"""ctypes binding of the CPU oracle of CosineCM with a CountMinSketchConfig (oracle/sized_oracle.c).

TEST INFRASTRUCTURE ONLY (tests/ and tools/ parity legs) -- never imported from mahout_b200/.  The library is built
from sized_oracle.c against libmahout_oracle.so, whose per-sketch primitives it calls.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from . import _HERE, _SO, _c, _p, max_threads
from . import build as _build_main

_SRC = os.path.join(_HERE, "sized_oracle.c")
_lib = None


def _cc() -> str:
    # the system gcc: the image's CC wrapper lacks libgomp.spec (see oracle/Makefile)
    return "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else (shutil.which("gcc") or "gcc")


def build() -> str:
    """libsized_oracle.so next to libmahout_oracle.so (a temporary directory when the tree is read-only)"""
    main = _build_main()
    out = os.path.join(_HERE, "libsized_oracle.so")
    if not os.access(_HERE, os.W_OK):
        out = os.path.join(tempfile.gettempdir(), f"libsized_oracle_{os.getuid()}.so")
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(_SRC), os.path.getmtime(main)):
        tmp = f"{out}.{os.getpid()}.tmp"
        where = os.path.dirname(os.path.abspath(main))
        rpath = "$ORIGIN" if os.path.dirname(out) == where else where
        subprocess.check_call([_cc(), "-O2", "-fPIC", "-fopenmp", "-Wall", "-Wextra", "-std=c11", "-shared", "-o", tmp,
                               _SRC, "-L", where, "-l:libmahout_oracle.so", f"-Wl,-rpath,{rpath}", "-lm"])
        os.replace(tmp, out)
    return out


def lib():
    global _lib
    if _lib is None:
        C.CDLL(_SO, mode=C.RTLD_GLOBAL)   # the primitives, shared with oracle.lib()
        L = C.CDLL(build())
        i64, i32, f64, P = C.c_int64, C.c_int32, C.c_double, C.c_void_p
        L.orc_sized_neighborhood.argtypes = [i64, P, P, P, P, P, P, P, P, i64, C.c_int, f64, C.c_int, P, P, P]
        L.orc_sized_estimate.argtypes = [i64, P, P, P, P, P, P, P, P, P, P, i32, P, P, P, i64, C.c_int, P]
        _lib = L
    return _lib


def _model(width, depth, user_ptr, item, pref):
    return (_c(width, np.int32), _c(depth, np.int32), _c(user_ptr, np.int64), _c(item, np.int64),
            _c(np.asarray(pref, np.float32), np.float64))


def sized_neighborhood(width, depth, a, b, user_ptr, item, pref, queries, n, min_similarity=-np.inf,
                       nthreads=None):
    """NearestNUserNeighborhood over CosineCM.userSimilarity with per-user sketch shapes (CountMinSketchConfig):
    (idx [q, n], sim [q, n], cnt [q]); unused slots -1 / 0.  pref: the float prefs, widened to double."""
    w, d, ptr, it, pr = _model(width, depth, user_ptr, item, pref)
    queries = _c(queries, np.int64)
    a, b = _c(a, np.int64), _c(b, np.int64)
    nthreads = max_threads() if nthreads is None else nthreads
    q = queries.shape[0]
    idx = np.zeros((q, n), np.int64)
    sim = np.zeros((q, n), np.float64)
    cnt = np.zeros(q, np.int32)
    lib().orc_sized_neighborhood(w.shape[0], _p(w), _p(d), _p(a), _p(b), _p(ptr), _p(it), _p(pr), _p(queries), q,
                                 int(n), float(min_similarity), nthreads, _p(idx), _p(sim), _p(cnt))
    return idx, sim, cnt


def sized_estimate(width, depth, a, b, user_ptr, item, pref, nb_idx, nb_sim, nb_cnt, user, item_id, nb_row=None,
                   nthreads=None):
    """doEstimatePreference with each neighbour's own sketch (getExportedCMProfile): float32 [q], NaN = none."""
    w, d, ptr, it, pr = _model(width, depth, user_ptr, item, pref)
    nb_idx, nb_sim, nb_cnt = _c(nb_idx, np.int64), _c(nb_sim, np.float64), _c(nb_cnt, np.int32)
    user, item_id = _c(user, np.int64), _c(item_id, np.int64)
    nb_row = _c(nb_row, np.int64) if nb_row is not None else None
    a, b = _c(a, np.int64), _c(b, np.int64)
    nthreads = max_threads() if nthreads is None else nthreads
    out = np.zeros(user.shape[0], np.float32)
    lib().orc_sized_estimate(w.shape[0], _p(w), _p(d), _p(a), _p(b), _p(ptr), _p(it), _p(pr), _p(nb_idx), _p(nb_sim),
                             _p(nb_cnt), int(nb_idx.shape[1]), _p(user), _p(nb_row), _p(item_id), user.shape[0],
                             nthreads, _p(out))
    return out
