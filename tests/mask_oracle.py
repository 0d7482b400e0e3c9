"""Exposed-point masks of the CPU oracle (tests/mask_oracle.c over the neighbour lists of oracle/sasa_oracle.c): what the GPU
masks are compared with bit for bit.  The C file is compiled once per process into a temporary directory (removed at exit),
with the oracle's strict floating-point flags, so the source tree may be read-only."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def _load():
    global _LIB
    if _LIB is None:
        d = tempfile.mkdtemp(prefix="sasa_mask_oracle_")
        atexit.register(shutil.rmtree, d, True)
        path = os.path.join(d, "libmask_oracle.so")
        subprocess.run(["/usr/bin/gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-fopenmp",
                        "-o", path, os.path.join(_HERE, "mask_oracle.c"), "-lm"], check=True)
        L = C.CDLL(path)
        vp = C.c_void_p
        L.mask_oracle_exposed.argtypes = [vp, vp, C.c_size_t, C.c_float, C.c_size_t, C.c_int, vp, vp, vp, vp, vp, vp, vp]
        L.mask_oracle_exposed.restype = None
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data


def exposed_masks(oracle, xyzr, probe=1.4, n_points=100, lanes=8, ids=None) -> np.ndarray:
    """(n, ceil(n_points / 32)) uint32: bit p % 32 of word p // 32 of row i set when point p of atom i is exposed, decided
    with the arithmetic of the oracle's calculate_sasa_internal on the oracle's neighbour lists (same id rule)."""
    assert lanes in (4, 8, 16)
    xyzr = np.ascontiguousarray(xyzr, dtype=np.float32).reshape(-1, 4)
    n = xyzr.shape[0]
    out = np.zeros((n, (n_points + 31) // 32), np.uint32)
    if n == 0:
        return out
    ids = None if ids is None else np.ascontiguousarray(ids, dtype=np.uint64)
    # the neighbour build of calculate_sasa_internal: max radius folded from 0, cell size probe + max radius (both f32)
    max_r = np.float32(max(0.0, float(xyzr[:, 3].max())))
    cell = float(np.float32(probe) + max_r)
    P = lambda a, ty: None if a is None else a.ctypes.data_as(C.POINTER(ty))   # noqa: E731
    off = np.zeros(n + 1, np.uint32)
    total = oracle.lib.oracle_neighbor_lists(P(xyzr, C.c_float), P(ids, C.c_uint64), n, probe, float(max_r), cell,
                                             P(off, C.c_uint32), None, None)
    if total < 0:
        raise ValueError(f"oracle: non-finite or invalid input (rc={total})")
    idx = np.zeros(max(total, 1), np.uint32)
    thr = np.zeros(max(total, 1), np.float32)
    oracle.lib.oracle_neighbor_lists(P(xyzr, C.c_float), P(ids, C.c_uint64), n, probe, float(max_r), cell, P(off, C.c_uint32),
                                     P(idx, C.c_uint32), P(thr, C.c_float))
    sphere = np.ascontiguousarray(oracle.sphere_points(n_points).T)   # (3, n_points) f32: x, y, z
    _load().mask_oracle_exposed(_p(xyzr), _p(ids), n, probe, n_points, lanes, _p(sphere[0]), _p(sphere[1]), _p(sphere[2]),
                                _p(off), _p(idx), _p(thr), _p(out))
    return out
