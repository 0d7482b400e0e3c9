"""ctypes binding of the C ABI in include/sasa_b200.h.

The library is loaded from rustsasa_b200/libsasa_b200.so (built in-tree by rustsasa_b200/build.py).
There is no fallback of any kind: a missing library raises ImportError-like RuntimeError at first
use, and a missing CUDA device makes ``sasa_b200_create`` fail.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SASA_B200_LIB") or os.path.join(HERE, "libsasa_b200.so")   # env override: another build of the library

OK, ERR_INVALID_ARGUMENT, ERR_CUDA, ERR_OUT_OF_MEMORY, ERR_NON_FINITE, ERR_UNSUPPORTED = range(6)
FLAG_BOUNDARY_STATS = 1
FLAG_FORCE_STREAMING = 2

EXPORTS = [
    "sasa_b200_abi_version", "sasa_b200_create", "sasa_b200_destroy", "sasa_b200_last_error",
    "sasa_b200_alloc_pinned", "sasa_b200_free_pinned", "sasa_b200_sphere_points",
    "sasa_b200_calculate_sasa_internal", "sasa_b200_batch_create", "sasa_b200_batch_destroy",
    "sasa_b200_batch_run_host", "sasa_b200_batch_run_device", "sasa_b200_batch_sync",
    "sasa_b200_batch_run_frames_host", "sasa_b200_run_batch", "sasa_b200_batch_run_atom_range_device",
    "sasa_b200_batch_run_atom_range_host", "sasa_b200_batch_reduce_device",
    "sasa_b200_batch_submit_host", "sasa_b200_batch_submit_frames_host", "sasa_b200_job_wait",
    "sasa_b200_device_count", "sasa_b200_batch_run_indexed_host", "sasa_b200_batch_submit_indexed_host",
    "sasa_b200_batch_run_atom_range_peers_device", "sasa_b200_batch_run_groups_host", "sasa_b200_batch_run_groups_device",
    "sasa_b200_batch_run_masks_host", "sasa_b200_batch_run_masks_device", "sasa_b200_batch_run_groups_masks_host",
    "sasa_b200_batch_run_groups_masks_device", "sasa_b200_batch_run_groups_frames_host", "sasa_b200_batch_submit_groups_frames_host",
    "sasa_b200_batch_run_group_pairs_host", "sasa_b200_batch_run_group_pairs_device",
    "sasa_b200_batch_run_group_pairs_frames_host", "sasa_b200_batch_submit_group_pairs_frames_host",
]


class Params(C.Structure):
    _fields_ = [("probe_radius", C.c_float), ("n_points", C.c_uint32), ("simd_lanes", C.c_uint32),
                ("threads", C.c_int32), ("flags", C.c_uint32)]


class Outputs(C.Structure):
    _fields_ = [("counts", C.c_void_p), ("atom_sasa", C.c_void_p), ("seg_sasa", C.c_void_p),
                ("protein", C.c_void_p)]


class PairOutputs(C.Structure):
    _fields_ = [("max_partners", C.c_uint32), ("partner", C.c_void_p), ("buried_counts", C.c_void_p),
                ("buried_area", C.c_void_p), ("partners_needed", C.c_void_p)]


class PairSums(C.Structure):
    _fields_ = [("n_labels", C.c_uint32), ("pair_area", C.c_void_p), ("seg_pair_area", C.c_void_p)]


class Stats(C.Structure):
    _fields_ = [("n_atoms", C.c_uint64), ("n_structures", C.c_uint64), ("boundary_points", C.c_uint64),
                ("neighbor_pairs", C.c_uint64), ("streamed_atoms", C.c_uint64),
                ("h2d_ms", C.c_float), ("kernel_ms", C.c_float), ("d2h_ms", C.c_float), ("total_ms", C.c_float),
                ("gpu_launches", C.c_uint32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m rustsasa_b200.build` (nvcc, sm_100a). "
            "rustsasa_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, sz = C.c_void_p, C.c_size_t
    L.sasa_b200_abi_version.restype = C.c_int
    L.sasa_b200_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.sasa_b200_device_count.argtypes = [C.POINTER(C.c_int)]
    L.sasa_b200_destroy.argtypes = [vp]
    L.sasa_b200_destroy.restype = None
    L.sasa_b200_last_error.argtypes = [vp]
    L.sasa_b200_last_error.restype = C.c_char_p
    L.sasa_b200_alloc_pinned.argtypes = [sz, C.POINTER(vp)]
    L.sasa_b200_free_pinned.argtypes = [vp]
    L.sasa_b200_sphere_points.argtypes = [C.c_uint32, vp]
    L.sasa_b200_calculate_sasa_internal.argtypes = [vp, vp, vp, sz, C.c_float, sz, C.c_ssize_t, vp, vp]
    L.sasa_b200_batch_create.argtypes = [vp, vp, sz, vp, vp, vp, C.POINTER(vp)]
    L.sasa_b200_batch_destroy.argtypes = [vp]
    L.sasa_b200_batch_destroy.restype = None
    L.sasa_b200_batch_run_host.argtypes = [vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(Stats)]
    L.sasa_b200_batch_run_device.argtypes = [vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), vp]
    L.sasa_b200_batch_sync.argtypes = [vp, C.POINTER(Stats)]
    L.sasa_b200_batch_run_groups_host.argtypes = [vp, vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(Outputs),
                                                  C.POINTER(Stats)]
    L.sasa_b200_batch_run_groups_device.argtypes = [vp, vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(Outputs), vp]
    L.sasa_b200_batch_run_masks_host.argtypes = [vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), vp, C.POINTER(Stats)]
    L.sasa_b200_batch_run_masks_device.argtypes = [vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), vp, vp]
    L.sasa_b200_batch_run_groups_masks_host.argtypes = [vp, vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(Outputs),
                                                        vp, vp, C.POINTER(Stats)]
    L.sasa_b200_batch_run_groups_masks_device.argtypes = [vp, vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(Outputs),
                                                          vp, vp, vp]
    L.sasa_b200_batch_run_groups_frames_host.argtypes = [vp, vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(Outputs),
                                                         C.POINTER(Stats)]
    L.sasa_b200_batch_submit_groups_frames_host.argtypes = [vp, vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(Outputs),
                                                            C.POINTER(vp)]
    L.sasa_b200_batch_run_group_pairs_host.argtypes = [vp, vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(Outputs),
                                                       C.POINTER(PairOutputs), C.POINTER(Stats)]
    L.sasa_b200_batch_run_group_pairs_device.argtypes = [vp, vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(Outputs),
                                                         C.POINTER(PairOutputs), vp]
    L.sasa_b200_batch_run_group_pairs_frames_host.argtypes = [vp, vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs),
                                                              C.POINTER(Outputs), C.POINTER(PairSums), C.POINTER(Stats)]
    L.sasa_b200_batch_submit_group_pairs_frames_host.argtypes = [vp, vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs),
                                                                 C.POINTER(Outputs), C.POINTER(PairSums), C.POINTER(vp)]
    L.sasa_b200_batch_submit_host.argtypes = [vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(vp)]
    L.sasa_b200_batch_submit_frames_host.argtypes = [vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(vp)]
    L.sasa_b200_job_wait.argtypes = [vp, C.POINTER(Stats)]
    L.sasa_b200_batch_run_indexed_host.argtypes = [vp, vp, vp, vp, sz, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(Stats)]
    L.sasa_b200_batch_submit_indexed_host.argtypes = [vp, vp, vp, vp, sz, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(vp)]
    L.sasa_b200_batch_run_frames_host.argtypes = [vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs), C.POINTER(Stats)]
    L.sasa_b200_batch_run_atom_range_device.argtypes = [vp, vp, vp, C.POINTER(Params), C.c_uint32, C.c_uint32, vp, vp, vp]
    L.sasa_b200_batch_run_atom_range_host.argtypes = [vp, vp, vp, C.POINTER(Params), C.c_uint32, C.c_uint32, vp, vp,
                                                      C.POINTER(Stats)]
    L.sasa_b200_batch_run_atom_range_peers_device.argtypes = [vp, vp, vp, C.POINTER(Params), C.c_uint32, C.c_uint32, vp, vp, vp]
    L.sasa_b200_batch_reduce_device.argtypes = [vp, vp, vp, vp, vp]
    L.sasa_b200_run_batch.argtypes = [vp, vp, vp, vp, sz, vp, vp, vp, C.POINTER(Params), C.POINTER(Outputs),
                                      C.POINTER(Stats)]
    for name in EXPORTS:
        fn = getattr(L, name)
        if fn.restype is C.c_int or name.startswith("sasa_b200_") and fn.restype not in (None, C.c_char_p):
            fn.restype = C.c_int
    _lib = L
    return L
