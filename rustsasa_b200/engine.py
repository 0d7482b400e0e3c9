"""Thin Python host layer over the C ABI: Engine (a context on one GPU) and Batch (a reusable topology).

numpy arrays are host buffers (pipelined H2D / kernels / D2H inside the library);
torch CUDA tensors are device buffers (``Batch.run_device``, no copies).  Nothing here computes SASA
on the CPU: every numeric result comes out of libsasa_b200.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Any, Optional

import numpy as np

from . import _lib


class SasaB200Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"[sasa_b200 status {code}] {message}")
        self.code = code


class _PinnedBlock:
    """Owns one cudaHostAlloc block and exposes it through the numpy array interface."""

    def __init__(self, L, ptr, nbytes, shape, dtype):
        self._L, self._ptr = L, ptr
        self.__array_interface__ = dict(shape=tuple(int(x) for x in shape), typestr=dtype.str,
                                        data=(ptr, False), version=3)

    def __del__(self):
        try:
            self._L.sasa_b200_free_pinned(self._ptr)
        except Exception:
            pass


def _ptr(a) -> Optional[int]:
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return int(a.data_ptr())   # torch tensor


def _stream(stream) -> int:
    """cudaStream_t handle for the device entry points.  None = torch's CURRENT stream, so that work enqueued here
    is ordered with the caller's other torch / NCCL work (the legacy default stream is passed as cudaStreamLegacy = 1,
    because NULL means "the context's own stream" in the C ABI); an int is passed through as a raw handle."""
    if stream is None:
        import torch
        h = int(torch.cuda.current_stream().cuda_stream)
        return h if h != 0 else 1
    return int(stream)


def index_radii(radii):
    """Palette + one-byte indices of a radius column (the indexed-radius wire format), or None when it holds more than 256
    distinct values."""
    pal, idx = np.unique(np.asarray(radii, np.float32), return_inverse=True)
    if pal.shape[0] > 256:
        return None
    return pal.astype(np.float32), idx.astype(np.uint8)


def _np(a, dtype, shape=None):
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=dtype)
    if shape is not None:
        a = a.reshape(shape)
    return a


@dataclass
class BatchResult:
    counts: Optional[np.ndarray] = None
    atom_sasa: Optional[np.ndarray] = None
    seg_sasa: Optional[np.ndarray] = None
    protein: Optional[np.ndarray] = None   # (S, 3): global, polar, non-polar
    stats: Optional[dict] = None
    exposed: Optional[np.ndarray] = None   # (n_atoms, W) uint32 exposed-point masks (run_masks_host, run_groups_masks_host),
                                           # W = ceil(n_points / 32)


@dataclass
class PairResult:
    """Partner slots of a pairwise buried-area run (``Batch.run_group_pairs_host`` / ``_device``), K = max_partners slots per
    atom in batch order: ``partner`` (N, K) uint32 partner group labels in ascending order, ``buried_counts`` (N, K) uint32 the
    points of the atom open with its group alone that the partner hides, ``buried_area`` (N, K) float32 the reference's area
    expression on that count.  Unused slots hold partner 0xFFFFFFFF, count 0 and area 0; a slot is in use exactly when its count
    is non-zero.  ``needed``: the largest number of partners of an atom (an int; a one-element device tensor for the device
    form)."""
    partner: Any = None
    buried_counts: Any = None
    buried_area: Any = None
    needed: Any = None


@dataclass
class PairSums:
    """Device-side sums of a pairwise buried-area run of MD frames (``Batch.run_group_pairs_frames_host``), labels 0 .. L - 1:
    ``pair_area`` (S, L, L) float64, element [s, g, h] the area of group g that group h buries in frame s, and ``seg_pair_area``
    (n_segments, L) float64, element [q, h] the area of segment q that h buries, or None.  Both are float64 sums of the per-atom
    slot areas in atom order, bit for bit what :func:`group_pair_table` and per-segment sums of the slots give on the host."""
    n_labels: int
    pair_area: Any = None
    seg_pair_area: Any = None


def group_pair_table(partner, buried_area, group, struct_off):
    """Pairwise interface table from the partner slots of a pairwise buried-area run: per structure a list of rows
    ``(g, h, area of g buried by h, area of h buried by g)``, one for each contacting pair of labels g < h, in ascending (g, h)
    order.  A slot counts when its partner label is not 0xFFFFFFFF or its area is positive.  Each area is a float64 sum over
    the per-atom float32 slot areas, added in batch atom order."""
    partner = np.asarray(partner, np.uint32)
    n = partner.shape[0]
    partner = partner.reshape(n, -1)
    area = np.asarray(buried_area, np.float32).reshape(n, -1)
    group = np.asarray(group, np.uint32).reshape(-1)
    off = np.asarray(struct_off, np.int64).reshape(-1)
    S = off.shape[0] - 1
    used = (partner != np.uint32(0xFFFFFFFF)) | (area > 0)
    atom, slot = np.nonzero(used)                        # atom-major: batch atom order
    sid = np.searchsorted(off, atom, side="right") - 1
    g = group[atom].astype(np.int64)
    h = partner[atom, slot].astype(np.int64)
    tables = [[] for _ in range(max(S, 0))]
    if atom.shape[0] == 0:
        return tables
    keys, inv = np.unique(np.stack([sid, g, h], axis=1), axis=0, return_inverse=True)
    sums = np.zeros(keys.shape[0], np.float64)
    np.add.at(sums, inv.reshape(-1), area[atom, slot].astype(np.float64))   # unbuffered, in index (= atom) order
    by_key = {tuple(int(x) for x in k): float(v) for k, v in zip(keys, sums)}
    for (s, a, b) in sorted({(s, min(a, b), max(a, b)) for (s, a, b) in by_key}):
        tables[s].append((a, b, by_key.get((s, a, b), 0.0), by_key.get((s, b, a), 0.0)))
    return tables


class Engine:
    """One sasa_b200 context on one CUDA device."""

    def __init__(self, device: int = -1):
        self._L = _lib.load()
        h = C.c_void_p()
        rc = self._L.sasa_b200_create(device, C.byref(h))
        if rc != _lib.OK:
            raise SasaB200Error(rc, self._L.sasa_b200_last_error(None).decode())
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._L.sasa_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != _lib.OK:
            raise SasaB200Error(rc, self._L.sasa_b200_last_error(self._h).decode())

    @staticmethod
    def sphere_points(n_points: int) -> np.ndarray:
        out = np.empty((n_points, 3), np.float32)
        rc = _lib.load().sasa_b200_sphere_points(n_points, out.ctypes.data)
        if rc != _lib.OK:
            raise SasaB200Error(rc, "sphere_points: invalid argument")
        return out

    def pinned_empty(self, shape, dtype) -> np.ndarray:
        """numpy array backed by page-locked memory (freed when the array is collected)."""
        dtype = np.dtype(dtype)
        shape = (int(shape),) if np.isscalar(shape) else tuple(int(x) for x in shape)
        n = int(np.prod(shape)) * dtype.itemsize
        p = C.c_void_p()
        rc = self._L.sasa_b200_alloc_pinned(n, C.byref(p))
        if rc != _lib.OK:
            raise SasaB200Error(rc, self._L.sasa_b200_last_error(None).decode())
        return np.asarray(_PinnedBlock(self._L, p.value, n, shape, dtype))

    def calculate_sasa_internal(self, xyzr, ids=None, probe_radius=1.4, n_points=100, threads=-1,
                                want_counts=False):
        """The reference's raw-atoms entry point (src/lib.rs:249-298) through the C ABI."""
        xyzr = _np(xyzr, np.float32, (-1, 4))
        n = xyzr.shape[0]
        ids = _np(ids, np.uint64)
        out = np.zeros(n, np.float32)
        counts = np.zeros(n, np.uint32) if want_counts else None
        self._check(self._L.sasa_b200_calculate_sasa_internal(
            self._h, _ptr(xyzr), _ptr(ids), n, probe_radius, n_points, threads, _ptr(out), _ptr(counts)))
        return (out, counts) if want_counts else out

    def batch(self, struct_off, seg_be=None, struct_seg_off=None, seg_polar=None) -> "Batch":
        return Batch(self, struct_off, seg_be, struct_seg_off, seg_polar)


class Batch:
    """Topology of a batch of structures (CSR offsets + output segments), reusable across runs."""

    def __init__(self, engine: Engine, struct_off, seg_be=None, struct_seg_off=None, seg_polar=None):
        self.engine = engine
        self._L = engine._L
        self.struct_off = _np(struct_off, np.uint64)
        self.S = self.struct_off.shape[0] - 1
        self.n_atoms = int(self.struct_off[-1]) if self.S >= 0 and self.struct_off.size else 0
        self.seg_be = _np(seg_be, np.uint32, (-1, 2))
        self.struct_seg_off = _np(struct_seg_off, np.uint64)
        self.seg_polar = _np(seg_polar, np.uint8)
        self.n_seg = 0 if self.seg_be is None else self.seg_be.shape[0]
        h = C.c_void_p()
        engine._check(self._L.sasa_b200_batch_create(
            engine._h, _ptr(self.struct_off), max(self.S, 0), _ptr(self.seg_be), _ptr(self.struct_seg_off),
            _ptr(self.seg_polar), C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and getattr(self.engine, "_h", None):
            self._L.sasa_b200_batch_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _params(probe_radius, n_points, simd_lanes, flags):
        return _lib.Params(probe_radius, n_points, simd_lanes, -1, flags)

    def _host_outputs(self, want, out):
        res = BatchResult()
        alloc = (lambda shape, dt: self.engine.pinned_empty(shape, dt)) if out == "pinned" else np.zeros
        if "counts" in want:
            res.counts = alloc(self.n_atoms, np.uint32)
        if "atom" in want:
            res.atom_sasa = alloc(self.n_atoms, np.float32)
        if "seg" in want and self.n_seg:
            res.seg_sasa = alloc(self.n_seg, np.float32)
        if "protein" in want:
            res.protein = alloc((max(self.S, 0), 3), np.float32)
        return res

    def run_host(self, xyzr, id_class=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                 want=("counts", "atom", "seg", "protein"), result: Optional[BatchResult] = None) -> BatchResult:
        xyzr = _np(xyzr, np.float32, (-1, 4))
        assert xyzr.shape[0] == self.n_atoms, "xyzr does not match struct_off"
        id_class = _np(id_class, np.uint32)
        res = result if result is not None else self._host_outputs(want, "numpy")
        outs = _lib.Outputs(_ptr(res.counts), _ptr(res.atom_sasa), _ptr(res.seg_sasa), _ptr(res.protein))
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        st = _lib.Stats()
        self.engine._check(self._L.sasa_b200_batch_run_host(self._h, _ptr(xyzr), _ptr(id_class), C.byref(prm),
                                                           C.byref(outs), C.byref(st)))
        res.stats = st.as_dict()
        return res

    def submit_host(self, xyzr, id_class=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                    want=("counts", "atom", "seg", "protein"), result: Optional[BatchResult] = None) -> "Job":
        """Asynchronous run_host: returns at once with a Job; `Job.wait()` blocks until the outputs are in host memory.
        Inputs and outputs should be page-locked (``Engine.pinned_empty``) and must stay alive until wait returns."""
        xyzr = _np(xyzr, np.float32, (-1, 4))
        assert xyzr.shape[0] == self.n_atoms, "xyzr does not match struct_off"
        id_class = _np(id_class, np.uint32)
        res = result if result is not None else self._host_outputs(want, "pinned")
        outs = _lib.Outputs(_ptr(res.counts), _ptr(res.atom_sasa), _ptr(res.seg_sasa), _ptr(res.protein))
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        h = C.c_void_p()
        self.engine._check(self._L.sasa_b200_batch_submit_host(self._h, _ptr(xyzr), _ptr(id_class), C.byref(prm),
                                                              C.byref(outs), C.byref(h)))
        return Job(self, h, res, (xyzr, id_class))

    def run_frames_host(self, xyz, radii, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                        want=("protein",), result: Optional[BatchResult] = None) -> BatchResult:
        """MD form: xyz (F, N, 3) float32 + radii (N,) shared by all frames."""
        xyz = _np(xyz, np.float32, (-1, 3))
        radii = _np(radii, np.float32)
        assert xyz.shape[0] == self.n_atoms
        res = result if result is not None else self._host_outputs(want, "numpy")
        outs = _lib.Outputs(_ptr(res.counts), _ptr(res.atom_sasa), _ptr(res.seg_sasa), _ptr(res.protein))
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        st = _lib.Stats()
        self.engine._check(self._L.sasa_b200_batch_run_frames_host(self._h, _ptr(xyz), _ptr(radii), C.byref(prm),
                                                                  C.byref(outs), C.byref(st)))
        res.stats = st.as_dict()
        return res

    def run_indexed_host(self, xyz, radius_index, palette, id_class=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                         want=("counts", "atom", "seg", "protein"), result: Optional[BatchResult] = None) -> BatchResult:
        """Indexed-radius form (13 B/atom on the wire): xyz (N, 3) float32, radius_index (N,) uint8 into palette (<= 256,)."""
        xyz = _np(xyz, np.float32, (-1, 3))
        radius_index = _np(radius_index, np.uint8)
        palette = _np(palette, np.float32)
        assert xyz.shape[0] == self.n_atoms == radius_index.shape[0]
        id_class = _np(id_class, np.uint32)
        res = result if result is not None else self._host_outputs(want, "numpy")
        outs = _lib.Outputs(_ptr(res.counts), _ptr(res.atom_sasa), _ptr(res.seg_sasa), _ptr(res.protein))
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        st = _lib.Stats()
        self.engine._check(self._L.sasa_b200_batch_run_indexed_host(self._h, _ptr(xyz), _ptr(radius_index), _ptr(palette),
                                                                   palette.shape[0], _ptr(id_class), C.byref(prm), C.byref(outs),
                                                                   C.byref(st)))
        res.stats = st.as_dict()
        return res

    def run_device(self, d_xyzr, d_id_class=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                   counts=None, atom_sasa=None, seg_sasa=None, protein=None, stream=None):
        """All tensors are torch CUDA tensors; enqueues on `stream` (None = torch's current stream, else a raw
        cudaStream_t handle) and returns without synchronising."""
        outs = _lib.Outputs(_ptr(counts), _ptr(atom_sasa), _ptr(seg_sasa), _ptr(protein))
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        self.engine._check(self._L.sasa_b200_batch_run_device(self._h, _ptr(d_xyzr), _ptr(d_id_class), C.byref(prm),
                                                             C.byref(outs), _stream(stream)))

    def run_masks_host(self, xyzr, id_class=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                       want=("counts", "atom", "seg", "protein")) -> BatchResult:
        """run_host plus every atom's exposed-point mask in ``exposed``, an (n_atoms, W) uint32 array with W = ceil(n_points /
        32): bit b of word w is set when point 32 w + b (the order of ``Engine.sphere_points``) is solvent-accessible."""
        xyzr = _np(xyzr, np.float32, (-1, 4))
        assert xyzr.shape[0] == self.n_atoms, "xyzr does not match struct_off"
        id_class = _np(id_class, np.uint32)
        res = self._host_outputs(want, "numpy")
        res.exposed = np.zeros((self.n_atoms, (n_points + 31) // 32), np.uint32)
        outs = _lib.Outputs(_ptr(res.counts), _ptr(res.atom_sasa), _ptr(res.seg_sasa), _ptr(res.protein))
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        st = _lib.Stats()
        self.engine._check(self._L.sasa_b200_batch_run_masks_host(self._h, _ptr(xyzr), _ptr(id_class), C.byref(prm), C.byref(outs),
                                                                 _ptr(res.exposed), C.byref(st)))
        res.stats = st.as_dict()
        return res

    def run_masks_device(self, d_xyzr, d_exposed, d_id_class=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                         counts=None, atom_sasa=None, seg_sasa=None, protein=None, stream=None):
        """run_device plus the exposed-point masks into ``d_exposed``, a torch CUDA tensor of n_atoms * ceil(n_points / 32)
        32-bit words (e.g. int32 of shape (n_atoms, W)); enqueues on `stream` and returns without synchronising."""
        if d_exposed is not None:
            assert d_exposed.numel() * d_exposed.element_size() >= self.n_atoms * ((n_points + 31) // 32) * 4, "d_exposed is too small"
        outs = _lib.Outputs(_ptr(counts), _ptr(atom_sasa), _ptr(seg_sasa), _ptr(protein))
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        self.engine._check(self._L.sasa_b200_batch_run_masks_device(self._h, _ptr(d_xyzr), _ptr(d_id_class), C.byref(prm),
                                                                   C.byref(outs), _ptr(d_exposed), _stream(stream)))

    def run_groups_host(self, xyzr, group, id_class=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                        want=("counts", "atom", "seg", "protein")):
        """Grouped run (buried surface area): one label per atom in `group`.  Returns (complex, isolated) BatchResults: the
        complex is what run_host gives; isolated is every atom with its group standing alone (only same-group neighbours
        occlude).  Buried area = isolated - complex."""
        xyzr = _np(xyzr, np.float32, (-1, 4))
        assert xyzr.shape[0] == self.n_atoms, "xyzr does not match struct_off"
        group = _np(group, np.uint32)
        assert group is None or group.shape[0] == self.n_atoms, "group does not match struct_off"
        id_class = _np(id_class, np.uint32)
        cpx, iso = self._host_outputs(want, "numpy"), self._host_outputs(want, "numpy")
        outs = [_lib.Outputs(_ptr(r.counts), _ptr(r.atom_sasa), _ptr(r.seg_sasa), _ptr(r.protein)) for r in (cpx, iso)]
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        st = _lib.Stats()
        self.engine._check(self._L.sasa_b200_batch_run_groups_host(self._h, _ptr(xyzr), _ptr(id_class), _ptr(group), C.byref(prm),
                                                                  C.byref(outs[0]), C.byref(outs[1]), C.byref(st)))
        cpx.stats = iso.stats = st.as_dict()
        return cpx, iso

    def run_group_pairs_host(self, xyzr, group, id_class=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                             want=("counts", "atom", "seg", "protein"), max_partners=4):
        """Pairwise buried area: run_groups_host plus, for every atom, which partner groups bury how much of it.  Returns
        (complex, isolated, pairs): the first two are run_groups_host's BatchResults bit for bit, pairs a :class:`PairResult` of
        (n_atoms, max_partners) arrays.  When an atom has more than max_partners partners, :class:`SasaB200Error` is raised
        with ``needed`` (the max_partners the batch needs) and ``result`` (the (complex, isolated, pairs) triple, complete
        except for the partners past the slots) set on the exception."""
        xyzr = _np(xyzr, np.float32, (-1, 4))
        assert xyzr.shape[0] == self.n_atoms, "xyzr does not match struct_off"
        group = _np(group, np.uint32)
        assert group is None or group.shape[0] == self.n_atoms, "group does not match struct_off"
        id_class = _np(id_class, np.uint32)
        cpx, iso = self._host_outputs(want, "numpy"), self._host_outputs(want, "numpy")
        K = int(max_partners)
        shape = (self.n_atoms, max(K, 0))
        pairs = PairResult(np.zeros(shape, np.uint32), np.zeros(shape, np.uint32), np.zeros(shape, np.float32))
        needed = np.zeros(1, np.uint32)
        outs = [_lib.Outputs(_ptr(r.counts), _ptr(r.atom_sasa), _ptr(r.seg_sasa), _ptr(r.protein)) for r in (cpx, iso)]
        po = _lib.PairOutputs(K, _ptr(pairs.partner), _ptr(pairs.buried_counts), _ptr(pairs.buried_area), _ptr(needed))
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        st = _lib.Stats()
        rc = self._L.sasa_b200_batch_run_group_pairs_host(self._h, _ptr(xyzr), _ptr(id_class), _ptr(group), C.byref(prm),
                                                          C.byref(outs[0]), C.byref(outs[1]), C.byref(po), C.byref(st))
        pairs.needed = int(needed[0])
        cpx.stats = iso.stats = st.as_dict()
        if rc != _lib.OK:
            err = SasaB200Error(rc, self._L.sasa_b200_last_error(self.engine._h).decode())
            err.needed, err.result = pairs.needed, (cpx, iso, pairs)
            raise err
        return cpx, iso, pairs

    def run_group_pairs_device(self, d_xyzr, d_group, d_id_class=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                               want=("counts", "atom", "seg", "protein"), max_partners=4, stream=None):
        """run_group_pairs_host on torch CUDA tensors: allocates every output on the input's device, enqueues on `stream` (None
        = torch's current stream) and returns (complex, isolated, pairs) of tensors without synchronising; ``pairs.needed`` is a
        one-element int32 tensor.  Too few slots is reported by ``Batch.sync`` (:class:`SasaB200Error`), like non-finite
        input."""
        import torch
        dev = d_xyzr.device
        cpx, iso = self._device_outputs(want, dev), self._device_outputs(want, dev)
        K = int(max_partners)
        shape = (self.n_atoms, max(K, 0))
        pairs = PairResult(torch.empty(shape, dtype=torch.int32, device=dev), torch.empty(shape, dtype=torch.int32, device=dev),
                           torch.empty(shape, dtype=torch.float32, device=dev), torch.zeros(1, dtype=torch.int32, device=dev))
        outs = [_lib.Outputs(_ptr(r.counts), _ptr(r.atom_sasa), _ptr(r.seg_sasa), _ptr(r.protein)) for r in (cpx, iso)]
        po = _lib.PairOutputs(K, _ptr(pairs.partner), _ptr(pairs.buried_counts), _ptr(pairs.buried_area), _ptr(pairs.needed))
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        self.engine._check(self._L.sasa_b200_batch_run_group_pairs_device(self._h, _ptr(d_xyzr), _ptr(d_id_class), _ptr(d_group),
                                                                         C.byref(prm), C.byref(outs[0]), C.byref(outs[1]), C.byref(po),
                                                                         _stream(stream)))
        return cpx, iso, pairs

    def _groups_frames_args(self, xyz, radii, group):
        xyz = _np(xyz, np.float32, (-1, 3))
        radii = _np(radii, np.float32)
        group = _np(group, np.uint32)
        assert xyz.shape[0] == self.n_atoms, "xyz does not match struct_off"
        assert group is None or radii is None or group.shape == radii.shape, "group and radii hold one value per atom of a frame"
        return xyz, radii, group

    def run_groups_frames_host(self, xyz, radii, group, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                               want=("protein",), result=None):
        """Grouped run in the MD form: xyz (F, N, 3) float32, radii (N,) and group (N,) labels shared by every frame.  Returns
        (complex, isolated) BatchResults: complex is run_frames_host's result, isolated what run_groups_host gives with the
        labels tiled over the frames.  Buried area per frame = isolated - complex.  `result`: a (complex, isolated) pair of
        BatchResults to write into instead of new arrays."""
        xyz, radii, group = self._groups_frames_args(xyz, radii, group)
        cpx, iso = result if result is not None else (self._host_outputs(want, "numpy"), self._host_outputs(want, "numpy"))
        outs = [_lib.Outputs(_ptr(r.counts), _ptr(r.atom_sasa), _ptr(r.seg_sasa), _ptr(r.protein)) for r in (cpx, iso)]
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        st = _lib.Stats()
        self.engine._check(self._L.sasa_b200_batch_run_groups_frames_host(self._h, _ptr(xyz), _ptr(radii), _ptr(group), C.byref(prm),
                                                                         C.byref(outs[0]), C.byref(outs[1]), C.byref(st)))
        cpx.stats = iso.stats = st.as_dict()
        return cpx, iso

    def submit_groups_frames_host(self, xyz, radii, group, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                                  want=("protein",), result=None) -> "Job":
        """Asynchronous run_groups_frames_host: returns at once with a Job whose ``wait()`` returns (complex, isolated).  The
        outputs are page-locked; xyz should be too (``Engine.pinned_empty``), and the inputs must stay alive until wait
        returns."""
        xyz, radii, group = self._groups_frames_args(xyz, radii, group)
        res = result if result is not None else (self._host_outputs(want, "pinned"), self._host_outputs(want, "pinned"))
        outs = [_lib.Outputs(_ptr(r.counts), _ptr(r.atom_sasa), _ptr(r.seg_sasa), _ptr(r.protein)) for r in res]
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        h = C.c_void_p()
        self.engine._check(self._L.sasa_b200_batch_submit_groups_frames_host(self._h, _ptr(xyz), _ptr(radii), _ptr(group),
                                                                            C.byref(prm), C.byref(outs[0]), C.byref(outs[1]),
                                                                            C.byref(h)))
        return Job(self, h, tuple(res), (xyz, radii, group))

    def _pair_sums(self, n_labels, seg_pairs, out):
        alloc = (lambda shape: self.engine.pinned_empty(shape, np.float64)) if out == "pinned" else (lambda shape: np.zeros(shape, np.float64))
        L = int(n_labels)
        return PairSums(L, alloc((max(self.S, 0), L, L)), alloc((self.n_seg, L)) if seg_pairs and self.n_seg else None)

    def run_group_pairs_frames_host(self, xyz, radii, group, n_labels=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                                    want=("protein",), seg_pairs=True, result=None):
        """Pairwise buried area of MD frames: run_groups_frames_host plus, per frame, how much of every group each partner group
        buries, summed on the device.  ``group`` (N,) holds labels 0 .. n_labels - 1 (default: max + 1), n_labels <= 17.  Returns
        (complex, isolated, sums): the first two are run_groups_frames_host's BatchResults bit for bit, ``sums`` a
        :class:`PairSums` (its ``seg_pair_area`` when the batch has segments and ``seg_pairs``).  `result`: a (complex, isolated,
        sums) triple to write into instead of new arrays."""
        xyz, radii, group = self._groups_frames_args(xyz, radii, group)
        if n_labels is None:
            n_labels = int(group.max()) + 1 if group is not None and group.size else 1
        cpx, iso, sums = result if result is not None else (self._host_outputs(want, "numpy"), self._host_outputs(want, "numpy"),
                                                            self._pair_sums(n_labels, seg_pairs, "numpy"))
        outs = [_lib.Outputs(_ptr(r.counts), _ptr(r.atom_sasa), _ptr(r.seg_sasa), _ptr(r.protein)) for r in (cpx, iso)]
        ps = _lib.PairSums(sums.n_labels, _ptr(sums.pair_area), _ptr(sums.seg_pair_area))
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        st = _lib.Stats()
        self.engine._check(self._L.sasa_b200_batch_run_group_pairs_frames_host(self._h, _ptr(xyz), _ptr(radii), _ptr(group), C.byref(prm),
                                                                              C.byref(outs[0]), C.byref(outs[1]), C.byref(ps), C.byref(st)))
        cpx.stats = iso.stats = st.as_dict()
        return cpx, iso, sums

    def submit_group_pairs_frames_host(self, xyz, radii, group, n_labels=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                                       want=("protein",), seg_pairs=True, result=None) -> "Job":
        """Asynchronous run_group_pairs_frames_host: returns at once with a Job whose ``wait()`` returns (complex, isolated,
        sums).  The outputs are page-locked; xyz should be too (``Engine.pinned_empty``), and the inputs must stay alive until
        wait returns."""
        xyz, radii, group = self._groups_frames_args(xyz, radii, group)
        if n_labels is None:
            n_labels = int(group.max()) + 1 if group is not None and group.size else 1
        res = result if result is not None else (self._host_outputs(want, "pinned"), self._host_outputs(want, "pinned"),
                                                 self._pair_sums(n_labels, seg_pairs, "pinned"))
        outs = [_lib.Outputs(_ptr(r.counts), _ptr(r.atom_sasa), _ptr(r.seg_sasa), _ptr(r.protein)) for r in res[:2]]
        ps = _lib.PairSums(res[2].n_labels, _ptr(res[2].pair_area), _ptr(res[2].seg_pair_area))
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        h = C.c_void_p()
        self.engine._check(self._L.sasa_b200_batch_submit_group_pairs_frames_host(self._h, _ptr(xyz), _ptr(radii), _ptr(group),
                                                                                 C.byref(prm), C.byref(outs[0]), C.byref(outs[1]),
                                                                                 C.byref(ps), C.byref(h)))
        return Job(self, h, tuple(res), (xyz, radii, group))

    def _device_outputs(self, want, dev) -> BatchResult:
        import torch
        r = BatchResult()
        if "counts" in want:
            r.counts = torch.zeros(self.n_atoms, dtype=torch.int32, device=dev)
        if "atom" in want:
            r.atom_sasa = torch.zeros(self.n_atoms, dtype=torch.float32, device=dev)
        if "seg" in want and self.n_seg:
            r.seg_sasa = torch.zeros(self.n_seg, dtype=torch.float32, device=dev)
        if "protein" in want:
            r.protein = torch.zeros((max(self.S, 0), 3), dtype=torch.float32, device=dev)
        return r

    def run_groups_device(self, d_xyzr, d_group, d_id_class=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                          want=("counts", "atom", "seg", "protein"), stream=None):
        """run_groups_host on torch CUDA tensors: allocates the outputs on the input's device, enqueues on `stream` (None =
        torch's current stream) and returns (complex, isolated) BatchResults of tensors without synchronising."""
        cpx, iso = self._device_outputs(want, d_xyzr.device), self._device_outputs(want, d_xyzr.device)
        outs = [_lib.Outputs(_ptr(r.counts), _ptr(r.atom_sasa), _ptr(r.seg_sasa), _ptr(r.protein)) for r in (cpx, iso)]
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        self.engine._check(self._L.sasa_b200_batch_run_groups_device(self._h, _ptr(d_xyzr), _ptr(d_id_class), _ptr(d_group),
                                                                    C.byref(prm), C.byref(outs[0]), C.byref(outs[1]),
                                                                    _stream(stream)))
        return cpx, iso

    def run_groups_masks_host(self, xyzr, group, id_class=None, probe_radius=1.4, n_points=100, simd_lanes=8, flags=0,
                              want=("counts", "atom", "seg", "protein")):
        """run_groups_host plus the exposed-point masks of both evaluations: complex.exposed is run_masks_host's mask, and
        isolated.exposed every atom's mask with its group standing alone, each (n_atoms, W) uint32.  The interface patch -- the
        points of atom i that other groups bury -- is ``isolated.exposed[i] & ~complex.exposed[i]``."""
        xyzr = _np(xyzr, np.float32, (-1, 4))
        assert xyzr.shape[0] == self.n_atoms, "xyzr does not match struct_off"
        group = _np(group, np.uint32)
        assert group is None or group.shape[0] == self.n_atoms, "group does not match struct_off"
        id_class = _np(id_class, np.uint32)
        cpx, iso = self._host_outputs(want, "numpy"), self._host_outputs(want, "numpy")
        for r in (cpx, iso):
            r.exposed = np.zeros((self.n_atoms, (n_points + 31) // 32), np.uint32)
        outs = [_lib.Outputs(_ptr(r.counts), _ptr(r.atom_sasa), _ptr(r.seg_sasa), _ptr(r.protein)) for r in (cpx, iso)]
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        st = _lib.Stats()
        self.engine._check(self._L.sasa_b200_batch_run_groups_masks_host(
            self._h, _ptr(xyzr), _ptr(id_class), _ptr(group), C.byref(prm), C.byref(outs[0]), C.byref(outs[1]), _ptr(cpx.exposed),
            _ptr(iso.exposed), C.byref(st)))
        cpx.stats = iso.stats = st.as_dict()
        return cpx, iso

    def run_groups_masks_device(self, d_xyzr, d_group, d_exposed, d_exposed_isolated, d_id_class=None, probe_radius=1.4,
                                n_points=100, simd_lanes=8, flags=0, want=("counts", "atom", "seg", "protein"), stream=None):
        """run_groups_device plus the masks of both evaluations into ``d_exposed`` (complex) and ``d_exposed_isolated``, torch
        CUDA tensors of n_atoms * ceil(n_points / 32) 32-bit words each.  Returns (complex, isolated) BatchResults of tensors,
        with ``exposed`` set to the two mask tensors, without synchronising."""
        W = (n_points + 31) // 32
        for m in (d_exposed, d_exposed_isolated):
            if m is not None:
                assert m.numel() * m.element_size() >= self.n_atoms * W * 4, "mask tensor is too small"
        cpx, iso = self._device_outputs(want, d_xyzr.device), self._device_outputs(want, d_xyzr.device)
        cpx.exposed, iso.exposed = d_exposed, d_exposed_isolated
        outs = [_lib.Outputs(_ptr(r.counts), _ptr(r.atom_sasa), _ptr(r.seg_sasa), _ptr(r.protein)) for r in (cpx, iso)]
        prm = self._params(probe_radius, n_points, simd_lanes, flags)
        self.engine._check(self._L.sasa_b200_batch_run_groups_masks_device(
            self._h, _ptr(d_xyzr), _ptr(d_id_class), _ptr(d_group), C.byref(prm), C.byref(outs[0]), C.byref(outs[1]),
            _ptr(d_exposed), _ptr(d_exposed_isolated), _stream(stream)))
        return cpx, iso

    def run_atom_range_device(self, d_xyzr, rank: int, n_ranks: int, d_id_class=None, probe_radius=1.4, n_points=100,
                              simd_lanes=8, counts=None, atom_sasa=None, stream=None):
        """Atom-range split (cfg5): slice `rank` of `n_ranks` of every structure's cell-sorted atom order; the
        output tensors are zero outside the slice, ready for an all-reduce(SUM) across ranks."""
        prm = self._params(probe_radius, n_points, simd_lanes, 0)
        self.engine._check(self._L.sasa_b200_batch_run_atom_range_device(
            self._h, _ptr(d_xyzr), _ptr(d_id_class), C.byref(prm), rank, n_ranks, _ptr(counts), _ptr(atom_sasa),
            _stream(stream)))

    def run_atom_range_peers_device(self, d_xyzr, rank: int, n_ranks: int, peer_counts=None, peer_atom_sasa=None, d_id_class=None,
                                    probe_radius=1.4, n_points=100, simd_lanes=8, stream=None):
        """Atom-range split with the exchange fused into the kernel: peer_counts / peer_atom_sasa are sequences of n_ranks
        raw device pointers (ints), valid on this device, of every rank's output vector (symmetric-memory buffer_ptrs)."""
        prm = self._params(probe_radius, n_points, simd_lanes, 0)
        pc = (C.c_void_p * n_ranks)(*[int(x) for x in peer_counts]) if peer_counts is not None else None
        pa = (C.c_void_p * n_ranks)(*[int(x) for x in peer_atom_sasa]) if peer_atom_sasa is not None else None
        self.engine._check(self._L.sasa_b200_batch_run_atom_range_peers_device(
            self._h, _ptr(d_xyzr), _ptr(d_id_class), C.byref(prm), rank, n_ranks, pc, pa, _stream(stream)))

    def run_atom_range_host(self, xyzr, rank: int, n_ranks: int, id_class=None, probe_radius=1.4, n_points=100,
                            simd_lanes=8) -> BatchResult:
        xyzr = _np(xyzr, np.float32, (-1, 4))
        assert xyzr.shape[0] == self.n_atoms, "xyzr does not match struct_off"
        id_class = _np(id_class, np.uint32)
        res = BatchResult(counts=np.zeros(self.n_atoms, np.uint32), atom_sasa=np.zeros(self.n_atoms, np.float32))
        prm = self._params(probe_radius, n_points, simd_lanes, 0)
        st = _lib.Stats()
        self.engine._check(self._L.sasa_b200_batch_run_atom_range_host(
            self._h, _ptr(xyzr), _ptr(id_class), C.byref(prm), rank, n_ranks, _ptr(res.counts), _ptr(res.atom_sasa),
            C.byref(st)))
        res.stats = st.as_dict()
        return res

    def reduce_device(self, d_atom_sasa, seg_sasa=None, protein=None, stream=None):
        """Level sums of a finished per-atom SASA vector (torch CUDA tensors)."""
        self.engine._check(self._L.sasa_b200_batch_reduce_device(self._h, _ptr(d_atom_sasa), _ptr(seg_sasa), _ptr(protein),
                                                                _stream(stream)))

    def sync(self) -> dict:
        st = _lib.Stats()
        self.engine._check(self._L.sasa_b200_batch_sync(self._h, C.byref(st)))
        return st.as_dict()


class Job:
    """A host-buffer run in flight (sasa_b200_batch_submit_host .. sasa_b200_job_wait).  `result` is a BatchResult, the
    (complex, isolated) pair of a grouped run, or the (complex, isolated, sums) triple of a pairwise run of frames."""

    def __init__(self, batch: Batch, handle, result, keep):
        self.batch, self._h, self.result, self._keep = batch, handle, result, keep

    def wait(self):
        if self._h is None:
            return self.result
        st = _lib.Stats()
        h, self._h = self._h, None
        self.batch.engine._check(self.batch._L.sasa_b200_job_wait(h, C.byref(st)))
        for r in (self.result if isinstance(self.result, tuple) else (self.result,)):
            if isinstance(r, BatchResult):
                r.stats = st.as_dict()
        self._keep = None
        return self.result
