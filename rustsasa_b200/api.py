"""Host-side mirror of the reference's public interface for the hot path.

Same names, argument meaning and error behaviour as the crate (rust-sasa 0.9.2):

* ``calculate_sasa_internal(atoms, probe_radius, n_points, threads)`` -- src/lib.rs:249-298
* ``SASAOptions`` builder with ``AtomLevel | ResidueLevel | ChainLevel | ProteinLevel`` and
  ``process()`` -- src/options.rs:60-70, :496-618; defaults probe 1.4, n_points 100, threads -1,
  hydrogens / HETATM / vdW fallback / occupancy radii all off (:498-510)
* result structs ``ResidueResult``, ``ChainResult``, ``ProteinResult`` -- src/structures/atomic.rs:26-70
* ``SASACalcError`` variants -- src/options.rs:466-494 (raised host-side, before / after the numeric core)

The numeric core is the C ABI (include/sasa_b200.h); there is no CPU path here.
``process_many`` is the batched form the CLI's directory mode (src/main.rs:342-480) maps onto.
``process_interface`` adds buried surface area: every structure in the complex and with each chain group standing alone,
from one grouped batch call.  ``process_surface`` and ``surface_points`` give the dot surface: the solvent-accessible test
points themselves, from the exposed-point masks of the same batch call.  ``process_interface_surface`` gives both: the buried
area and the interface patches, the test points that partner groups bury, from one grouped batch call with masks.
``process_interface_pairs`` gives the pairwise interfaces: how much of every chain group each other group buries, from one
grouped batch call with partner slots.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Any, List, Optional, Sequence

import numpy as np

from .engine import Batch, Engine, SasaB200Error, group_pair_table
from .structure import (PackedStructure, SASACalcError, Structure, build_atoms_and_mapping,  # noqa: F401
                        load_radii_from_file, read_structure)

_ENGINE: Optional[Engine] = None


def default_engine() -> Engine:
    global _ENGINE
    if _ENGINE is None:
        _ENGINE = Engine()
    return _ENGINE


@dataclass
class Atom:
    """src/structures/atomic.rs:13-24."""
    position: Sequence[float]
    radius: float
    id: int
    parent_id: Optional[int] = None


@dataclass
class ChainResult:
    name: str
    value: float


@dataclass
class ResidueResult:
    serial_number: int
    insertion_code: str
    value: float
    name: str
    is_polar: bool
    chain_id: str


@dataclass
class ProteinResult:
    global_total: float
    polar_total: float
    non_polar_total: float


@dataclass
class InterfaceResult:
    """One structure of ``SASAOptions.process_interface``: the level's result in the complex and with every chain group
    standing alone, and the buried area isolated - complex of the protein totals (global)."""
    complex: Any
    isolated: Any
    buried_area: float


@dataclass
class SurfaceResult:
    """One structure of ``SASAOptions.process_surface``: the level's result, the exposed test points (M, 3) float32 and for
    each point the index of its atom in the order of an atom-level result (M,) int64."""
    result: Any
    points: np.ndarray
    atom_index: np.ndarray


@dataclass
class InterfaceSurfaceResult:
    """One structure of ``SASAOptions.process_interface_surface``: the :class:`InterfaceResult` and the interface patches, the
    test points exposed with the atom's group standing alone but buried in the complex, (M, 3) float32, with for each point
    the index of its atom in the order of an atom-level result (M,) int64."""
    interface: InterfaceResult
    points: np.ndarray
    atom_index: np.ndarray


@dataclass
class GroupPairResult:
    """One contacting pair of chain groups of ``SASAOptions.process_interface_pairs``: their group labels (a < b), the chain ids
    of each, and the area of group a that group b buries and the area of group b that group a buries (float64 sums over the
    per-atom areas in atom order)."""
    group_a: int
    group_b: int
    chains_a: str
    chains_b: str
    buried_a: float
    buried_b: float


@dataclass
class InterfacePairsResult:
    """One structure of ``SASAOptions.process_interface_pairs``: the :class:`InterfaceResult` of ``process_interface``, the
    contacting pairs of chain groups, and at residue level, per residue, ``{partner group: buried area}`` (float64 sums over the
    residue's atoms in atom order; None at the other levels)."""
    interface: InterfaceResult
    pairs: List[GroupPairResult]
    residue_partners: Optional[List[dict]] = None


@dataclass
class TrajectoryInterfaceResult:
    """``trajectory_interface``: per frame the protein totals (global, polar, non-polar) in the complex and with every group
    standing alone, (F, 3) float32 each, the buried area isolated - complex of the global totals (F,), and with residue ranges
    given, the segment sums (F, G) of both.  With ``pairs=True``: ``pair_labels`` (L,) the distinct labels in ascending order,
    ``pair_area`` (F, L, L) float64, element [f, a, b] the area of group pair_labels[a] that group pair_labels[b] buries in frame f,
    and with residue ranges given ``seg_pair_area`` (F, G, L) float64, the area of each residue that each group buries."""
    complex: np.ndarray
    isolated: np.ndarray
    buried: np.ndarray
    complex_seg: Optional[np.ndarray] = None
    isolated_seg: Optional[np.ndarray] = None
    pair_labels: Optional[np.ndarray] = None
    pair_area: Optional[np.ndarray] = None
    seg_pair_area: Optional[np.ndarray] = None


class AtomLevel:
    name = "atom"


class ResidueLevel:
    name = "residue"


class ChainLevel:
    name = "chain"


class ProteinLevel:
    name = "protein"


def calculate_sasa_internal(atoms, probe_radius: float = 1.4, n_points: int = 100, threads: int = -1,
                            engine: Optional[Engine] = None) -> np.ndarray:
    """SASA per atom.  ``atoms`` is a sequence of :class:`Atom` or an (N, 4) float32 array of x, y, z, radius
    (ids then default to the index).  ``threads`` is accepted and ignored (the GPU path has no thread pool)."""
    eng = engine or default_engine()
    if isinstance(atoms, np.ndarray):
        return eng.calculate_sasa_internal(atoms, None, probe_radius, n_points, threads)
    atoms = list(atoms)
    if not atoms:
        return np.zeros(0, np.float32)
    xyzr = np.array([[a.position[0], a.position[1], a.position[2], a.radius] for a in atoms], dtype=np.float32)
    ids = np.array([a.id & 0xFFFFFFFFFFFFFFFF for a in atoms], dtype=np.uint64)
    return eng.calculate_sasa_internal(xyzr, ids, probe_radius, n_points, threads)


def surface_points(xyzr, exposed, n_points: int, probe_radius: float = 1.4):
    """The dot surface from exposed-point masks: for every set bit b of word w of atom i (``Batch.run_masks_host``'s
    ``exposed``, (N, W) uint32) the point centre_i + (r_i + probe) * p_(32 w + b), in float32 with the engine's sphere points.
    Returns (points (M, 3) float32, atom (M,) int64), atom-major and in point order within an atom."""
    xyzr = np.ascontiguousarray(xyzr, np.float32).reshape(-1, 4)
    exposed = np.ascontiguousarray(exposed, np.uint32).reshape(xyzr.shape[0], -1)
    bits = np.unpackbits(exposed.view(np.uint8), axis=1, bitorder="little")[:, :n_points]
    atom, k = np.nonzero(bits)
    sphere = Engine.sphere_points(n_points)
    r = xyzr[atom, 3] + np.float32(probe_radius)
    points = xyzr[atom, :3] + r[:, None] * sphere[k]
    return points.astype(np.float32, copy=False), atom.astype(np.int64)


# Page-locked staging of one block of trajectory_interface's frames (two blocks are staged at once).
_TRAJECTORY_STAGING_BYTES = 256 << 20


def trajectory_interface(xyz, radii, group, seg_be=None, seg_polar=None, probe_radius: float = 1.4, n_points: int = 100,
                         frames_per_call: Optional[int] = None, engine: Optional[Engine] = None,
                         pairs: bool = False) -> TrajectoryInterfaceResult:
    """Buried surface area along an MD trajectory.  ``xyz`` (F, N, 3) frames (any array, a numpy memmap included: blocks of
    frames are copied into page-locked staging), ``radii`` (N,) and ``group`` (N,) labels shared by every frame; ``seg_be``
    (G, 2) residue ranges within a frame and ``seg_polar`` (G,) their polar flags, both optional.

    Frames go through ``Batch.submit_groups_frames_host`` in blocks of ``frames_per_call`` (default: the whole trajectory when
    it fits 256 MB of staging, else as many frames as do).  Two batches alternate, so the next block is staged and submitted
    before the current one is waited for: the host copy of block k + 1 and its transfer overlap the kernels of block k, and a
    trajectory of any length runs with bounded memory.  The results equal one ``run_groups_frames_host`` over all frames bit
    for bit.

    ``pairs=True`` adds, per frame, how much of every group each other group buries (and per residue, with residue ranges),
    summed on the device by ``Batch.submit_group_pairs_frames_host``: the labels are numbered 0 .. L - 1 in ascending order, and
    more than 17 distinct labels raise ValueError."""
    eng = engine or default_engine()
    if not isinstance(xyz, np.ndarray):
        xyz = np.asarray(xyz, np.float32)
    if xyz.ndim != 3 or xyz.shape[2] != 3:
        raise ValueError(f"xyz must be (F, N, 3), got {xyz.shape}")
    F, N = int(xyz.shape[0]), int(xyz.shape[1])
    radii = np.ascontiguousarray(radii, np.float32).reshape(-1)
    group = np.ascontiguousarray(group, np.uint32).reshape(-1)
    if radii.shape[0] != N or group.shape[0] != N:
        raise ValueError(f"radii and group need one value per atom of a frame ({N}), got {radii.shape[0]} and {group.shape[0]}")
    seg = None if seg_be is None else np.ascontiguousarray(seg_be, np.uint32).reshape(-1, 2)
    pol = None if seg_polar is None or seg is None else np.ascontiguousarray(seg_polar, np.uint8).reshape(-1)
    G = 0 if seg is None else seg.shape[0]
    labels = None
    if pairs:
        labels, dense = np.unique(group, return_inverse=True)
        if labels.shape[0] > 17:
            raise ValueError(f"pairs=True supports at most 17 distinct group labels, got {labels.shape[0]}")
        group = dense.astype(np.uint32).reshape(-1)
    L = 1 if labels is None else max(1, labels.shape[0])
    if frames_per_call is None:
        frames_per_call = max(1, _TRAJECTORY_STAGING_BYTES // max(1, N * 12))
    B = max(1, min(int(frames_per_call), F))
    want = ("protein", "seg") if G else ("protein",)
    out = TrajectoryInterfaceResult(np.zeros((F, 3), np.float32), np.zeros((F, 3), np.float32), np.zeros(F, np.float32),
                                    np.zeros((F, G), np.float32) if G else None, np.zeros((F, G), np.float32) if G else None)
    if pairs:
        out.pair_labels = labels
        out.pair_area = np.zeros((F, L, L), np.float64)
        out.seg_pair_area = np.zeros((F, G, L), np.float64) if G else None
    if F == 0:
        return out

    class _Slot:   # one batch of `fb` frames with its staging and page-locked outputs
        def __init__(self, fb):
            self.fb = fb
            topo = (np.tile(seg, (fb, 1)), (np.arange(fb + 1) * G).astype(np.uint64),
                    None if pol is None else np.tile(pol, fb)) if G else (None, None, None)
            self.batch = Batch(eng, (np.arange(fb + 1) * N).astype(np.uint64), *topo)
            self.stage = eng.pinned_empty((fb, N, 3), np.float32)
            self.res = (self.batch._host_outputs(want, "pinned"), self.batch._host_outputs(want, "pinned"))
            if pairs:
                self.res += (self.batch._pair_sums(L, True, "pinned"),)

    slots = {}

    def slot_for(k, fb):
        key = (k % 2, fb)
        if key not in slots:
            slots[key] = _Slot(fb)
        return slots[key]

    blocks = [(f0, min(f0 + B, F)) for f0 in range(0, F, B)]

    def submit(k):
        f0, f1 = blocks[k]
        s = slot_for(k, f1 - f0)
        np.copyto(s.stage, xyz[f0:f1], casting="same_kind")
        if pairs:
            return s, s.batch.submit_group_pairs_frames_host(s.stage, radii, group, L, probe_radius, n_points, want=want, result=s.res)
        return s, s.batch.submit_groups_frames_host(s.stage, radii, group, probe_radius, n_points, want=want, result=s.res)

    pending = None
    try:
        pending = submit(0)
        for k in range(len(blocks)):
            s, job = pending
            pending = submit(k + 1) if k + 1 < len(blocks) else None
            cpx, iso, *sums = job.wait()
            f0, f1 = blocks[k]
            out.complex[f0:f1] = cpx.protein
            out.isolated[f0:f1] = iso.protein
            if G:
                out.complex_seg[f0:f1] = cpx.seg_sasa.reshape(f1 - f0, G)
                out.isolated_seg[f0:f1] = iso.seg_sasa.reshape(f1 - f0, G)
            if pairs:
                out.pair_area[f0:f1] = sums[0].pair_area
                if G:
                    out.seg_pair_area[f0:f1] = sums[0].seg_pair_area.reshape(f1 - f0, G, L)
    finally:
        if pending is not None:   # an error left a block in flight: its buffers stay alive until it is done
            try:
                pending[1].wait()
            except Exception:
                pass
        for s in slots.values():
            s.batch.close()
    out.buried[:] = out.isolated[:, 0] - out.complex[:, 0]
    return out


def _dense_classes(ids: np.ndarray) -> Optional[np.ndarray]:
    uniq, inv = np.unique(ids, return_inverse=True)
    return None if uniq.shape[0] == ids.shape[0] else inv.astype(np.uint32)


class SASAOptions:
    """``SASAOptions::<Level>::new()`` with the reference's ``with_*`` builder methods."""

    def __init__(self, level=ResidueLevel):
        self.level = level
        self.probe_radius = 1.4
        self.n_points = 100
        self.threads = -1
        self.include_hydrogens = False
        self.radii_config = None
        self.allow_vdw_fallback = False
        self.include_hetatms = False
        self.read_radii_from_occupancy = False

    # convenience constructors (src/options.rs:565-587)
    @classmethod
    def atom_level(cls): return cls(AtomLevel)
    @classmethod
    def residue_level(cls): return cls(ResidueLevel)
    @classmethod
    def chain_level(cls): return cls(ChainLevel)
    @classmethod
    def protein_level(cls): return cls(ProteinLevel)

    def with_probe_radius(self, radius): self.probe_radius = float(radius); return self
    def with_include_hetatms(self, v): self.include_hetatms = bool(v); return self
    def with_n_points(self, points): self.n_points = int(points); return self
    def with_read_radii_from_occupancy(self, v): self.read_radii_from_occupancy = bool(v); return self
    def with_threads(self, threads): self.threads = int(threads); return self
    def with_include_hydrogens(self, v): self.include_hydrogens = bool(v); return self
    def with_allow_vdw_fallback(self, v): self.allow_vdw_fallback = bool(v); return self

    def with_radii_file(self, path):
        try:
            self.radii_config = load_radii_from_file(path)
        except OSError as e:
            raise SASACalcError("RadiiFileLoad", f"Failed to load radii file: {e}") from e
        return self

    def _pack(self, st: Structure) -> PackedStructure:
        return build_atoms_and_mapping(st, self.level.name, self.radii_config, self.allow_vdw_fallback,
                                       self.include_hydrogens, self.include_hetatms, self.read_radii_from_occupancy)

    def process(self, st: Structure, engine: Optional[Engine] = None):
        """One structure -> the level's result type (src/options.rs:606-618)."""
        return self.process_many([st], engine)[0]

    def process_many(self, structures: Sequence[Structure], engine: Optional[Engine] = None) -> List:
        """Batched form: all structures go through ONE pipelined batch call.  A structure whose extraction
        fails is reported as its ``SASACalcError`` in the result list (directory mode logs and continues,
        src/main.rs:447-453)."""
        return self._run_many(structures, engine, None)

    def process_surface(self, structures: Sequence[Structure], engine: Optional[Engine] = None) -> List:
        """The dot surface: per structure a :class:`SurfaceResult` with the level's result and the solvent-accessible test
        points, both from ONE batch call with exposed-point masks.  A structure whose extraction fails is reported as its
        ``SASACalcError``, as in ``process_many``."""
        return self._run_many(structures, engine, None, surface=True)

    def process_interface(self, structures: Sequence[Structure], chain_groups: Optional[Sequence[str]] = None,
                          engine: Optional[Engine] = None) -> List:
        """Buried surface area: per structure an :class:`InterfaceResult` with the level's result in the complex and
        with every chain group standing alone (only atoms of its own group occlude an atom), both from ONE grouped batch
        call.  ``chain_groups``: strings of chain ids, e.g. ``["AB", "C"]`` puts chains A and B in one group; a chain not
        listed is a group of its own; None: one group per chain.  Chains are keyed by chain id across models.  A structure
        whose extraction fails is reported as its ``SASACalcError``, as in ``process_many``."""
        return self._run_many(structures, engine, list(chain_groups) if chain_groups is not None else [])

    def process_interface_surface(self, structures: Sequence[Structure], chain_groups: Optional[Sequence[str]] = None,
                                  engine: Optional[Engine] = None) -> List:
        """Interface patches: per structure an :class:`InterfaceSurfaceResult` with what ``process_interface`` gives for the
        same arguments and the buried test points -- exposed with the atom's chain group standing alone, buried in the complex
        -- all from ONE grouped batch call with exposed-point masks.  Chain grouping and error reporting are those of
        ``process_interface``."""
        return self._run_many(structures, engine, list(chain_groups) if chain_groups is not None else [], surface=True)

    def process_interface_pairs(self, structures: Sequence[Structure], chain_groups: Optional[Sequence[str]] = None,
                                max_partners: int = 4, engine: Optional[Engine] = None) -> List:
        """Pairwise interfaces: per structure an :class:`InterfacePairsResult` with what ``process_interface`` gives for the
        same arguments, one :class:`GroupPairResult` per contacting pair of chain groups, and at residue level the buried area
        of every residue by each partner group -- all from ONE grouped batch call with ``max_partners`` partner slots per atom
        (rerun once with as many slots as the batch needs when an atom has more partners; an atom with more than 16 partners
        raises the run's :class:`SasaB200Error`).  Chain grouping and error reporting are those of ``process_interface``."""
        return self._run_many(structures, engine, list(chain_groups) if chain_groups is not None else [],
                              max_partners=int(max_partners))

    @staticmethod
    def _chain_groups(atom_chain: np.ndarray, chain_groups: List[str]) -> np.ndarray:
        """Dense per-atom group labels of one structure."""
        label = {}
        for g, ids in enumerate(chain_groups):
            for c in ids:
                label.setdefault(c, g)
        out = np.empty(atom_chain.shape[0], np.uint32)
        for i, c in enumerate(atom_chain):
            if c not in label:
                label[c] = len(chain_groups) + len(label)
            out[i] = label[c]
        return out

    @staticmethod
    def _pairs_result(interface: InterfaceResult, p: PackedStructure, group: np.ndarray, partner: np.ndarray, area: np.ndarray,
                      level: str) -> InterfacePairsResult:
        chains = {}
        for g, c in zip(group.tolist(), p.atom_chain):
            if c not in chains.setdefault(g, ""):
                chains[g] += c
        table = group_pair_table(partner, area, group, [0, group.shape[0]])[0]
        rows = [GroupPairResult(a, b, chains.get(a, ""), chains.get(b, ""), ab, ba) for a, b, ab, ba in table]
        residue = None
        if level == "residue":
            residue = []
            for b0, b1 in p.seg_be.tolist():
                acc = {}
                for i in range(b0, b1):
                    for h, v in zip(partner[i].tolist(), area[i].tolist()):
                        if h != 0xFFFFFFFF or v > 0:
                            acc[h] = acc.get(h, 0.0) + v
                residue.append(acc)
        return InterfacePairsResult(interface, rows, residue)

    def _run_many(self, structures: Sequence[Structure], engine: Optional[Engine], chain_groups: Optional[List[str]],
                  surface: bool = False, max_partners: Optional[int] = None) -> List:
        eng = engine or default_engine()
        packed: List[Optional[PackedStructure]] = []
        results: List = [None] * len(structures)
        for i, st in enumerate(structures):
            try:
                packed.append(self._pack(st))
            except SASACalcError as e:
                packed.append(None)
                results[i] = e
        good = [i for i, p in enumerate(packed) if p is not None]
        if not good:
            return results
        xyzr = np.concatenate([packed[i].xyzr for i in good]) if good else np.zeros((0, 4), np.float32)
        struct_off = np.cumsum([0] + [packed[i].xyzr.shape[0] for i in good]).astype(np.uint64)
        seg_be = np.concatenate([packed[i].seg_be for i in good]).astype(np.uint32)
        seg_off = np.cumsum([0] + [packed[i].seg_be.shape[0] for i in good]).astype(np.uint64)
        polar = np.concatenate([packed[i].seg_polar for i in good]).astype(np.uint8)
        # Atom.id equality classes (atoms with equal ids never occlude each other); None when all distinct
        cls_parts, base, any_dup = [], 0, False
        for i in good:
            c = _dense_classes(packed[i].ids)
            any_dup = any_dup or c is not None
            n = packed[i].ids.shape[0]
            cls_parts.append((np.arange(n, dtype=np.uint32) if c is None else c) + np.uint32(base))
            base += n
        id_class = np.concatenate(cls_parts) if any_dup else None
        level = self.level.name
        want = {"atom": ("atom",), "residue": ("seg",), "chain": ("seg",), "protein": ("protein",)}[level]
        batch = Batch(eng, struct_off, seg_be if seg_be.shape[0] else None, seg_off if seg_be.shape[0] else None,
                      polar if seg_be.shape[0] else None)
        try:
            if chain_groups is None:
                run = batch.run_masks_host if surface else batch.run_host
                res = run(xyzr, id_class, self.probe_radius, self.n_points, want=want)
            else:   # the protein totals give the buried area: always requested
                group = np.concatenate([self._chain_groups(packed[i].atom_chain, chain_groups) for i in good])
                gwant = tuple(set(want) | {"protein"})
                if max_partners is not None:
                    try:
                        cpx, iso, pairs = batch.run_group_pairs_host(xyzr, group, id_class, self.probe_radius, self.n_points,
                                                                     want=gwant, max_partners=max_partners)
                    except SasaB200Error as e:
                        if not max_partners < getattr(e, "needed", 0) <= 16:   # (a run holds at most 16 slots per atom)
                            raise
                        cpx, iso, pairs = batch.run_group_pairs_host(xyzr, group, id_class, self.probe_radius, self.n_points,
                                                                     want=gwant, max_partners=e.needed)
                else:
                    run = batch.run_groups_masks_host if surface else batch.run_groups_host
                    cpx, iso = run(xyzr, group, id_class, self.probe_radius, self.n_points, want=gwant)
        finally:
            batch.close()

        def level_result(res, k, p):
            a0, a1 = int(struct_off[k]), int(struct_off[k + 1])
            g0, g1 = int(seg_off[k]), int(seg_off[k + 1])
            if level == "atom":
                return res.atom_sasa[a0:a1].copy()
            if level == "residue":
                return [ResidueResult(m["serial_number"], m["insertion_code"], float(v), m["name"],
                                      m["is_polar"], m["chain_id"])
                        for m, v in zip(p.seg_meta, res.seg_sasa[g0:g1])] if g1 > g0 else []
            if level == "chain":
                return [ChainResult(m["name"], float(v)) for m, v in zip(p.seg_meta, res.seg_sasa[g0:g1])] \
                    if g1 > g0 else []
            t = res.protein[k]
            return ProteinResult(float(t[0]), float(t[1]), float(t[2]))

        for k, i in enumerate(good):
            a0, a1 = int(struct_off[k]), int(struct_off[k + 1])
            if chain_groups is None and surface:
                pts, atom = surface_points(xyzr[a0:a1], res.exposed[a0:a1], self.n_points, self.probe_radius)
                results[i] = SurfaceResult(level_result(res, k, packed[i]), pts, atom)
            elif chain_groups is None:
                results[i] = level_result(res, k, packed[i])
            else:
                r = InterfaceResult(level_result(cpx, k, packed[i]), level_result(iso, k, packed[i]),
                                    float(iso.protein[k, 0]) - float(cpx.protein[k, 0]))
                if surface:
                    buried = iso.exposed[a0:a1] & ~cpx.exposed[a0:a1]
                    pts, atom = surface_points(xyzr[a0:a1], buried, self.n_points, self.probe_radius)
                    r = InterfaceSurfaceResult(r, pts, atom)
                if max_partners is not None:
                    r = self._pairs_result(r, packed[i], group[a0:a1], pairs.partner[a0:a1], pairs.buried_area[a0:a1], level)
                results[i] = r
        return results
