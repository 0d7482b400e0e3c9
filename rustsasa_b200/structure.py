"""Minimal PDB / mmCIF ATOM-record reader and the atom-extraction step (row A0).

This is host-side glue that sits *in front of* the hot path: it turns a structure file
into the packed float4 atoms + contiguous segment ranges the C ABI consumes.  It follows
the ordering and filtering rules of the reference's extraction layer so that the atom
order (and therefore every per-atom output) lines up with RustSASA's:

* hierarchy and first-seen ordering -- pdbtbx ``read/pdb/parser.rs:144-251`` (chains and
  residues kept in insertion order per model, conformers keyed by (residue name, alt-loc)),
  ``read/mmcif/parser.rs:456-600`` (auth_asym_id / auth_seq_id with label_* fallback,
  serial number = running atom count per model);
* blank alt-loc atoms are appended to every other conformer --
  ``pdbtbx/src/validate.rs:302-325`` (``reshuffle_conformers``);
* extraction -- ``src/options.rs:81-116`` (``build_atom!``) and the four
  ``build_atoms_and_mapping`` bodies (``:151-189, :234-287, :317-365, :412-464``):
  all models, first conformer only, hydrogens / HETATM filtered, radius from
  occupancy | custom | ProtOr | vdW fallback | ``RadiusMissing``.

It is not a general structure parser (no symmetry, no bonds, no validation).
"""
from __future__ import annotations

import os
import shlex
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np

# Alvarez (2013) van der Waals radii as tabulated by pdbtbx/src/structs/elements.rs:631-647+
VDW_RADII = {
    "H": 1.2, "HE": 1.43, "LI": 2.12, "BE": 1.98, "B": 1.91, "C": 1.77, "N": 1.66, "O": 1.5,
    "F": 1.46, "NE": 1.58, "NA": 2.5, "MG": 2.51, "AL": 2.25, "SI": 2.19, "P": 1.9, "S": 1.89,
    "CL": 1.82, "AR": 1.83, "K": 2.73, "CA": 2.62, "SC": 2.58, "TI": 2.46, "V": 2.42, "CR": 2.45,
    "MN": 2.45, "FE": 2.44, "CO": 2.4, "NI": 2.4, "CU": 2.38, "ZN": 2.39, "GA": 2.32, "GE": 2.29,
    "AS": 1.88, "SE": 1.82, "BR": 1.86, "KR": 2.25,
}
_ELEMENTS = set(
    "H HE LI BE B C N O F NE NA MG AL SI P S CL AR K CA SC TI V CR MN FE CO NI CU ZN GA GE AS SE BR KR RB SR Y ZR "
    "NB MO TC RU RH PD AG CD IN SN SB TE I XE CS BA LA CE PR ND PM SM EU GD TB DY HO ER TM YB LU HF TA W RE OS IR "
    "PT AU HG TL PB BI PO AT RN FR RA AC TH PA U NP PU AM CM BK CF ES FM MD NO LR RF DB SG BH HS MT DS RG CN NH FL "
    "MC LV TS OG".split())

# src/utils/consts.rs:7-16
POLAR_AMINO_ACIDS = frozenset({"SER", "THR", "CYS", "ASN", "GLN", "TYR"})

_PROTOR_PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "radii", "protor.config")


class SASACalcError(Exception):
    """Mirrors ``SASACalcError`` (src/options.rs:466-494); ``kind`` is the variant name."""

    def __init__(self, kind: str, message: str):
        super().__init__(message)
        self.kind = kind


def parse_radii_config(content: str) -> Dict[str, Dict[str, float]]:
    """FreeSASA-style classifier file -> {residue: {atom: radius}} (src/utils/consts.rs:31-81)."""
    types: Dict[str, float] = {}
    atoms: Dict[str, Dict[str, float]] = {}
    section = None
    for raw in content.splitlines():
        line = raw.strip()
        if not line or line.startswith("#") or line.startswith("name:"):
            continue
        if line == "types:":
            section = "types"
            continue
        if line == "atoms:":
            section = "atoms"
            continue
        parts = line.split()
        if section == "types" and len(parts) >= 2:
            try:
                types[parts[0]] = float(np.float32(parts[1]))
            except ValueError:
                pass
        elif section == "atoms" and len(parts) >= 3 and parts[2] in types:
            atoms.setdefault(parts[0], {})[parts[1]] = types[parts[2]]
    return atoms


def load_radii_from_file(path: str) -> Dict[str, Dict[str, float]]:
    with open(path, "r") as fh:
        return parse_radii_config(fh.read())


_PROTOR: Optional[Dict[str, Dict[str, float]]] = None


def protor_radii() -> Dict[str, Dict[str, float]]:
    global _PROTOR
    if _PROTOR is None:
        _PROTOR = load_radii_from_file(_PROTOR_PATH)
    return _PROTOR


def get_protor_radius(residue: str, atom: str) -> Optional[float]:
    """src/utils.rs:35-37."""
    return protor_radii().get(residue, {}).get(atom)


def get_radius(residue: str, atom: str, radii_config=None) -> Optional[float]:
    """Custom table first, then ProtOr (src/utils.rs:40-56)."""
    if radii_config is not None:
        r = radii_config.get(residue, {}).get(atom)
        if r is not None:
            return r
    return get_protor_radius(residue, atom)


def serialize_chain_id(s: str) -> int:
    """src/utils.rs:24-33 (lossy: letters only, A->1 .. Z->26, base-10 fold)."""
    result = 0
    for c in s:
        if c.isascii() and c.isalpha():
            result = result * 10 + (ord(c.upper()) - 64)
    return result


@dataclass
class AtomRec:
    hetero: bool
    serial: int
    name: str
    x: float
    y: float
    z: float
    occupancy: float
    element: Optional[str]


@dataclass
class Conformer:
    name: str
    altloc: Optional[str]
    atoms: List[AtomRec] = field(default_factory=list)


@dataclass
class Residue:
    serial: int
    icode: Optional[str]
    conformers: List[Conformer] = field(default_factory=list)

    def name(self) -> Optional[str]:
        names = {c.name for c in self.conformers}
        return next(iter(names)) if len(names) == 1 else None


@dataclass
class Chain:
    id: str
    residues: Dict[Tuple[int, Optional[str]], Residue] = field(default_factory=dict)


@dataclass
class Model:
    serial: int
    chains: Dict[str, Chain] = field(default_factory=dict)
    atom_count: int = 0


@dataclass
class Structure:
    models: List[Model] = field(default_factory=list)

    def chains(self):
        for m in self.models:
            yield from m.chains.values()

    def residues(self):
        for c in self.chains():
            yield from c.residues.values()

    def atoms(self):
        """pdb.atoms(): every atom of every conformer, hierarchy order."""
        for r in self.residues():
            for conf in r.conformers:
                yield from conf.atoms


def _element(element: str, atom_name: str) -> Optional[str]:
    """pdbtbx Atom::new element resolution (structs/atom.rs:74-87)."""
    e = element.strip().upper()
    if e in _ELEMENTS:
        return e
    n = atom_name.strip().upper()
    if n in _ELEMENTS:
        return n
    if n and n[0] in "CHNOS":
        return n[0]
    return None


def _add_atom(model: Model, chain_id: str, res_key, conf_key, atom: AtomRec) -> None:
    chain = model.chains.get(chain_id)
    if chain is None:
        chain = model.chains[chain_id] = Chain(chain_id)
    res = chain.residues.get(res_key)
    if res is None:
        res = chain.residues[res_key] = Residue(res_key[0], res_key[1])
    for conf in res.conformers:
        if (conf.name, conf.altloc) == conf_key:
            conf.atoms.append(atom)
            break
    else:
        res.conformers.append(Conformer(conf_key[0], conf_key[1], [atom]))
    model.atom_count += 1


def _reshuffle_conformers(st: Structure) -> None:
    for res in st.residues():
        if len(res.conformers) > 1:
            blank = None
            for i, c in enumerate(res.conformers):
                if c.altloc is None:
                    blank = i
            if blank is not None:
                shared = res.conformers.pop(blank)
                count = len(res.conformers) + 1
                for c in res.conformers:
                    c.atoms.extend(
                        AtomRec(a.hetero, a.serial, a.name, a.x, a.y, a.z, a.occupancy / count, a.element)
                        for a in shared.atoms
                    )


def read_pdb(path: str) -> Structure:
    st = Structure()
    model = Model(0)
    serial_add = 0
    res_add = 0
    last_serial = -1
    last_res = -1
    # blank chain IDs take the letter of an 'A'..'Z' cycle advanced by every TER record and never reset
    # (pdbtbx/src/read/pdb/parser.rs:113-115, :176-180, :511)
    chain_letter = 0
    model_no = 0
    with open(path, "r", errors="replace") as fh:
        for line in fh:
            line = line.rstrip("\r\n")
            if len(line) <= 6:          # short lines: only TER counts (pdbtbx lexer.rs:87-91)
                if line[:3] == "TER":
                    chain_letter = (chain_letter + 1) % 26
                continue
            rec = line[:6]
            if rec in ("ATOM  ", "HETATM"):
                line = line.rstrip("\n").ljust(80)
                try:
                    serial = int(line[6:11])
                except ValueError:
                    serial = 0
                name = line[12:16].strip().upper()
                alt = line[16]
                resname = line[17:20].strip().upper()
                chain_id = line[21]
                resseq = int(line[22:26])
                icode = line[26]
                x, y, z = float(line[30:38]), float(line[38:46]), float(line[46:54])
                occ_s = line[54:60].strip()
                occ = float(occ_s) if occ_s else 1.0
                if serial == 0 and last_serial == 99_999:
                    serial_add += 100_000
                if resseq == 0 and last_res == 9999:
                    res_add += 10000
                atom = AtomRec(rec == "HETATM", serial + serial_add, name, x, y, z, occ,
                               _element(line[76:78], name))
                _add_atom(model, chain_id if chain_id.strip() else chr(ord("A") + chain_letter),
                          (resseq + res_add, None if icode == " " else icode),
                          (resname, None if alt == " " else alt), atom)
                last_serial, last_res = serial, resseq
            elif rec == "MODEL ":
                # closed by the NEXT MODEL record (or MASTER, or the end of the file); ENDMDL is ignored (parser.rs:282-306)
                model.serial = model_no
                if model.chains:
                    st.models.append(model)
                try:
                    model_no = int(line[6:].strip())
                except ValueError:
                    model_no = 0
                model = Model(model_no)
            elif rec == "MASTER":
                model.serial = model_no
                if model.chains:
                    st.models.append(model)
                model = Model(model_no)
            elif rec == "TER   ":
                chain_letter = (chain_letter + 1) % 26
    model.serial = model_no
    if model.chains:
        st.models.append(model)
    _reshuffle_conformers(st)
    return st


def _cif_tokens(line: str) -> List[str]:
    if "'" in line or '"' in line:
        return shlex.split(line, posix=True)
    return line.split()


def read_mmcif(path: str) -> Structure:
    st = Structure()
    models: Dict[int, Model] = {}
    with open(path, "r", errors="replace") as fh:
        lines = fh.read().splitlines()
    i = 0
    n = len(lines)
    while i < n:
        if lines[i].strip() == "loop_" and i + 1 < n and lines[i + 1].strip().startswith("_atom_site."):
            i += 1
            cols = []
            while i < n and lines[i].strip().startswith("_atom_site."):
                cols.append(lines[i].strip().split(".", 1)[1])
                i += 1
            col = {c: k for k, c in enumerate(cols)}

            def get(tok, key):
                k = col.get(key)
                if k is None:
                    return None
                v = tok[k]
                return None if v in (".", "?") else v

            while i < n:
                s = lines[i].strip()
                if not s or s.startswith("#") or s.startswith("_") or s == "loop_":
                    break
                tok = _cif_tokens(s)
                i += 1
                if len(tok) < len(cols):
                    continue
                model_no = int(get(tok, "pdbx_PDB_model_num") or 1)
                model = models.get(model_no)
                if model is None:
                    model = models[model_no] = Model(model_no)
                    st.models.append(model)
                group = get(tok, "group_PDB") or "ATOM"
                name = (get(tok, "label_atom_id") or "").upper()
                resname = (get(tok, "label_comp_id") or "").upper()
                seq = get(tok, "auth_seq_id") or get(tok, "label_seq_id")
                resseq = int(seq) if seq is not None else 0
                chain_id = get(tok, "auth_asym_id") or get(tok, "label_asym_id")
                occ = get(tok, "occupancy")
                atom = AtomRec(group == "HETATM", model.atom_count, name,
                               float(get(tok, "Cartn_x")), float(get(tok, "Cartn_y")), float(get(tok, "Cartn_z")),
                               float(occ) if occ is not None else 1.0,
                               _element(get(tok, "type_symbol") or "", name))
                _add_atom(model, chain_id, (resseq, get(tok, "pdbx_PDB_ins_code")),
                          (resname, get(tok, "label_alt_id")), atom)
            continue
        i += 1
    _reshuffle_conformers(st)
    return st


def read_structure(path: str) -> Structure:
    ext = os.path.splitext(path)[1].lower()
    if ext in (".cif", ".mmcif"):
        return read_mmcif(path)
    return read_pdb(path)


@dataclass
class PackedStructure:
    """Output of row A0: what the C ABI consumes for one structure."""

    xyzr: np.ndarray            # (N, 4) float32: x, y, z, radius
    ids: np.ndarray             # (N,) uint64 atom ids (only equality matters)
    seg_be: np.ndarray          # (n_seg, 2) uint32 [begin, end) atom ranges, relative to atom 0
    seg_polar: np.ndarray       # (n_seg,) uint8, residue-level polar flag
    seg_meta: list              # per segment: dict of the host-side result fields
    atom_chain: Optional[np.ndarray] = None   # (N,) chain id of every atom (str), the key of grouped runs


def build_atoms_and_mapping(st: Structure, level: str = "residue", radii_config=None, allow_vdw_fallback=False,
                            include_hydrogens=False, include_hetatms=False,
                            read_radii_from_occupancy=False) -> PackedStructure:
    """Flatten a structure into packed atoms + contiguous segment ranges.

    ``level`` in {"atom", "residue", "chain", "protein"}.  Key collisions follow the
    reference's ``HashMap::insert`` (last writer wins): a later residue / chain with the
    same key replaces the range every earlier holder of that key reports.
    """
    xyzr: List[Tuple[float, float, float, float]] = []
    ids: List[int] = []
    atom_chain: List[str] = []
    key_to_range: Dict[object, Tuple[int, int]] = {}
    order: List[Tuple[object, dict]] = []

    def push(atom: AtomRec, resname: str, altloc: str, chain_id: str) -> bool:
        if atom.element is None:
            raise SASACalcError("ElementMissing", "Element missing for atom")
        if atom.element == "H" and not include_hydrogens:
            return False
        if atom.hetero and not include_hetatms:
            return False
        if read_radii_from_occupancy:
            radius = np.float32(atom.occupancy)
        else:
            r = get_radius(resname, atom.name, radii_config)
            if r is None:
                if allow_vdw_fallback:
                    r = VDW_RADII.get(atom.element)
                    if r is None:
                        raise SASACalcError("VanDerWaalsMissing", "Van der Waals radius missing for element")
                else:
                    raise SASACalcError(
                        "RadiusMissing",
                        f"Radius not found for residue '{resname}' atom '{atom.name}' of type '{atom.element}'.")
            radius = np.float32(r)
        xyzr.append((np.float32(atom.x), np.float32(atom.y), np.float32(atom.z), radius))
        # id = FNV(altloc, serial): only equality is observable, so a tuple hash stands in.
        ids.append(hash((altloc, atom.serial)) & 0xFFFFFFFFFFFFFFFF)
        atom_chain.append(chain_id)
        return True

    if level == "atom":
        for chain in st.chains():   # (st.residues() order)
            for res in chain.residues.values():
                resname = res.name()
                if resname is None:
                    raise SASACalcError("FailedToGetResidueName", "Failed to get residue name")
                if res.conformers:
                    conf = res.conformers[0]
                    for a in conf.atoms:
                        push(a, resname, conf.altloc or "", chain.id)
    else:
        for chain in st.chains():
            chain_key = serialize_chain_id(chain.id)
            chain_begin = len(xyzr)
            for res in chain.residues.values():
                resname = res.name()
                if resname is None:
                    raise SASACalcError("FailedToGetResidueName", "Failed to get residue name")
                begin = len(xyzr)
                if res.conformers:
                    conf = res.conformers[0]
                    for a in conf.atoms:
                        push(a, resname, "" if level == "protein" else (conf.altloc or ""), chain.id)
                    if level in ("residue", "protein"):
                        key_to_range[(chain.id, res.serial, res.icode or "")] = (begin, len(xyzr))
                if level in ("residue", "protein"):
                    order.append(((chain.id, res.serial, res.icode or ""),
                                  dict(serial_number=res.serial, insertion_code=res.icode or "", name=resname,
                                       is_polar=resname in POLAR_AMINO_ACIDS, chain_id=chain.id)))
            if level == "chain":
                key_to_range[chain_key] = (chain_begin, len(xyzr))
                order.append((chain_key, dict(name=chain.id)))

    seg_be = np.zeros((len(order), 2), dtype=np.uint32)
    seg_polar = np.zeros(len(order), dtype=np.uint8)
    meta = []
    for k, (key, m) in enumerate(order):
        if key not in key_to_range:
            raise SASACalcError("AtomMapToLevelElementFailed", "Failed to map atoms back to level element")
        seg_be[k] = key_to_range[key]
        seg_polar[k] = 1 if m.get("is_polar") else 0
        meta.append(m)
    arr = np.asarray(xyzr, dtype=np.float32).reshape(-1, 4)
    return PackedStructure(arr, np.asarray(ids, dtype=np.uint64), seg_be, seg_polar, meta, np.asarray(atom_chain, dtype=object))
