"""Exposed-point masks: sasa_b200_batch_run_masks_host / _device.

Every mask row must equal the CPU oracle's (tests/mask_oracle.py, the reference's arithmetic point by point) bit for bit, and
the other outputs must equal a plain run's bit for bit, on every kernel path: the fused kernel for n_points <= 128 (pairs of
atoms and single atoms), the fused chunked-table kernel, the large-structure cells / atoms kernels, id classes, the streaming
routine and the cold paths, the statistics and forced-streaming flags.
"""
import ctypes as C

import numpy as np
import pytest

from tests.mask_oracle import exposed_masks

pytestmark = pytest.mark.gpu

PROBE = 1.4
ALL = ("counts", "atom", "seg", "protein")


@pytest.fixture(scope="module")
def eng():
    from rustsasa_b200 import Engine
    e = Engine()
    yield e
    e.close()


def popcount_rows(m):
    return np.unpackbits(np.ascontiguousarray(m, np.uint32).view(np.uint8), axis=1).sum(axis=1).astype(np.uint32)


def same_outputs(a, b):
    for f in ("counts", "atom_sasa", "seg_sasa", "protein"):
        x, y = getattr(a, f), getattr(b, f)
        assert (x is None) == (y is None), f
        if x is not None:
            assert np.array_equal(x, y, equal_nan=f != "counts"), f


def check_run(b, xyzr, oracle, structs, n_points=100, lanes=8, probe=PROBE, cls=None, ids=None, flags=0, want=("counts", "atom")):
    """Masked run against the plain run (outputs) and the oracle (masks, per structure); returns (masked, plain)."""
    plain = b.run_host(xyzr, cls, probe, n_points, lanes, flags, want=want)
    got = b.run_masks_host(xyzr, cls, probe, n_points, lanes, flags, want=want)
    same_outputs(got, plain)
    W = (n_points + 31) // 32
    assert got.exposed.shape == (xyzr.shape[0], W) and got.exposed.dtype == np.uint32
    if got.counts is not None:
        assert np.array_equal(popcount_rows(got.exposed), got.counts)
    if n_points % 32:
        assert not np.any(got.exposed[:, -1] >> np.uint32(n_points % 32))
    a0 = 0
    for i, s in enumerate(structs):
        a1 = a0 + s.shape[0]
        want_m = exposed_masks(oracle, s, probe, n_points, lanes, ids=None if ids is None else ids[i])
        assert np.array_equal(got.exposed[a0:a1], want_m), (i, n_points, lanes)
        a0 = a1
    return got, plain


def golden_batch(eng, golden, names):
    ss = [golden.structure(n) for n in names]
    off = np.cumsum([0] + [s["xyzr"].shape[0] for s in ss]).astype(np.uint64)
    seg_off = np.cumsum([0] + [len(s["seg_be"]) for s in ss]).astype(np.uint64)
    b = eng.batch(off, np.concatenate([s["seg_be"] for s in ss]), seg_off, np.concatenate([s["polar"] for s in ss]))
    return b, [s["xyzr"] for s in ss]


@pytest.mark.parametrize("n_points", [100, 960])
def test_golden_structures(eng, oracle, golden, n_points):
    b, structs = golden_batch(eng, golden, golden.names)
    r, _ = check_run(b, np.concatenate(structs), oracle, structs, n_points, want=ALL)
    assert r.stats["streamed_atoms"] == 0
    b.close()


@pytest.mark.parametrize("n_points,lanes", [(1, 8), (37, 4), (96, 16), (100, 4), (100, 16), (128, 8), (129, 16), (200, 4),
                                            (960, 16), (1024, 8), (1025, 4), (1100, 16)])
def test_body_tail_splits(eng, oracle, golden, n_points, lanes):
    names = ["example.cif", "2drt", "4xfj"]
    b, structs = golden_batch(eng, golden, names)
    check_run(b, np.concatenate(structs), oracle, structs, n_points, lanes, want=ALL)
    b.close()


@pytest.mark.parametrize("n_points", [1, 37, 100, 128, 129, 960])
@pytest.mark.parametrize("seed", range(3))
def test_randomised_geometry(eng, oracle, seed, n_points):
    rng = np.random.default_rng(9100 + 10 * seed + n_points)
    lanes = int(rng.choice([4, 8, 16]))
    probe = float(rng.choice([0.0, 1.4, 3.0]))
    structs = []
    for t in range(8):
        n = int(rng.integers(1, 700))
        density = float(rng.choice([0.005, 0.03, 0.057, 0.12]))
        side = (n / density) ** (1.0 / 3.0)
        xyz = rng.uniform(0.0, side, size=(n, 3)) + rng.uniform(-300, 300, size=3)
        rad = rng.uniform(0.4, 3.2, size=n) if t % 2 else rng.choice([1.42, 1.61, 1.76, 1.88], size=n)
        if n > 20:
            xyz[1] = xyz[0]
            xyz[3] = xyz[2] + 1e-4
            rad[7], xyz[7] = 3.2, xyz[6] + 0.2
        structs.append(np.concatenate([xyz, rad[:, None]], axis=1).astype(np.float32))
    off = np.cumsum([0] + [s.shape[0] for s in structs]).astype(np.uint64)
    b = eng.batch(off)
    check_run(b, np.concatenate(structs), oracle, structs, n_points, lanes, probe)
    b.close()


def _cluster(rng, n, side):
    xyz = rng.uniform(0.0, side, size=(n, 3))
    return np.concatenate([xyz, rng.uniform(1.2, 2.0, size=(n, 1))], axis=1).astype(np.float32)


def _classes(ids, off):
    return np.concatenate([np.unique(ids[i], return_inverse=True)[1].astype(np.uint32) + np.uint32(off[i]) for i in range(len(ids))])


@pytest.mark.parametrize("n_points", [100, 960])
@pytest.mark.parametrize("with_cls", [False, True])
def test_large_dense_and_elongated(eng, oracle, n_points, with_cls):
    """A structure above the fused kernels' capacity (large-structure path), a dense cluster (more than 96 neighbours per atom:
    the streaming routine), and two protein-density clusters 3,000 A apart (the grid's cells grow until every cell's candidate
    list overflows: the fused kernel's cold path), with and without duplicate ids."""
    rng = np.random.default_rng(41 + with_cls + n_points)
    big = _cluster(rng, 40000, 95.0)
    dense = _cluster(rng, 600, 12.0)
    pair = np.concatenate([_cluster(rng, 500, 20.6), _cluster(rng, 500, 20.6) + np.array([3000, 0, 0, 0], np.float32)])
    structs = [dense, big, pair]
    off = np.cumsum([0] + [s.shape[0] for s in structs]).astype(np.uint64)
    ids = [rng.integers(0, s.shape[0] // 2, size=s.shape[0]).astype(np.uint64) for s in structs] if with_cls else None
    cls = _classes(ids, off) if with_cls else None
    b = eng.batch(off)
    r, plain = check_run(b, np.concatenate(structs), oracle, structs, n_points, cls=cls, ids=ids)
    assert plain.stats["streamed_atoms"] > dense.shape[0] // 2
    # atoms the plain run sends through atom_fast stream in a masked run
    extra = r.stats["streamed_atoms"] - plain.stats["streamed_atoms"]
    if n_points <= 128:
        assert extra > pair.shape[0] // 2     # the clusters' cells overflow the fused kernel's candidate list: cold atoms
    elif with_cls:
        assert extra >= big.shape[0]          # id classes above 128 points on the large path
    else:
        assert extra == 0                     # the chunked-table kernels have no list cap
    b.close()


def test_pair_path_and_duplicate_ids(eng, oracle, golden):
    """The fused kernel with id classes (no atom pairs) next to the plain pairs path on the same structures."""
    s = golden.structure("2drt")["xyzr"]
    two = np.concatenate([s, s + np.array([0.3, 0, 0, 0], np.float32)])
    n = s.shape[0]
    ids = [np.concatenate([np.arange(n), np.arange(n)]).astype(np.uint64), np.arange(s.shape[0], dtype=np.uint64)]
    ids[1][1] = ids[1][0]
    structs = [two, s]
    off = np.cumsum([0] + [x.shape[0] for x in structs]).astype(np.uint64)
    b = eng.batch(off)
    check_run(b, np.concatenate(structs), oracle, structs, cls=_classes(ids, off), ids=ids)
    check_run(b, np.concatenate(structs), oracle, structs)
    b.close()


@pytest.mark.parametrize("n_points", [100, 960])
def test_flags_give_the_default_masks(eng, golden, n_points):
    from rustsasa_b200 import _lib
    rng = np.random.default_rng(5)
    structs = [golden.structure("example.cif")["xyzr"], _cluster(rng, 30000, 85.0)]
    off = np.cumsum([0] + [s.shape[0] for s in structs]).astype(np.uint64)
    xyzr = np.concatenate(structs)
    b = eng.batch(off)
    ref = b.run_masks_host(xyzr, n_points=n_points)
    for flags in (_lib.FLAG_FORCE_STREAMING, _lib.FLAG_BOUNDARY_STATS):
        plain = b.run_host(xyzr, n_points=n_points, flags=flags)
        got = b.run_masks_host(xyzr, n_points=n_points, flags=flags)
        same_outputs(got, plain)
        assert np.array_equal(got.exposed, ref.exposed), flags
        assert got.stats["boundary_points"] == plain.stats["boundary_points"]
        assert got.stats["streamed_atoms"] == xyzr.shape[0]
    b.close()


def test_full_size_fingerprints(eng):
    """BASELINE cfg4 (150k atoms x 100 points) and cfg5 (1M atoms x 960 points): the mask row popcounts, as little-endian u32 in
    atom order, have the sha256 and sum of the oracle's counts stored in tests/golden/cfg_hashes.json."""
    import hashlib
    import json
    import os
    from rustsasa_b200 import workloads as W
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    gold = json.load(open(os.path.join(root, "tests", "golden", "cfg_hashes.json")))
    for key, data in (("cfg4", W.large_assembly(150000)), ("cfg5", W.capsid_shell(1000000))):
        g = gold[key]
        assert data.n_atoms == g["atoms"]
        b = eng.batch(data.struct_off)
        r = b.run_masks_host(data.xyzr, n_points=g["n_points"], want=("counts",))
        pc = popcount_rows(r.exposed)
        assert int(pc.astype(np.int64).sum()) == g["sum_counts"], key
        assert hashlib.sha256(np.ascontiguousarray(pc, dtype="<u4").tobytes()).hexdigest() == g["sha256_counts"], key
        assert np.array_equal(pc, r.counts)
        b.close()


@pytest.mark.parametrize("n_points", [100, 960])
def test_device_entry_equals_host(eng, golden, n_points):
    import torch
    b, structs = golden_batch(eng, golden, golden.names[:30])
    xyzr = np.concatenate(structs)
    h = b.run_masks_host(xyzr, n_points=n_points)
    W = (n_points + 31) // 32
    d_mask = torch.full((xyzr.shape[0], W), -1, dtype=torch.int32, device="cuda")
    d = dict(counts=torch.zeros(xyzr.shape[0], dtype=torch.int32, device="cuda"),
             atom_sasa=torch.zeros(xyzr.shape[0], dtype=torch.float32, device="cuda"),
             seg_sasa=torch.zeros(b.n_seg, dtype=torch.float32, device="cuda"),
             protein=torch.zeros((b.S, 3), dtype=torch.float32, device="cuda"))
    b.run_masks_device(torch.from_numpy(xyzr).cuda(), d_mask, n_points=n_points, **d)
    torch.cuda.synchronize()
    b.sync()
    assert np.array_equal(d_mask.cpu().numpy().view(np.uint32), h.exposed)
    assert np.array_equal(d["counts"].cpu().numpy().view(np.uint32), h.counts)
    for f in ("atom_sasa", "seg_sasa", "protein"):
        assert np.array_equal(d[f].cpu().numpy(), getattr(h, f)), f
    b.close()


def test_non_finite_structure_in_the_middle(eng, golden):
    import torch
    from rustsasa_b200 import _lib
    from rustsasa_b200.engine import SasaB200Error
    s = golden.structure("example.cif")["xyzr"]
    rng = np.random.default_rng(3)
    big = _cluster(rng, 30000, 85.0)
    structs = [s, s, big, s, big]
    off = np.cumsum([0] + [x.shape[0] for x in structs]).astype(np.uint64)
    xyzr = np.concatenate(structs)
    b = eng.batch(off)
    for n_points in (100, 960):
        good = b.run_masks_host(xyzr, n_points=n_points)
        bad = xyzr.copy()
        bad[int(off[1]) + 5, 2] = np.nan     # fused-kernel structure
        bad[int(off[4]) + 7, 0] = np.inf     # large-path structure
        W = (n_points + 31) // 32
        exposed = np.full((xyzr.shape[0], W), 0xFFFFFFFF, np.uint32)
        counts = np.full(xyzr.shape[0], 7, np.uint32)
        outs = _lib.Outputs(counts.ctypes.data, None, None, None)
        prm = _lib.Params(PROBE, n_points, 8, -1, 0)
        rc = b._L.sasa_b200_batch_run_masks_host(b._h, bad.ctypes.data, None, C.byref(prm), C.byref(outs), exposed.ctypes.data, None)
        assert rc == _lib.ERR_NON_FINITE
        for k in range(len(structs)):
            a0, a1 = int(off[k]), int(off[k + 1])
            if k in (1, 4):
                assert not np.any(exposed[a0:a1]) and not np.any(counts[a0:a1]), k
            else:
                assert np.array_equal(exposed[a0:a1], good.exposed[a0:a1]), k
                assert np.array_equal(counts[a0:a1], good.counts[a0:a1]), k
        d_mask = torch.full((xyzr.shape[0], W), -1, dtype=torch.int32, device="cuda")
        b.run_masks_device(torch.from_numpy(bad).cuda(), d_mask, n_points=n_points)
        torch.cuda.synchronize()
        with pytest.raises(SasaB200Error) as e:
            b.sync()
        assert e.value.code == _lib.ERR_NON_FINITE
        assert np.array_equal(d_mask.cpu().numpy().view(np.uint32), exposed)
    # the context stays usable
    assert np.array_equal(b.run_masks_host(xyzr, n_points=960).exposed, good.exposed)
    b.close()


def test_empty_batch_empty_structures_and_null_mask(eng, oracle):
    from rustsasa_b200 import _lib
    b = eng.batch([0])
    r = b.run_masks_host(np.zeros((0, 4), np.float32))
    assert r.exposed.shape == (0, 4) and r.counts.shape == (0,)
    rc = b._L.sasa_b200_batch_run_masks_host(b._h, None, None, C.byref(_lib.Params(PROBE, 100, 8, -1, 0)),
                                             C.byref(_lib.Outputs(None, None, None, None)), None, None)
    assert rc == _lib.OK
    b.close()
    xyzr = np.array([[1, 2, 3, 1.5], [5, 5, 5, 1.8], [5, 5, 5, 1.8], [5.5, 5, 5, 1.2]], np.float32)
    b = eng.batch([0, 0, 1, 1, 4, 4])
    r, _ = check_run(b, xyzr, oracle, [xyzr[:1], xyzr[1:]])
    assert r.exposed[0, :3].tolist() == [0xFFFFFFFF] * 3 and r.exposed[0, 3] == 0xF
    outs = _lib.Outputs(None, None, None, None)
    prm = _lib.Params(PROBE, 100, 8, -1, 0)
    assert b._L.sasa_b200_batch_run_masks_host(b._h, xyzr.ctypes.data, None, C.byref(prm), C.byref(outs), None, None) == \
        _lib.ERR_INVALID_ARGUMENT
    assert b._L.sasa_b200_batch_run_masks_device(b._h, xyzr.ctypes.data, None, C.byref(prm), C.byref(outs), None, None) == \
        _lib.ERR_INVALID_ARGUMENT
    b.close()


def test_process_surface(eng, oracle, tmp_path):
    from rustsasa_b200 import AtomLevel, ProteinLevel, ResidueLevel, SASAOptions, read_structure, surface_points
    from tests import synthetic_pdb as sp
    pa, _ = sp.write(tmp_path, "surf", sp.make_atoms(11, n_res=80, chains="AB"))
    st = read_structure(pa)
    for level in (AtomLevel, ResidueLevel, ProteinLevel):
        opt = SASAOptions(level)
        r = opt.process_surface([st], engine=eng)[0]
        plain = opt.process(st, eng)
        if level is AtomLevel:
            assert np.array_equal(r.result, plain)
        else:
            assert r.result == plain
        p = opt._pack(st)
        m = exposed_masks(oracle, p.xyzr, opt.probe_radius, opt.n_points, 8, ids=p.ids)
        pts, atom = surface_points(p.xyzr, m, opt.n_points, opt.probe_radius)
        assert np.array_equal(r.points, pts) and np.array_equal(r.atom_index, atom)
        assert r.points.shape[0] > 0
    counts = np.bincount(r.atom_index, minlength=opt._pack(st).xyzr.shape[0])
    atom_sasa = SASAOptions(AtomLevel).process(st, eng)
    assert np.array_equal(counts == 0, atom_sasa == 0)
