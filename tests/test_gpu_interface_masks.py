"""Grouped runs with exposed-point masks (interface patches): sasa_b200_batch_run_groups_masks_host / _device.

The complex masks must equal the CPU oracle's masks of the whole structure (tests/mask_oracle.py) and the masked run's bit for
bit; the isolated masks must equal the oracle's masks of every group's atoms run alone, scattered back to the original atom
order (neighbour membership is result-neutral, so that reference is exact).  The other outputs must equal the grouped run's bit
for bit, on every path a grouped run takes: the fused kernel's cap path and streaming cold path, the large-structure path's cap
branch and its streamed atoms (k < 0), and n_points > 128, where every structure takes the large-structure path.
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


def valid_rows(n, n_points):
    """Mask rows with every existing point set."""
    bits = np.zeros((n, ((n_points + 31) // 32) * 32), np.uint8)
    bits[:, :n_points] = 1
    return np.packbits(bits, axis=1, bitorder="little").view(np.uint32)


def iso_masks(oracle, xyzr, group, probe=PROBE, n_points=100, lanes=8, ids=None):
    """The oracle's masks of every group's atoms alone, scattered back to the original atom order."""
    out = np.zeros((xyzr.shape[0], (n_points + 31) // 32), np.uint32)
    for g in np.unique(group):
        m = np.nonzero(group == g)[0]
        out[m] = exposed_masks(oracle, xyzr[m], probe, n_points, lanes, ids=None if ids is None else ids[m])
    return out


def same_outputs(a, b):
    for f in ("counts", "atom_sasa", "seg_sasa", "protein"):
        x, y = getattr(a, f), getattr(b, f)
        assert (x is None) == (y is None), f
        if x is not None:
            assert np.array_equal(x, y, equal_nan=f != "counts"), f


def check_invariants(cpx, iso):
    assert np.array_equal(popcount_rows(cpx.exposed), cpx.counts)
    assert np.array_equal(popcount_rows(iso.exposed), iso.counts)
    assert not np.any(cpx.exposed & ~iso.exposed)
    buried = iso.exposed & ~cpx.exposed
    assert np.array_equal(popcount_rows(buried).astype(np.int64), iso.counts.astype(np.int64) - cpx.counts.astype(np.int64))


def check_run(b, xyzr, group, oracle, structs, groups, n_points=100, lanes=8, probe=PROBE, cls=None, ids=None,
              want=("counts", "atom")):
    """Masked grouped run against the grouped run and the masked run (outputs, complex masks) and the oracle (both mask sets,
    per structure).  Returns (complex, isolated) of the masked grouped run."""
    ref = b.run_groups_host(xyzr, group, cls, probe, n_points, lanes, want=want)
    masked = b.run_masks_host(xyzr, cls, probe, n_points, lanes, want=("counts",))
    cpx, iso = b.run_groups_masks_host(xyzr, group, cls, probe, n_points, lanes, want=want)
    same_outputs(cpx, ref[0])
    same_outputs(iso, ref[1])
    W = (n_points + 31) // 32
    for r in (cpx, iso):
        assert r.exposed.shape == (xyzr.shape[0], W) and r.exposed.dtype == np.uint32
    assert np.array_equal(cpx.exposed, masked.exposed)
    if "counts" in want:
        check_invariants(cpx, iso)
    a0 = 0
    for i, s in enumerate(structs):
        a1 = a0 + s.shape[0]
        sid = None if ids is None else ids[i]
        assert np.array_equal(cpx.exposed[a0:a1], exposed_masks(oracle, s, probe, n_points, lanes, ids=sid)), (i, n_points, lanes)
        assert np.array_equal(iso.exposed[a0:a1], iso_masks(oracle, s, groups[i], probe, n_points, lanes, ids=sid)), (i, n_points, lanes)
        a0 = a1
    return cpx, iso


def chain_groups(golden, s):
    g = np.zeros(s["xyzr"].shape[0], np.uint32)
    for ci, (b, e) in enumerate(golden.chain_ranges(s)):
        g[b:e] = ci
    return g


def multichain_batch(eng, golden, limit=None):
    names = [n for n in golden.names if len(np.unique(golden.structure(n)["res_chain"])) > 1][:limit]
    ss = [golden.structure(n) for n in names]
    off = np.cumsum([0] + [s["xyzr"].shape[0] for s in ss]).astype(np.uint64)
    seg_off = np.cumsum([0] + [len(s["seg_be"]) for s in ss]).astype(np.uint64)
    b = eng.batch(off, np.concatenate([s["seg_be"] for s in ss]), seg_off, np.concatenate([s["polar"] for s in ss]))
    return b, [s["xyzr"] for s in ss], [chain_groups(golden, s) for s in ss]


@pytest.mark.parametrize("n_points", [100, 960])
def test_multichain_golden_one_group_per_chain(eng, oracle, golden, n_points):
    b, structs, groups = multichain_batch(eng, golden)
    assert len(structs) == 44
    cpx, iso = check_run(b, np.concatenate(structs), np.concatenate(groups), oracle, structs, groups, n_points, want=ALL)
    if n_points <= 128:
        assert cpx.stats["streamed_atoms"] == 0
    assert np.any(iso.exposed & ~cpx.exposed)   # chains touch: there are interface patches
    b.close()


@pytest.mark.parametrize("n_points", [100, 960])
def test_invariants(eng, golden, n_points):
    s = golden.structure("4xfj")
    n = s["xyzr"].shape[0]
    b = eng.batch([0, n], s["seg_be"], [0, len(s["seg_be"])], s["polar"])
    masked = b.run_masks_host(s["xyzr"], n_points=n_points)
    cpx, iso = b.run_groups_masks_host(s["xyzr"], np.full(n, 7, np.uint32), n_points=n_points)
    check_invariants(cpx, iso)
    assert np.array_equal(cpx.exposed, masked.exposed) and np.array_equal(iso.exposed, masked.exposed)
    cpx, iso = b.run_groups_masks_host(s["xyzr"], np.arange(n, dtype=np.uint32), n_points=n_points)
    check_invariants(cpx, iso)
    assert np.array_equal(cpx.exposed, masked.exposed)
    assert np.array_equal(iso.exposed, valid_rows(n, n_points))
    b.close()


@pytest.mark.parametrize("n_points", [1, 37, 100, 128, 129, 960])
@pytest.mark.parametrize("seed", range(3))
def test_randomised_geometry_random_groups(eng, oracle, seed, n_points):
    rng = np.random.default_rng(8300 + 10 * seed + n_points)
    lanes = (4, 8, 16)[seed]   # body / tail splits: every lane count at every n_points
    probe = float(rng.choice([0.0, 1.4, 3.0]))
    structs, groups = [], []
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
        groups.append(rng.integers(0, int((1, 2, 3, 7)[t % 4]), size=n).astype(np.uint32))
    off = np.cumsum([0] + [s.shape[0] for s in structs]).astype(np.uint64)
    b = eng.batch(off)
    check_run(b, np.concatenate(structs), np.concatenate(groups), oracle, structs, groups, n_points, lanes, probe)
    b.close()


def _cluster(rng, n, side):
    xyz = rng.uniform(0.0, side, size=(n, 3))
    return np.concatenate([xyz, rng.uniform(1.2, 2.0, size=(n, 1))], axis=1).astype(np.float32)


def _plane_groups(s):
    key = s[:, 0] + 0.3 * s[:, 1]
    return (key > np.median(key)).astype(np.uint32)


@pytest.mark.parametrize("n_points", [100, 960])
@pytest.mark.parametrize("with_cls", [False, True])
def test_every_path(eng, oracle, n_points, with_cls):
    """A dense cluster (more than 96 neighbours per atom: the fused kernel's streaming cold path), a structure above the fused
    kernels' capacity with a dense cluster beside it (the large-structure path: cap branch and streamed atoms), and two
    protein-density clusters 3,000 A apart (every cell's candidate list overflows: cold atoms), each cut in two by a plane, with
    and without duplicate ids.  With 960 points every structure takes the large-structure path and streams."""
    rng = np.random.default_rng(61 + with_cls + n_points)
    dense = _cluster(rng, 600, 12.0)
    big = np.concatenate([_cluster(rng, 40000, 95.0), _cluster(rng, 600, 12.0) + np.array([200, 0, 0, 0], np.float32)])
    pair = np.concatenate([_cluster(rng, 500, 20.6), _cluster(rng, 500, 20.6) + np.array([3000, 0, 0, 0], np.float32)])
    structs = [dense, big, pair]
    groups = [_plane_groups(s) for s in structs]
    off = np.cumsum([0] + [s.shape[0] for s in structs]).astype(np.uint64)
    ids = [rng.integers(0, s.shape[0] // 2, size=s.shape[0]).astype(np.uint64) for s in structs] if with_cls else None
    cls = None
    if with_cls:
        cls = np.concatenate([np.unique(ids[i], return_inverse=True)[1].astype(np.uint32) + np.uint32(off[i])
                              for i in range(len(structs))])
    b = eng.batch(off)
    cpx, iso = check_run(b, np.concatenate(structs), np.concatenate(groups), oracle, structs, groups, n_points, cls=cls, ids=ids)
    streamed = cpx.stats["streamed_atoms"]
    if n_points <= 128:
        assert streamed > 2 * (dense.shape[0] // 2)   # both evaluations of the dense clusters' atoms stream
    else:
        assert streamed == 2 * sum(s.shape[0] for s in structs)
    assert np.any(iso.exposed & ~cpx.exposed)
    b.close()


@pytest.mark.parametrize("n_points", [100, 960])
def test_device_entry_equals_host(eng, golden, n_points):
    import torch
    b, structs, groups = multichain_batch(eng, golden, 10)
    xyzr, group = np.concatenate(structs), np.concatenate(groups)
    h = b.run_groups_masks_host(xyzr, group, n_points=n_points)
    W = (n_points + 31) // 32
    m = [torch.full((xyzr.shape[0], W), -1, dtype=torch.int32, device="cuda") for _ in range(2)]
    d = b.run_groups_masks_device(torch.from_numpy(xyzr).cuda(), torch.from_numpy(group.view(np.int32)).cuda(), m[0], m[1],
                                  n_points=n_points)
    torch.cuda.synchronize()
    b.sync()
    for hr, dr in zip(h, d):
        assert np.array_equal(dr.exposed.cpu().numpy().view(np.uint32), hr.exposed)
        assert np.array_equal(dr.counts.cpu().numpy().view(np.uint32), hr.counts)
        for f in ("atom_sasa", "seg_sasa", "protein"):
            assert np.array_equal(getattr(dr, f).cpu().numpy(), getattr(hr, f)), f
    b.close()


def test_errors(eng, golden):
    from rustsasa_b200 import _lib
    from rustsasa_b200.engine import SasaB200Error
    s = golden.structure("example.cif")["xyzr"]
    n = s.shape[0]
    b = eng.batch([0, n])
    group = (np.arange(n) % 2).astype(np.uint32)
    for flags in (_lib.FLAG_BOUNDARY_STATS, _lib.FLAG_FORCE_STREAMING):
        with pytest.raises(SasaB200Error) as e:
            b.run_groups_masks_host(s, group, flags=flags)
        assert e.value.code == _lib.ERR_UNSUPPORTED
    ex, ei = np.zeros((n, 4), np.uint32), np.zeros((n, 4), np.uint32)
    outs = _lib.Outputs(None, None, None, None)
    prm = _lib.Params(PROBE, 100, 8, -1, 0)
    L, h, x, g = b._L, b._h, s.ctypes.data, group.ctypes.data
    for args in ((None, ex.ctypes.data, ei.ctypes.data), (g, None, ei.ctypes.data), (g, ex.ctypes.data, None)):
        assert L.sasa_b200_batch_run_groups_masks_host(h, x, None, args[0], C.byref(prm), C.byref(outs), C.byref(outs), args[1], args[2],
                                                       None) == _lib.ERR_INVALID_ARGUMENT, args
        assert L.sasa_b200_batch_run_groups_masks_device(h, x, None, args[0], C.byref(prm), C.byref(outs), C.byref(outs), args[1],
                                                         args[2], None) == _lib.ERR_INVALID_ARGUMENT, args
    assert L.sasa_b200_batch_run_groups_masks_host(h, x, None, g, C.byref(prm), C.byref(outs), None, ex.ctypes.data, ei.ctypes.data,
                                                   None) == _lib.ERR_INVALID_ARGUMENT
    # The size check shared with the masked entry points (n_atoms * ceil(n_points / 32) * 4 bytes must fit a size_t) cannot
    # fail with a 64-bit size_t: a batch holds fewer than 2^32 atoms and n_points is at most 2^24.  Past that bound the
    # point count itself is rejected.
    big = _lib.Params(PROBE, (1 << 24) + 1, 8, -1, 0)
    assert L.sasa_b200_batch_run_groups_masks_host(h, x, None, g, C.byref(big), C.byref(outs), C.byref(outs), ex.ctypes.data,
                                                   ei.ctypes.data, None) == _lib.ERR_INVALID_ARGUMENT
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
    group = np.concatenate([_plane_groups(x) for x in structs])
    b = eng.batch(off)
    for n_points in (100, 960):
        good = b.run_groups_masks_host(xyzr, group, n_points=n_points)
        bad = xyzr.copy()
        bad[int(off[1]) + 5, 2] = np.nan     # fused-kernel structure (n_points <= 128)
        bad[int(off[4]) + 7, 0] = np.inf     # large-path structure
        W = (n_points + 31) // 32
        ex = [np.full((xyzr.shape[0], W), 0xFFFFFFFF, np.uint32) for _ in range(2)]
        counts = [np.full(xyzr.shape[0], 7, np.uint32) for _ in range(2)]
        atom = [np.zeros(xyzr.shape[0], np.float32) for _ in range(2)]
        outs = [_lib.Outputs(counts[i].ctypes.data, atom[i].ctypes.data, None, None) for i in range(2)]
        prm = _lib.Params(PROBE, n_points, 8, -1, 0)
        rc = b._L.sasa_b200_batch_run_groups_masks_host(b._h, bad.ctypes.data, None, group.ctypes.data, C.byref(prm), C.byref(outs[0]),
                                                        C.byref(outs[1]), ex[0].ctypes.data, ex[1].ctypes.data, None)
        assert rc == _lib.ERR_NON_FINITE
        for i in range(2):
            for k in range(len(structs)):
                a0, a1 = int(off[k]), int(off[k + 1])
                if k in (1, 4):
                    assert not np.any(ex[i][a0:a1]) and not np.any(counts[i][a0:a1]), (i, k)
                    assert np.all(np.isnan(atom[i][a0:a1])), (i, k)
                else:
                    assert np.array_equal(ex[i][a0:a1], good[i].exposed[a0:a1]), (i, k)
                    assert np.array_equal(counts[i][a0:a1], good[i].counts[a0:a1]), (i, k)
        dm = [torch.full((xyzr.shape[0], W), -1, dtype=torch.int32, device="cuda") for _ in range(2)]
        b.run_groups_masks_device(torch.from_numpy(bad).cuda(), torch.from_numpy(group.view(np.int32)).cuda(), dm[0], dm[1],
                                  n_points=n_points)
        torch.cuda.synchronize()
        with pytest.raises(SasaB200Error) as e:
            b.sync()
        assert e.value.code == _lib.ERR_NON_FINITE
        for i in range(2):
            assert np.array_equal(dm[i].cpu().numpy().view(np.uint32), ex[i])
    # the context stays usable
    again = b.run_groups_masks_host(xyzr, group, n_points=960)
    assert np.array_equal(again[0].exposed, good[0].exposed) and np.array_equal(again[1].exposed, good[1].exposed)
    b.close()


def test_empty_batch_and_empty_structures(eng, oracle):
    from rustsasa_b200 import _lib
    b = eng.batch([0])
    cpx, iso = b.run_groups_masks_host(np.zeros((0, 4), np.float32), np.zeros(0, np.uint32))
    assert cpx.exposed.shape == (0, 4) and iso.exposed.shape == (0, 4) and iso.counts.shape == (0,)
    outs = _lib.Outputs(None, None, None, None)
    rc = b._L.sasa_b200_batch_run_groups_masks_host(b._h, None, None, None, C.byref(_lib.Params(PROBE, 100, 8, -1, 0)), C.byref(outs),
                                                    C.byref(outs), None, None, None)
    assert rc == _lib.OK
    b.close()
    xyzr = np.array([[1, 2, 3, 1.5], [5, 5, 5, 1.8], [5, 5, 5, 1.8], [5.5, 5, 5, 1.2]], np.float32)
    groups = [np.zeros(1, np.uint32), np.array([0, 1, 1], np.uint32)]
    b = eng.batch([0, 0, 1, 1, 4, 4])
    cpx, iso = check_run(b, xyzr, np.concatenate(groups), oracle, [xyzr[:1], xyzr[1:]], groups)
    assert cpx.exposed[0].tolist() == iso.exposed[0].tolist() == [0xFFFFFFFF] * 3 + [0xF]
    assert np.array_equal(iso.exposed[1], valid_rows(1, 100)[0])   # atom 1 alone in its group
    b.close()


def test_full_size_cfg4_cut_in_two(eng):
    """BASELINE cfg4 (150k atoms, 100 points) cut in two by a plane through its centroid."""
    from rustsasa_b200 import workloads as W
    d = W.large_assembly(150000)
    x = d.xyzr[:, :3].astype(np.float64)
    group = ((x - x.mean(axis=0)) @ np.array([0.6, -0.3, 0.74]) > 0.0).astype(np.uint32)
    b = eng.batch(d.struct_off)
    masked = b.run_masks_host(d.xyzr, want=("counts",))
    _, ref_iso = b.run_groups_host(d.xyzr, group, want=("counts",))
    cpx, iso = b.run_groups_masks_host(d.xyzr, group, want=("counts",))
    assert np.array_equal(cpx.exposed, masked.exposed)
    assert np.array_equal(popcount_rows(iso.exposed), ref_iso.counts)
    assert not np.any(cpx.exposed & ~iso.exposed)
    assert int(popcount_rows(iso.exposed & ~cpx.exposed).sum()) > 0
    b.close()


def test_process_interface_surface(eng, tmp_path):
    from rustsasa_b200 import InterfaceSurfaceResult, ProteinLevel, ResidueLevel, SASAOptions, read_structure
    from rustsasa_b200.api import _dense_classes
    from tests import synthetic_pdb as sp
    pa, _ = sp.write(tmp_path, "ab", sp.make_atoms(5, n_res=60, chains="AB"))
    st = read_structure(pa)
    for level in (ResidueLevel, ProteinLevel):
        opt = SASAOptions(level)
        r = opt.process_interface_surface([st], engine=eng)[0]
        assert isinstance(r, InterfaceSurfaceResult)
        assert r.interface == opt.process_interface([st], engine=eng)[0]
        assert r.interface.buried_area > 0
        # buried points per atom: isolated - complex counts of the grouped run (one group per chain)
        p = opt._pack(st)
        n = p.xyzr.shape[0]
        b = eng.batch([0, n])
        cpx, iso = b.run_groups_host(p.xyzr, SASAOptions._chain_groups(p.atom_chain, []), _dense_classes(p.ids), opt.probe_radius,
                                     opt.n_points, want=("counts",))
        b.close()
        buried = np.bincount(r.atom_index, minlength=n)
        assert np.array_equal(buried, iso.counts.astype(np.int64) - cpx.counts.astype(np.int64))
        assert r.points.shape == (buried.sum(), 3) and r.points.dtype == np.float32 and r.atom_index.dtype == np.int64
        assert r.points.shape[0] > 0
        # every buried point lies on its atom's probe sphere
        d = np.linalg.norm(r.points.astype(np.float64) - p.xyzr[r.atom_index, :3], axis=1)
        assert np.allclose(d, p.xyzr[r.atom_index, 3] + opt.probe_radius, rtol=0, atol=1e-3)
    # one chain, or both chains in one group: no interface
    pb, _ = sp.write(tmp_path, "a", sp.make_atoms(6, n_res=60, chains="A"))
    one = SASAOptions(ProteinLevel).process_interface_surface([read_structure(pb)], engine=eng)[0]
    assert one.points.shape == (0, 3) and one.atom_index.shape == (0,) and one.interface.buried_area == 0.0
    both = SASAOptions(ProteinLevel).process_interface_surface([st], chain_groups=["AB"], engine=eng)[0]
    assert both.points.shape == (0, 3)
