"""Grouped runs (buried surface area): sasa_b200_batch_run_groups_host / _device against the CPU oracle.

The complex outputs must equal a plain run bit for bit; the isolated outputs must equal the oracle run on each group's atoms
alone (same order, same id rule), counts and per-atom areas exactly, residue / chain sums bit-identical to the oracle's sums
over the isolated per-atom vector.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PROBE = 1.4
REL, ABS = 1e-4, 1e-3


@pytest.fixture(scope="module")
def eng():
    from rustsasa_b200 import Engine
    e = Engine()
    yield e
    e.close()


def close_enough(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return np.all(np.abs(a - b) <= np.maximum(ABS, REL * np.abs(b)))


def iso_oracle(oracle, xyzr, group, probe=PROBE, n_points=100, lanes=8, ids=None):
    """The oracle on every group's atoms alone, scattered back to the original atom order."""
    counts = np.zeros(xyzr.shape[0], np.uint32)
    sasa = np.zeros(xyzr.shape[0], np.float32)
    for g in np.unique(group):
        m = np.nonzero(group == g)[0]
        o = oracle.calculate_sasa_internal(xyzr[m], probe, n_points, lanes=lanes, threads=0 if m.size > 10000 else 1,
                                           ids=None if ids is None else ids[m])
        counts[m] = o["counts"]
        sasa[m] = o["sasa"]
    return counts, sasa


def chain_groups(golden, s):
    g = np.zeros(s["xyzr"].shape[0], np.uint32)
    for ci, (b, e) in enumerate(golden.chain_ranges(s)):
        g[b:e] = ci
    return g


@pytest.mark.parametrize("n_points", [100, 960])
def test_multichain_golden_one_group_per_chain(eng, oracle, golden, n_points):
    names = [n for n in golden.names if len(np.unique(golden.structure(n)["res_chain"])) > 1]
    assert len(names) == 44
    ss = [golden.structure(n) for n in names]
    off = np.cumsum([0] + [s["xyzr"].shape[0] for s in ss]).astype(np.uint64)
    seg_off = np.cumsum([0] + [len(s["seg_be"]) for s in ss]).astype(np.uint64)
    xyzr = np.concatenate([s["xyzr"] for s in ss])
    group = np.concatenate([chain_groups(golden, s) for s in ss])
    b = eng.batch(off, np.concatenate([s["seg_be"] for s in ss]), seg_off, np.concatenate([s["polar"] for s in ss]))
    plain = b.run_host(xyzr, n_points=n_points)
    cpx, iso = b.run_groups_host(xyzr, group, n_points=n_points)
    for f in ("counts", "atom_sasa", "seg_sasa", "protein"):
        assert np.array_equal(getattr(cpx, f), getattr(plain, f)), f
    for i, s in enumerate(ss):
        a0, a1, g0, g1 = int(off[i]), int(off[i + 1]), int(seg_off[i]), int(seg_off[i + 1])
        counts, sasa = iso_oracle(oracle, s["xyzr"], group[a0:a1], n_points=n_points)
        assert np.array_equal(iso.counts[a0:a1], counts), names[i]
        assert np.array_equal(iso.atom_sasa[a0:a1], sasa), names[i]
        assert np.array_equal(iso.seg_sasa[g0:g1], oracle.segment_sums(sasa, s["seg_be"])), names[i]
        assert close_enough(iso.protein[i], oracle.protein_totals(sasa, s["seg_be"], s["polar"])), names[i]
        assert np.all(iso.counts[a0:a1] >= cpx.counts[a0:a1])
    b.close()
    # chain level: one segment per chain
    cr = [golden.chain_ranges(s) for s in ss]
    cb = eng.batch(off, np.concatenate(cr), np.cumsum([0] + [len(c) for c in cr]).astype(np.uint64))
    _, iso_c = cb.run_groups_host(xyzr, group, n_points=n_points, want=("seg",))
    k = 0
    for i, s in enumerate(ss):
        a0, a1 = int(off[i]), int(off[i + 1])
        want = oracle.segment_sums(iso.atom_sasa[a0:a1], cr[i])
        assert np.array_equal(iso_c.seg_sasa[k:k + len(cr[i])], want), names[i]
        k += len(cr[i])
    cb.close()


@pytest.mark.parametrize("n_points", [100, 960])
def test_invariants(eng, golden, n_points):
    s = golden.structure("4xfj")
    n = s["xyzr"].shape[0]
    b = eng.batch([0, n], s["seg_be"], [0, len(s["seg_be"])], s["polar"])
    plain = b.run_host(s["xyzr"], n_points=n_points)
    cpx, iso = b.run_groups_host(s["xyzr"], np.full(n, 7, np.uint32), n_points=n_points)
    for f in ("counts", "atom_sasa", "seg_sasa", "protein"):
        assert np.array_equal(getattr(cpx, f), getattr(plain, f))
        assert np.array_equal(getattr(iso, f), getattr(plain, f))
    cpx, iso = b.run_groups_host(s["xyzr"], np.arange(n, dtype=np.uint32), n_points=n_points)
    assert np.array_equal(cpx.counts, plain.counts)
    assert np.all(iso.counts == n_points)
    b.close()


@pytest.mark.parametrize("n_points", [1, 37, 100, 128, 129])
@pytest.mark.parametrize("seed", range(3))
def test_randomised_geometry_random_groups(eng, oracle, seed, n_points):
    rng = np.random.default_rng(7100 + 10 * seed + n_points)
    lanes = int(rng.choice([4, 8, 16]))
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
        groups.append(rng.integers(0, int(rng.choice([1, 2, 3, 7])), size=n).astype(np.uint32))
    off = np.cumsum([0] + [s.shape[0] for s in structs]).astype(np.uint64)
    xyzr, group = np.concatenate(structs), np.concatenate(groups)
    b = eng.batch(off)
    plain = b.run_host(xyzr, probe_radius=probe, n_points=n_points, simd_lanes=lanes, want=("counts", "atom"))
    cpx, iso = b.run_groups_host(xyzr, group, probe_radius=probe, n_points=n_points, simd_lanes=lanes, want=("counts", "atom"))
    assert np.array_equal(cpx.counts, plain.counts) and np.array_equal(cpx.atom_sasa, plain.atom_sasa)
    for i, s in enumerate(structs):
        a0, a1 = int(off[i]), int(off[i + 1])
        counts, sasa = iso_oracle(oracle, s, groups[i], probe, n_points, lanes)
        assert np.array_equal(iso.counts[a0:a1], counts), (seed, i, n_points)
        assert np.array_equal(iso.atom_sasa[a0:a1], sasa), (seed, i, n_points)
    b.close()


def _cluster(rng, n, side):
    xyz = rng.uniform(0.0, side, size=(n, 3))
    return np.concatenate([xyz, rng.uniform(1.2, 2.0, size=(n, 1))], axis=1).astype(np.float32)


@pytest.mark.parametrize("with_cls", [False, True])
def test_cold_paths(eng, oracle, with_cls):
    """A dense cluster cut in two by a plane (more than 96 neighbours per atom: the streaming routine) and a structure above
    the fused kernels' capacity (the large-structure path), with and without id classes."""
    rng = np.random.default_rng(31 + with_cls)
    dense = _cluster(rng, 600, 12.0)
    big = _cluster(rng, 40000, 95.0)
    structs = [dense, big]
    groups = [(s[:, 0] + 0.3 * s[:, 1] > np.median(s[:, 0] + 0.3 * s[:, 1])).astype(np.uint32) for s in structs]
    ids = [rng.integers(0, s.shape[0] // 2, size=s.shape[0]).astype(np.uint64) for s in structs] if with_cls else None
    off = np.cumsum([0] + [s.shape[0] for s in structs]).astype(np.uint64)
    xyzr, group = np.concatenate(structs), np.concatenate(groups)
    cls = None
    if with_cls:
        cls = np.concatenate([np.unique(ids[i], return_inverse=True)[1].astype(np.uint32) + np.uint32(off[i])
                              for i in range(len(structs))])
    b = eng.batch(off)
    plain = b.run_host(xyzr, cls, want=("counts", "atom"))
    cpx, iso = b.run_groups_host(xyzr, group, cls, want=("counts", "atom"))
    assert plain.stats["streamed_atoms"] > 0
    assert np.array_equal(cpx.counts, plain.counts) and np.array_equal(cpx.atom_sasa, plain.atom_sasa)
    for i, s in enumerate(structs):
        a0, a1 = int(off[i]), int(off[i + 1])
        counts, sasa = iso_oracle(oracle, s, groups[i], ids=None if ids is None else ids[i])
        assert np.array_equal(iso.counts[a0:a1], counts), i
        assert np.array_equal(iso.atom_sasa[a0:a1], sasa), i
        assert np.all(iso.counts[a0:a1] >= cpx.counts[a0:a1])
    b.close()


def test_device_entry_equals_host(eng, golden):
    import torch
    names = [n for n in golden.names if len(np.unique(golden.structure(n)["res_chain"])) > 1][:10]
    ss = [golden.structure(n) for n in names]
    off = np.cumsum([0] + [s["xyzr"].shape[0] for s in ss]).astype(np.uint64)
    seg_off = np.cumsum([0] + [len(s["seg_be"]) for s in ss]).astype(np.uint64)
    xyzr = np.concatenate([s["xyzr"] for s in ss])
    group = np.concatenate([chain_groups(golden, s) for s in ss])
    b = eng.batch(off, np.concatenate([s["seg_be"] for s in ss]), seg_off, np.concatenate([s["polar"] for s in ss]))
    h = b.run_groups_host(xyzr, group)
    d = b.run_groups_device(torch.from_numpy(xyzr).cuda(), torch.from_numpy(group.astype(np.int32)).cuda())
    torch.cuda.synchronize()
    b.sync()
    for hr, dr in zip(h, d):
        assert np.array_equal(hr.counts, dr.counts.cpu().numpy().astype(np.uint32))
        for f in ("atom_sasa", "seg_sasa", "protein"):
            assert np.array_equal(getattr(hr, f), getattr(dr, f).cpu().numpy()), f
    b.close()


def test_errors_and_non_finite(eng, golden):
    import ctypes as C
    from rustsasa_b200 import _lib
    from rustsasa_b200.engine import SasaB200Error
    s = golden.structure("example.cif")
    n = s["xyzr"].shape[0]
    b = eng.batch([0, n, 2 * n], np.concatenate([s["seg_be"], s["seg_be"]]), [0, len(s["seg_be"]), 2 * len(s["seg_be"])],
                  np.concatenate([s["polar"], s["polar"]]))
    xyzr = np.concatenate([s["xyzr"], s["xyzr"]])
    group = np.tile(np.arange(n, dtype=np.uint32) % 2, 2)
    with pytest.raises(SasaB200Error) as e:
        b.run_groups_host(xyzr, group, flags=_lib.FLAG_BOUNDARY_STATS)
    assert e.value.code == _lib.ERR_UNSUPPORTED
    with pytest.raises(SasaB200Error) as e:
        b.run_groups_host(xyzr, group, flags=_lib.FLAG_FORCE_STREAMING)
    assert e.value.code == _lib.ERR_UNSUPPORTED
    # NULL group through the C ABI directly
    outs = _lib.Outputs(None, None, None, None)
    prm = _lib.Params(PROBE, 100, 8, -1, 0)
    rc = b._L.sasa_b200_batch_run_groups_host(b._h, xyzr.ctypes.data, None, None, C.byref(prm), C.byref(outs), C.byref(outs), None)
    assert rc == _lib.ERR_INVALID_ARGUMENT
    good_cpx, good_iso = b.run_groups_host(xyzr, group)
    bad = xyzr.copy()
    bad[n + 3, 1] = np.nan
    with pytest.raises(SasaB200Error) as e:
        b.run_groups_host(bad, group)
    assert e.value.code == _lib.ERR_NON_FINITE
    # the outputs of the bad structure are NaN in both sets (checked through explicit result buffers)
    from rustsasa_b200.engine import BatchResult
    cpx, iso = BatchResult(), BatchResult()
    for r in (cpx, iso):
        r.atom_sasa = np.zeros(2 * n, np.float32)
        r.seg_sasa = np.zeros(2 * len(s["seg_be"]), np.float32)
        r.protein = np.zeros((2, 3), np.float32)
    o = [_lib.Outputs(None, r.atom_sasa.ctypes.data, r.seg_sasa.ctypes.data, r.protein.ctypes.data) for r in (cpx, iso)]
    gp = np.ascontiguousarray(group)
    rc = b._L.sasa_b200_batch_run_groups_host(b._h, bad.ctypes.data, None, gp.ctypes.data, C.byref(prm), C.byref(o[0]),
                                              C.byref(o[1]), None)
    assert rc == _lib.ERR_NON_FINITE
    for r, good in ((cpx, good_cpx), (iso, good_iso)):
        assert np.all(np.isnan(r.atom_sasa[n:])) and np.all(np.isnan(r.protein[1]))
        assert np.array_equal(r.atom_sasa[:n], good.atom_sasa[:n])
    # the context stays usable
    again = b.run_groups_host(xyzr, group)
    assert np.array_equal(again[1].counts, good_iso.counts)
    b.close()


def test_process_interface_two_chains(eng, tmp_path):
    from rustsasa_b200 import ChainLevel, ProteinLevel, ResidueLevel, SASAOptions, read_structure
    from tests import synthetic_pdb as sp
    atoms = sp.make_atoms(5, n_res=60, chains="AB")
    pa, _ = sp.write(tmp_path, "ab", atoms)
    alone = [sp.write(tmp_path, c, [a for a in atoms if a["chain"] == c])[0] for c in "AB"]
    st = read_structure(pa)
    for level in (ResidueLevel, ChainLevel, ProteinLevel):
        opt = SASAOptions(level)
        r = opt.process_interface([st], engine=eng)[0]
        assert r.complex == opt.process(st, eng)
        sa, sb = (opt.process(read_structure(p), eng) for p in alone)
        if level is ProteinLevel:
            assert close_enough(r.isolated.global_total, sa.global_total + sb.global_total)
            assert r.buried_area == pytest.approx(r.isolated.global_total - r.complex.global_total)
            assert r.buried_area > 0
        else:
            assert r.isolated == sa + sb
        # both chains in one group: isolated == complex
        r1 = opt.process_interface([st], chain_groups=["AB"], engine=eng)[0]
        assert r1.isolated == r1.complex and r1.buried_area == 0.0
    a = SASAOptions.atom_level().process_interface([st], engine=eng)[0]
    sa, sb = (SASAOptions.atom_level().process(read_structure(p), eng) for p in alone)
    assert np.array_equal(a.isolated, np.concatenate([sa, sb]))
