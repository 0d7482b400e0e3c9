"""Pairwise buried area: sasa_b200_batch_run_group_pairs_host / _device against the CPU oracle.

For atom i of group g and another group h, the reference is buried_h(i) = count_iso(i) - count_{g+h}(i): the oracle on every group
alone, and the oracle on the atoms of g and h together (original order, same id rule) for every contacting pair.  The slots must
hold the partners with a non-zero count in ascending label order, the areas must be the reference's area expression on those
counts bit for bit, and the complex / isolated outputs must equal run_groups_host bit for bit.
"""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PROBE = 1.4
NONE = 0xFFFFFFFF
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def eng():
    from rustsasa_b200 import Engine
    e = Engine()
    yield e
    e.close()


@pytest.fixture(scope="module")
def grouped_capacity(tmp_path_factory):
    """Atom capacity of the widest fused configuration (1024 threads x 1 CTA) in grouped runs, read from max_atoms of
    rustsasa_b200/csrc/sasa_small.cuh (host code, compiled with nvcc; no GPU needed)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = shutil.which("nvcc")
    assert nvcc, "nvcc is needed to read the fused kernel's capacity"
    d = tmp_path_factory.mktemp("cap")
    src, exe = str(d / "cap.cu"), str(d / "cap")
    with open(src, "w") as fh:
        fh.write('#include <cstdio>\n#include "sasa_small.cuh"\n'
                 'int main() { printf("%u\\n", sasa::max_atoms(1024, 1, 16384, false, true)); return 0; }\n')
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-I",
                        os.path.join(ROOT, "rustsasa_b200", "csrc"), "-o", exe, src],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    assert r.returncode == 0, r.stdout
    return int(subprocess.run([exe], stdout=subprocess.PIPE, text=True, check=True).stdout.split()[0])


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


def contacting_pairs(xyzr, group, probe):
    """Pairs of labels (a < b) with at least one pair of atoms close enough to occlude each other."""
    from scipy.spatial import cKDTree
    rmax = float(xyzr[:, 3].max()) if xyzr.shape[0] else 0.0
    pairs = cKDTree(xyzr[:, :3].astype(np.float64)).query_pairs(2 * rmax + 2 * probe + 0.01, output_type="ndarray")
    ga, gb = group[pairs[:, 0]], group[pairs[:, 1]]
    x = ga != gb
    return sorted({(int(min(a, b)), int(max(a, b))) for a, b in zip(ga[x], gb[x])})


def pair_reference(oracle, xyzr, group, probe=PROBE, n_points=100, lanes=8, ids=None):
    """(iso counts, per atom {partner: buried count > 0}) from the oracle on every group alone and every contacting g + h."""
    iso, _ = iso_oracle(oracle, xyzr, group, probe, n_points, lanes, ids)
    buried = [dict() for _ in range(xyzr.shape[0])]
    for a, b in contacting_pairs(xyzr, group, probe):
        m = np.nonzero((group == a) | (group == b))[0]
        o = oracle.calculate_sasa_internal(xyzr[m], probe, n_points, lanes=lanes, threads=0 if m.size > 10000 else 1,
                                           ids=None if ids is None else ids[m])
        d = iso[m].astype(np.int64) - o["counts"].astype(np.int64)
        assert np.all(d >= 0)
        for i, di in zip(m[d > 0], d[d > 0]):
            buried[i][int(b if group[i] == a else a)] = int(di)
    return iso, buried


def area_expr(radius, probe, count, n_points):
    """The oracle's area expression ((4*pi_f32 * r^2) * count) * (1/n) in float32, same operation order."""
    r = (np.asarray(radius, np.float32) + np.float32(probe)).astype(np.float32)
    sa = (np.float32(4.0) * np.float32(np.pi)) * (r * r)
    return ((sa * np.asarray(count, np.float32)) * (np.float32(1.0) / np.float32(n_points))).astype(np.float32)


def expected_slots(buried, radius, K, probe, n_points):
    n = len(buried)
    partner = np.full((n, K), NONE, np.uint32)
    counts = np.zeros((n, K), np.uint32)
    for i, b in enumerate(buried):
        for s, h in enumerate(sorted(b)[:K]):
            partner[i, s], counts[i, s] = h, b[h]
    area = area_expr(np.repeat(np.asarray(radius, np.float32)[:, None], K, axis=1), probe, counts, n_points)
    area[counts == 0] = 0.0
    return partner, counts, area


def check_slots(pairs, buried, xyzr, K, probe, n_points, a0=0, tag=None):
    n = len(buried)
    partner, counts, area = expected_slots(buried, xyzr[:, 3], K, probe, n_points)
    assert np.array_equal(pairs.partner[a0:a0 + n], partner), tag
    assert np.array_equal(pairs.buried_counts[a0:a0 + n], counts), tag
    assert np.array_equal(pairs.buried_area[a0:a0 + n].view(np.uint32), area.view(np.uint32)), tag


def check_invariants(pairs, cpx, iso, a0, a1):
    bc = pairs.buried_counts[a0:a1].astype(np.int64)
    total = iso.counts[a0:a1].astype(np.int64) - cpx.counts[a0:a1].astype(np.int64)
    assert np.all(bc.max(axis=1) <= total)
    assert np.all(total <= bc.sum(axis=1))
    used = bc > 0
    assert np.array_equal(used, pairs.partner[a0:a1] != NONE)
    # slots in use come first, in strictly ascending label order
    for row, u in zip(pairs.partner[a0:a1], used):
        k = int(u.sum())
        assert np.all(u[:k]) and not np.any(u[k:])
        assert np.all(np.diff(row[:k].astype(np.int64)) > 0)


def run_and_compare(b, xyzr, group, cls=None, K=4, **kw):
    cpx, iso, pairs = b.run_group_pairs_host(xyzr, group, cls, max_partners=K, **kw)
    rc, ri = b.run_groups_host(xyzr, group, cls, **kw)
    for f in ("counts", "atom_sasa", "seg_sasa", "protein"):
        for x, y in ((cpx, rc), (iso, ri)):
            u, v = getattr(x, f), getattr(y, f)
            assert (u is None and v is None) or np.array_equal(np.asarray(u).view(np.uint32), np.asarray(v).view(np.uint32)), f
    return cpx, iso, pairs


def chain_groups(golden, s):
    g = np.zeros(s["xyzr"].shape[0], np.uint32)
    for ci, (b, e) in enumerate(golden.chain_ranges(s)):
        g[b:e] = ci
    return g


def octants(xyzr, n_groups):
    """4 or 8 spatial groups: quadrants / octants about the centroid, so atoms near the cuts have 2-3 partners."""
    c = xyzr[:, :3] - xyzr[:, :3].mean(axis=0)
    g = (c[:, 0] > 0).astype(np.uint32) + 2 * (c[:, 1] > 0).astype(np.uint32)
    if n_groups == 8:
        g += 4 * (c[:, 2] > 0).astype(np.uint32)
    return g


def sectors(xyzr, n_groups):
    c = xyzr[:, :3] - xyzr[:, :3].mean(axis=0)
    ang = np.arctan2(c[:, 1], c[:, 0]) + np.pi
    return np.minimum((ang / (2 * np.pi) * n_groups).astype(np.uint32), n_groups - 1)


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
    K = 8
    cpx, iso, pairs = run_and_compare(b, xyzr, group, K=K, n_points=n_points)
    assert pairs.needed <= K
    for i, s in enumerate(ss):
        a0, a1 = int(off[i]), int(off[i + 1])
        iso_ref, buried = pair_reference(oracle, s["xyzr"], group[a0:a1], n_points=n_points)
        assert np.array_equal(iso.counts[a0:a1], iso_ref), names[i]
        check_slots(pairs, buried, s["xyzr"], K, PROBE, n_points, a0, names[i])
        check_invariants(pairs, cpx, iso, a0, a1)
    assert pairs.needed == int((pairs.buried_counts > 0).sum(axis=1).max()) > 0
    b.close()


@pytest.mark.parametrize("lanes", [4, 8])
def test_many_partners(eng, oracle, golden, lanes):
    rng = np.random.default_rng(4100 + lanes)
    structs, groups = [], []
    for name, ng in (("4xfj", 8), ("example.cif", 4)):
        s = golden.structure(name)["xyzr"]
        structs.append(s)
        groups.append(octants(s, ng))
    for t in range(4):
        n = int(rng.integers(300, 1500))
        density = float(rng.choice([0.03, 0.057, 0.12]))
        side = (n / density) ** (1.0 / 3.0)
        xyz = rng.uniform(0.0, side, size=(n, 3)) + rng.uniform(-200, 200, size=3)
        rad = rng.uniform(0.8, 2.4, size=n)
        s = np.concatenate([xyz, rad[:, None]], axis=1).astype(np.float32)
        structs.append(s)
        groups.append(sectors(s, int(rng.integers(4, 9))) + np.uint32(t * 100))
    off = np.cumsum([0] + [s.shape[0] for s in structs]).astype(np.uint64)
    xyzr, group = np.concatenate(structs), np.concatenate(groups)
    b = eng.batch(off)
    K = 16
    cpx, iso, pairs = run_and_compare(b, xyzr, group, K=K, simd_lanes=lanes, want=("counts", "atom"))
    assert pairs.needed >= 3   # atoms near where three or more regions meet
    for i, s in enumerate(structs):
        a0, a1 = int(off[i]), int(off[i + 1])
        _, buried = pair_reference(oracle, s, groups[i], lanes=lanes)
        check_slots(pairs, buried, s, K, PROBE, 100, a0, i)
        check_invariants(pairs, cpx, iso, a0, a1)
    b.close()


def test_two_groups(eng, golden):
    s = golden.structure("4xfj")["xyzr"]
    n = s.shape[0]
    group = (s[:, 0] > np.median(s[:, 0])).astype(np.uint32) * 5 + 2
    b = eng.batch([0, n])
    cpx, iso, pairs = run_and_compare(b, s, group, K=2, want=("counts", "atom"))
    total = iso.counts.astype(np.int64) - cpx.counts.astype(np.int64)
    assert np.array_equal(pairs.buried_counts[:, 0].astype(np.int64), total)
    assert np.array_equal(pairs.partner[:, 0] != NONE, total > 0)
    assert np.all(pairs.partner[total > 0, 0] == np.where(group[total > 0] == 2, 7, 2))
    assert np.all(pairs.partner[:, 1] == NONE) and np.all(pairs.buried_counts[:, 1] == 0) and np.all(pairs.buried_area[:, 1] == 0)
    assert pairs.needed == 1
    # one group for the whole structure: no partners
    _, _, one = run_and_compare(b, s, np.full(n, 3, np.uint32), K=1, want=("counts",))
    assert np.all(one.partner == NONE) and np.all(one.buried_counts == 0) and one.needed == 0
    b.close()


def _cluster(rng, n, side):
    xyz = rng.uniform(0.0, side, size=(n, 3))
    return np.concatenate([xyz, rng.uniform(1.2, 2.0, size=(n, 1))], axis=1).astype(np.float32)


@pytest.mark.parametrize("with_cls", [False, True])
def test_paths(eng, oracle, golden, grouped_capacity, with_cls):
    """The fused kernel, a structure above the grouped fused capacity (the large-structure path), a dense cluster with more than
    96 neighbours per atom (the streaming routine) -- at 100 points -- and every one of them again at 960 points (the
    large-structure path throughout), with and without id classes."""
    rng = np.random.default_rng(77 + with_cls)
    small = golden.structure("example.cif")["xyzr"]
    n_big = grouped_capacity + 300
    big = _cluster(rng, n_big, (n_big / 0.057) ** (1.0 / 3.0))
    dense = _cluster(rng, 600, 12.0)
    structs = [small, big, dense]
    groups = [sectors(s, 3) for s in structs]
    ids = [rng.integers(0, s.shape[0] // 2, size=s.shape[0]).astype(np.uint64) for s in structs] if with_cls else None
    off = np.cumsum([0] + [s.shape[0] for s in structs]).astype(np.uint64)
    xyzr, group = np.concatenate(structs), np.concatenate(groups)
    cls = None
    if with_cls:
        cls = np.concatenate([np.unique(ids[i], return_inverse=True)[1].astype(np.uint32) + np.uint32(off[i])
                              for i in range(len(structs))])
    b = eng.batch(off)
    for n_points in (100, 960):
        cpx, iso, pairs = run_and_compare(b, xyzr, group, cls, K=4, n_points=n_points, want=("counts", "atom"))
        if n_points == 100:
            assert cpx.stats["streamed_atoms"] > 0
        for i, s in enumerate(structs):
            a0, a1 = int(off[i]), int(off[i + 1])
            _, buried = pair_reference(oracle, s, groups[i], n_points=n_points, ids=None if ids is None else ids[i])
            check_slots(pairs, buried, s, 4, PROBE, n_points, a0, (i, n_points))
            check_invariants(pairs, cpx, iso, a0, a1)
            assert np.any(pairs.buried_counts[a0:a1] > 0), (i, n_points)
    b.close()


def test_too_few_slots(eng, oracle, golden):
    from rustsasa_b200 import _lib
    from rustsasa_b200.engine import SasaB200Error
    # 17 atoms, one group per atom: no atom can have more partners than the 16 slots a run may ask for
    s = golden.structure("example.cif")["xyzr"][:17]
    n = s.shape[0]
    group = np.arange(n, dtype=np.uint32)[::-1].copy()   # labels against atom order
    _, buried = pair_reference(oracle, s, group)
    need = max(len(x) for x in buried)
    assert 1 < need <= 16
    b = eng.batch([0, n])
    rc, ri = b.run_groups_host(s, group)
    with pytest.raises(SasaB200Error) as e:
        b.run_group_pairs_host(s, group, max_partners=1)
    assert e.value.code == _lib.ERR_INVALID_ARGUMENT
    assert e.value.needed == need and ("max_partners = %d" % need) in str(e.value)
    cpx, iso, pairs = e.value.result
    assert pairs.needed == need
    for x, y in ((cpx, rc), (iso, ri)):
        for f in ("counts", "atom_sasa", "protein"):
            assert np.array_equal(getattr(x, f), getattr(y, f)), f
    check_slots(pairs, buried, s, 1, PROBE, 100)   # the lowest label of every atom
    _, _, full = b.run_group_pairs_host(s, group, max_partners=need)
    check_slots(full, buried, s, need, PROBE, 100)
    assert full.needed == need
    # the device form defers the error to sync
    import torch
    _, _, d = b.run_group_pairs_device(torch.from_numpy(s).cuda(), torch.from_numpy(group.view(np.int32)).cuda(), max_partners=1)
    with pytest.raises(SasaB200Error) as e:
        b.sync()
    assert e.value.code == _lib.ERR_INVALID_ARGUMENT and ("max_partners = %d" % need) in str(e.value)
    assert int(d.needed.cpu()[0]) == need
    assert np.array_equal(d.partner.cpu().numpy().view(np.uint32), pairs.partner)
    b.sync()   # cleared
    b.close()


def test_device_entry_equals_host(eng, golden):
    import torch
    names = [n for n in golden.names if len(np.unique(golden.structure(n)["res_chain"])) > 1][:10]
    ss = [golden.structure(n) for n in names]
    off = np.cumsum([0] + [s["xyzr"].shape[0] for s in ss]).astype(np.uint64)
    seg_off = np.cumsum([0] + [len(s["seg_be"]) for s in ss]).astype(np.uint64)
    xyzr = np.concatenate([s["xyzr"] for s in ss])
    group = np.concatenate([octants(s["xyzr"], 8) for s in ss])
    b = eng.batch(off, np.concatenate([s["seg_be"] for s in ss]), seg_off, np.concatenate([s["polar"] for s in ss]))
    h = b.run_group_pairs_host(xyzr, group, max_partners=8)
    d = b.run_group_pairs_device(torch.from_numpy(xyzr).cuda(), torch.from_numpy(group.astype(np.int32)).cuda(), max_partners=8)
    torch.cuda.synchronize()
    b.sync()
    for hr, dr in zip(h[:2], d[:2]):
        assert np.array_equal(hr.counts, dr.counts.cpu().numpy().astype(np.uint32))
        for f in ("atom_sasa", "seg_sasa", "protein"):
            assert np.array_equal(getattr(hr, f), getattr(dr, f).cpu().numpy()), f
    hp, dp = h[2], d[2]
    assert np.array_equal(hp.partner, dp.partner.cpu().numpy().view(np.uint32))
    assert np.array_equal(hp.buried_counts, dp.buried_counts.cpu().numpy().view(np.uint32))
    assert np.array_equal(hp.buried_area.view(np.uint32), dp.buried_area.cpu().numpy().view(np.uint32))
    assert hp.needed == int(dp.needed.cpu()[0])
    b.close()


def test_errors(eng, golden):
    from rustsasa_b200 import _lib
    from rustsasa_b200.engine import SasaB200Error
    s = golden.structure("example.cif")["xyzr"]
    n = s.shape[0]
    b = eng.batch([0, n])
    group = (np.arange(n) % 3).astype(np.uint32)
    for flags in (_lib.FLAG_BOUNDARY_STATS, _lib.FLAG_FORCE_STREAMING):
        with pytest.raises(SasaB200Error) as e:
            b.run_group_pairs_host(s, group, flags=flags)
        assert e.value.code == _lib.ERR_UNSUPPORTED
    for K in (0, 17):
        with pytest.raises(SasaB200Error) as e:
            b.run_group_pairs_host(s, group, max_partners=K)
        assert e.value.code == _lib.ERR_INVALID_ARGUMENT
    outs = _lib.Outputs(None, None, None, None)
    prm = _lib.Params(PROBE, 100, 8, -1, 0)
    part = np.zeros((n, 2), np.uint32)
    good = _lib.PairOutputs(2, part.ctypes.data, None, None, None)
    no_partner = _lib.PairOutputs(2, None, None, None, None)
    run = b._L.sasa_b200_batch_run_group_pairs_host
    assert run(b._h, s.ctypes.data, None, None, C.byref(prm), C.byref(outs), C.byref(outs), C.byref(good), None) == _lib.ERR_INVALID_ARGUMENT
    assert run(b._h, s.ctypes.data, None, group.ctypes.data, C.byref(prm), C.byref(outs), C.byref(outs), None, None) == _lib.ERR_INVALID_ARGUMENT
    assert run(b._h, s.ctypes.data, None, group.ctypes.data, C.byref(prm), C.byref(outs), C.byref(outs), C.byref(no_partner),
               None) == _lib.ERR_INVALID_ARGUMENT
    assert run(b._h, s.ctypes.data, None, group.ctypes.data, C.byref(prm), C.byref(outs), None, C.byref(good), None) == _lib.ERR_INVALID_ARGUMENT
    # every output but the partner labels NULL is a valid call
    assert run(b._h, s.ctypes.data, None, group.ctypes.data, C.byref(prm), C.byref(outs), C.byref(outs), C.byref(good), None) == _lib.OK
    _, _, ref = b.run_group_pairs_host(s, group, max_partners=2)
    assert np.array_equal(part, ref.partner)
    # the device form checks alike
    dev = b._L.sasa_b200_batch_run_group_pairs_device
    bad_k = _lib.PairOutputs(0, part.ctypes.data, None, None, None)
    assert dev(b._h, s.ctypes.data, None, group.ctypes.data, C.byref(prm), C.byref(outs), C.byref(outs), C.byref(bad_k),
               None) == _lib.ERR_INVALID_ARGUMENT
    assert dev(b._h, s.ctypes.data, None, group.ctypes.data, C.byref(prm), C.byref(outs), C.byref(outs), None, None) == _lib.ERR_INVALID_ARGUMENT
    b.close()


def test_non_finite_and_empty(eng, oracle, golden):
    from rustsasa_b200 import _lib
    from rustsasa_b200.engine import SasaB200Error
    s = golden.structure("example.cif")["xyzr"]
    n = s.shape[0]
    group = octants(s, 4)
    b = eng.batch([0, n, 2 * n, 3 * n])
    xyzr = np.concatenate([s, s, s])
    groups = np.tile(group, 3)
    _, _, good = b.run_group_pairs_host(xyzr, groups, max_partners=4)
    bad = xyzr.copy()
    bad[n + 5, 2] = np.inf
    with pytest.raises(SasaB200Error) as e:
        b.run_group_pairs_host(bad, groups, max_partners=4)
    assert e.value.code == _lib.ERR_NON_FINITE
    cpx, iso, pairs = e.value.result
    for lo, hi in ((0, n), (2 * n, 3 * n)):
        for f in ("partner", "buried_counts"):
            assert np.array_equal(getattr(pairs, f)[lo:hi], getattr(good, f)[lo:hi])
        assert np.array_equal(pairs.buried_area[lo:hi].view(np.uint32), good.buried_area[lo:hi].view(np.uint32))
    assert np.all(pairs.partner[n:2 * n] == NONE) and np.all(pairs.buried_counts[n:2 * n] == 0)
    assert np.all(np.isnan(pairs.buried_area[n:2 * n]))
    assert np.all(np.isnan(cpx.atom_sasa[n:2 * n])) and np.all(np.isnan(iso.atom_sasa[n:2 * n]))
    _, buried = pair_reference(oracle, s, group)
    check_slots(good, buried, s, 4, PROBE, 100, 2 * n)
    b.close()
    # an empty batch: nothing to do
    e0 = eng.batch(np.zeros(1, np.uint64))
    cpx, iso, pairs = e0.run_group_pairs_host(np.zeros((0, 4), np.float32), np.zeros(0, np.uint32))
    assert pairs.partner.shape == (0, 4) and pairs.needed == 0
    e0.close()


def test_process_interface_pairs(eng, oracle, tmp_path):
    from rustsasa_b200 import ProteinLevel, ResidueLevel, SASAOptions, group_pair_table, read_structure
    from tests import synthetic_pdb as sp
    pa, _ = sp.write(tmp_path, "abc", sp.make_atoms(5, n_res=60, chains="ABC"))
    st = read_structure(pa)
    for level in (ResidueLevel, ProteinLevel):
        opt = SASAOptions(level)
        r = opt.process_interface_pairs([st], engine=eng, max_partners=1)[0]   # too few slots: reruns with as many as needed
        ref = opt.process_interface([st], engine=eng)[0]
        assert r.interface == ref
        p = opt._pack(st)
        group = SASAOptions._chain_groups(p.atom_chain, [])
        _, buried = pair_reference(oracle, p.xyzr, group)
        K = max(1, max(len(x) for x in buried))
        partner, _, area = expected_slots(buried, p.xyzr[:, 3], K, PROBE, 100)
        table = group_pair_table(partner, area, group, [0, group.shape[0]])[0]
        assert len(table) >= 2
        assert [(x.group_a, x.group_b, x.buried_a, x.buried_b) for x in r.pairs] == table
        chains = {int(g): c for g, c in zip(group, p.atom_chain)}
        assert all(x.chains_a == chains[x.group_a] and x.chains_b == chains[x.group_b] for x in r.pairs)
        if level is ResidueLevel:
            assert len(r.residue_partners) == len(p.seg_be)
            tot = sum(v for d in r.residue_partners for v in d.values())
            assert tot == pytest.approx(sum(x.buried_a + x.buried_b for x in r.pairs))
        else:
            assert r.residue_partners is None
