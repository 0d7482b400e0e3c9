"""Pairwise buried area of MD frames: sasa_b200_batch_run_group_pairs_frames_host / _submit_, and trajectory_interface(pairs=True).

The complex and isolated outputs must equal the frames run and the grouped frames run bit for bit.  The device-side sums must
equal, bit for bit, the host reduction of today's route: the pairs run on the float4 packing with the labels tiled over the
frames, reduced with group_pair_table (pair_area) and with float64 atom-order sums per segment (seg_pair_area).  A few frames are
also checked against the CPU oracle run on every group alone and on every contacting pair of groups.  Every path a grouped frames
run takes is reached: the fused kernel reading the 12-byte coordinates, frames above the grouped fused capacity, and n_points >
128.
"""
import ctypes as C

import numpy as np
import pytest

from tests.test_gpu_frames_groups import float4_frames, frames_batch, grouped_capacity, plane_groups  # noqa: F401
from tests.test_gpu_group_pairs import area_expr, pair_reference, sectors

pytestmark = pytest.mark.gpu

PROBE = 1.4
ALL = ("counts", "atom", "seg", "protein")
FIELDS = ("counts", "atom_sasa", "seg_sasa", "protein")


@pytest.fixture(scope="module")
def eng():
    from rustsasa_b200 import Engine
    e = Engine()
    yield e
    e.close()


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64 if a.dtype == np.float64 else np.uint32)


def same(a, b, fields=FIELDS):
    for f in fields:
        x, y = getattr(a, f), getattr(b, f)
        assert (x is None) == (y is None), f
        if x is not None:
            assert np.array_equal(bits(x), bits(y)), f


def host_sums(b, xyz, radii, group, L, n_points=100, lanes=8, seg_be=None):
    """Today's route: the pairs run on float4 frames with tiled labels (K = max(1, L - 1)), reduced on the host -- the dense
    form of group_pair_table, and per segment the float64 atom-order sums of the slots."""
    from rustsasa_b200 import group_pair_table
    F, N = xyz.shape[:2]
    tiled = np.tile(group, F)
    _, _, pairs = b.run_group_pairs_host(float4_frames(xyz, radii), tiled, None, PROBE, n_points, lanes, want=("protein",),
                                         max_partners=max(1, L - 1))
    dense = np.zeros((F, L, L), np.float64)
    for s, rows in enumerate(group_pair_table(pairs.partner, pairs.buried_area, tiled, np.arange(F + 1) * N)):
        for g, h, gh, hg in rows:
            dense[s, g, h], dense[s, h, g] = gh, hg
    seg = None
    if seg_be is not None:
        # per atom and label the area of the slot with that partner, or 0.0 (an atom has each partner at most once; adding 0.0
        # leaves a sum of non-negative terms unchanged), summed sequentially (cumsum) over each segment in atom order
        per = np.zeros((F * N, L), np.float64)
        for r in range(pairs.partner.shape[1]):
            p = pairs.partner[:, r]
            m = p < L
            per[np.nonzero(m)[0], p[m]] = pairs.buried_area[m, r].astype(np.float64)
        seg = np.zeros((F * len(seg_be), L), np.float64)
        for f in range(F):
            for q, (b0, b1) in enumerate(seg_be):
                if b1 > b0:
                    seg[f * len(seg_be) + q] = np.cumsum(per[f * N + b0:f * N + b1], axis=0)[-1]
    return dense, seg


def check_route(b, md, group, L, n_points=100, lanes=8, want=ALL):
    """The new entry against the frames run, the grouped frames run and the host route, bit for bit."""
    cpx, iso, sums = b.run_group_pairs_frames_host(md.xyz, md.radii, group, L, PROBE, n_points, lanes, want=want)
    same(cpx, b.run_frames_host(md.xyz, md.radii, PROBE, n_points, lanes, want=want))
    ref_cpx, ref_iso = b.run_groups_frames_host(md.xyz, md.radii, group, PROBE, n_points, lanes, want=want)
    same(cpx, ref_cpx)
    same(iso, ref_iso)
    dense, seg = host_sums(b, md.xyz, md.radii, group, L, n_points, lanes, md.seg_be if b.n_seg else None)
    assert sums.n_labels == L and sums.pair_area.shape == dense.shape
    assert np.array_equal(bits(sums.pair_area), bits(dense))
    if b.n_seg:
        assert np.array_equal(bits(sums.seg_pair_area), bits(seg))
    else:
        assert sums.seg_pair_area is None
    P = sums.pair_area
    assert np.all(P >= 0) and not np.any(np.einsum("fgg->fg", P))
    present = np.zeros(L, bool)
    present[np.unique(group)] = True
    assert not np.any(P[:, ~present, :]) and not np.any(P[:, :, ~present])
    return cpx, iso, sums


@pytest.mark.parametrize("lanes", [4, 8])
@pytest.mark.parametrize("n_points", [100, 960])
def test_bit_equal_to_host_route(eng, n_points, lanes):
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=12, n_atoms=1200, seed=11)
    F, N = md.xyz.shape[:2]
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    for L, group in ((2, plane_groups(md.xyz)), (4, sectors(md.xyz.mean(axis=0), 4))):
        cpx, _, sums = check_route(b, md, group, L, n_points, lanes)
        assert np.all(sums.pair_area[:, 0, 1] > 0) and np.all(sums.pair_area[:, 1, 0] > 0)
        if n_points <= 128:
            assert cpx.stats["gpu_launches"] < F   # the fused kernel reads the 12-byte frames: a few launches per chunk
        else:
            assert cpx.stats["gpu_launches"] > F   # every frame on the large-structure path
    b.close()


@pytest.mark.parametrize("n_points", [100, 960])
def test_oracle_parity(eng, oracle, n_points):
    """The sums against the oracle: float64 atom-order sums of the area expression over the buried counts of every atom."""
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=2, n_atoms=700, seed=5)
    F, N = md.xyz.shape[:2]
    G = len(md.seg_be)
    group = sectors(md.xyz.mean(axis=0), 3)
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    _, _, sums = b.run_group_pairs_frames_host(md.xyz, md.radii, group, 3, n_points=n_points)
    for f in range(F):
        xyzr = np.concatenate([md.xyz[f], md.radii[:, None]], axis=1).astype(np.float32)
        _, buried = pair_reference(oracle, xyzr, group, n_points=n_points)
        P = np.zeros((3, 3), np.float64)
        per = np.zeros((N, 3), np.float64)
        for i, d in enumerate(buried):
            for h, c in d.items():
                v = float(area_expr(md.radii[i], PROBE, c, n_points))
                P[group[i], h] += v
                per[i, h] = v
        assert np.array_equal(bits(sums.pair_area[f]), bits(P)), f
        for q, (b0, b1) in enumerate(md.seg_be):
            acc = [0.0, 0.0, 0.0]
            for i in range(b0, b1):
                for h in range(3):
                    acc[h] += per[i, h]
            assert np.array_equal(bits(sums.seg_pair_area[f * G + q]), bits(np.array(acc))), (f, q)
    b.close()


@pytest.mark.parametrize("n_points", [100, 128])
def test_frames_above_grouped_fused_capacity(eng, grouped_capacity, n_points):  # noqa: F811
    from rustsasa_b200 import workloads as W
    cap, plain_cap = grouped_capacity
    md = W.md_trajectory(n_frames=3, n_atoms=cap + 300, seed=21)
    F, N = md.xyz.shape[:2]
    assert cap < N <= plain_cap, (cap, N, plain_cap)
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    cpx, _, _ = check_route(b, md, plane_groups(md.xyz), 2, n_points, want=("counts", "protein"))
    assert cpx.stats["gpu_launches"] > F
    check_route(b, md, np.random.default_rng(3).integers(0, 5, size=N).astype(np.uint32), 5, n_points, want=("protein",))
    b.close()


@pytest.mark.parametrize("n_points", [129, 960])
def test_more_than_128_points_every_frame_on_the_large_path(eng, n_points):
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=4, n_atoms=700, seed=9)
    F, N = md.xyz.shape[:2]
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    cpx, _, _ = check_route(b, md, sectors(md.xyz.mean(axis=0), 6), 6, n_points)
    assert cpx.stats["gpu_launches"] > F
    b.close()


def test_labels(eng):
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=5, n_atoms=1000, seed=13)
    F, N = md.xyz.shape[:2]
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    # one label: nothing is buried by a partner
    _, _, sums = check_route(b, md, np.zeros(N, np.uint32), 1)
    assert sums.pair_area.shape == (F, 1, 1) and not np.any(sums.pair_area) and not np.any(sums.seg_pair_area)
    # two labels: the one partner buries everything the complex hides of an atom, exactly
    group = plane_groups(md.xyz)
    cpx, iso, sums = check_route(b, md, group, 2)
    area = area_expr(np.tile(md.radii, F), PROBE, iso.counts.astype(np.int64) - cpx.counts.astype(np.int64), 100)
    for f in range(F):
        a = slice(f * N, (f + 1) * N)
        for g in (0, 1):
            m = np.nonzero(group == g)[0]
            expect = np.cumsum(area[a][m].astype(np.float64))[-1]
            assert bits(sums.pair_area[f, g, 1 - g]) == bits(expect), (f, g)
    # random labels, some of them with no atoms
    rng = np.random.default_rng(7)
    for L in (3, 5, 7):
        group = rng.integers(0, L, size=N).astype(np.uint32)
        group[group == L - 2] = L - 1 if L > 3 else 0
        check_route(b, md, group, L, want=("protein",))
    # seventeen labels: sectors, and random labels, where atoms have many partners and the sixteen slots fill up
    check_route(b, md, sectors(md.xyz.mean(axis=0), 17), 17, want=("protein",))
    group = rng.integers(0, 17, size=N).astype(np.uint32)
    _, _, sums = check_route(b, md, group, 17, want=("protein",))
    _, _, pairs = b.run_group_pairs_host(float4_frames(md.xyz, md.radii), np.tile(group, F), max_partners=16, want=("protein",))
    assert pairs.needed >= 6
    b.close()


@pytest.mark.parametrize("n_points", [100, 960])
def test_non_finite_frame(eng, n_points):
    from rustsasa_b200 import SasaB200Error, _lib
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=5, n_atoms=900, seed=3)
    F, N = md.xyz.shape[:2]
    G = len(md.seg_be)
    group = sectors(md.xyz.mean(axis=0), 3)
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    good = b.run_group_pairs_frames_host(md.xyz, md.radii, group, 3, n_points=n_points, want=ALL)
    bad = md.xyz.copy()
    bad[2, 17, 1] = np.nan
    res = (b._host_outputs(ALL, "numpy"), b._host_outputs(ALL, "numpy"), b._pair_sums(3, True, "numpy"))
    res[2].pair_area[:] = 7.0
    res[2].seg_pair_area[:] = 7.0
    with pytest.raises(SasaB200Error) as e:
        b.run_group_pairs_frames_host(bad, md.radii, group, 3, n_points=n_points, want=ALL, result=res)
    assert e.value.code == _lib.ERR_NON_FINITE
    for f in range(F):
        a, s = slice(f * N, (f + 1) * N), slice(f * G, (f + 1) * G)
        if f == 2:
            assert np.all(np.isnan(res[2].pair_area[f])) and np.all(np.isnan(res[2].seg_pair_area[s]))
            assert np.all(np.isnan(res[0].atom_sasa[a])) and np.all(np.isnan(res[1].protein[f]))
        else:
            assert np.array_equal(bits(res[2].pair_area[f]), bits(good[2].pair_area[f])), f
            assert np.array_equal(bits(res[2].seg_pair_area[s]), bits(good[2].seg_pair_area[s])), f
            for r, g in zip(res[:2], good[:2]):
                assert np.array_equal(bits(r.atom_sasa[a]), bits(g.atom_sasa[a])) and np.array_equal(r.counts[a], g.counts[a]), f
    # the context stays usable
    again = b.run_group_pairs_frames_host(md.xyz, md.radii, group, 3, n_points=n_points, want=ALL)
    assert np.array_equal(bits(again[2].pair_area), bits(good[2].pair_area))
    b.close()


def test_errors_and_empty_batch(eng):
    from rustsasa_b200 import SasaB200Error, _lib
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=2, n_atoms=300, seed=1)
    F, N = md.xyz.shape[:2]
    group = plane_groups(md.xyz)
    b = frames_batch(eng, F, N)
    L, h = b._L, b._h
    x, r, g = md.xyz.ctypes.data, md.radii.ctypes.data, group.ctypes.data
    outs = _lib.Outputs(None, None, None, None)
    prm = _lib.Params(PROBE, 100, 8, -1, 0)
    area = np.zeros((F, 2, 2), np.float64)
    sums = _lib.PairSums(2, area.ctypes.data, None)

    def run(*args, o=C.byref(outs), oi=C.byref(outs), s=C.byref(sums), p=C.byref(prm), batch=h):
        rc = L.sasa_b200_batch_run_group_pairs_frames_host(batch, *args, p, o, oi, s, None)
        job = C.c_void_p()
        rc2 = L.sasa_b200_batch_submit_group_pairs_frames_host(batch, *args, p, o, oi, s, C.byref(job))
        if rc2 == _lib.OK:
            L.sasa_b200_job_wait(job, None)
        assert rc == rc2, (rc, rc2)
        return rc

    assert run(x, r, g) == _lib.OK
    for args in ((None, r, g), (x, None, g), (x, r, None)):
        assert run(*args) == _lib.ERR_INVALID_ARGUMENT, args
    assert run(x, r, g, oi=None) == _lib.ERR_INVALID_ARGUMENT
    assert run(x, r, g, s=None) == _lib.ERR_INVALID_ARGUMENT
    assert run(x, r, g, s=C.byref(_lib.PairSums(2, None, None))) == _lib.ERR_INVALID_ARGUMENT
    big = np.zeros((F, 18, 18), np.float64)
    for n_labels in (0, 18):
        assert run(x, r, g, s=C.byref(_lib.PairSums(n_labels, big.ctypes.data, None))) == _lib.ERR_INVALID_ARGUMENT, n_labels
    g3 = group.copy()
    g3[N - 1] = 2   # a label >= n_labels
    assert run(x, r, g3.ctypes.data) == _lib.ERR_INVALID_ARGUMENT
    assert b"n_labels" in L.sasa_b200_last_error(eng._h)
    for flags in (_lib.FLAG_BOUNDARY_STATS, _lib.FLAG_FORCE_STREAMING):
        with pytest.raises(SasaB200Error) as e:
            b.run_group_pairs_frames_host(md.xyz, md.radii, group, 2, flags=flags)
        assert e.value.code == _lib.ERR_UNSUPPORTED
    b.close()
    # frames of unequal size
    u = eng.batch(np.array([0, N, 2 * N - 1], np.uint64))
    assert run(x, r, g, batch=u._h) == _lib.ERR_INVALID_ARGUMENT
    u.close()
    # a batch of no frames: nothing to do, with or without sums
    e0 = eng.batch([0])
    cpx, iso, s0 = e0.run_group_pairs_frames_host(np.zeros((0, 0, 3), np.float32), np.zeros(0, np.float32), np.zeros(0, np.uint32),
                                                  want=ALL)
    assert cpx.protein.shape == (0, 3) and iso.counts.shape == (0,) and s0.pair_area.shape == (0, 1, 1)
    assert run(None, None, None, s=None, batch=e0._h) == _lib.OK
    e0.close()


def test_submit_wait(eng):
    from rustsasa_b200 import SasaB200Error, _lib
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=8, n_atoms=1000, seed=4)
    F, N = md.xyz.shape[:2]
    G = len(md.seg_be)
    group = sectors(md.xyz.mean(axis=0), 3)
    b1 = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    b2 = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    ref = b1.run_group_pairs_frames_host(md.xyz, md.radii, group, 3, want=ALL)
    x1 = eng.pinned_empty(md.xyz.shape, np.float32)
    x1[:] = md.xyz
    x2 = eng.pinned_empty(md.xyz.shape, np.float32)
    x2[:] = md.xyz[::-1]
    for _ in range(2):
        j1 = b1.submit_group_pairs_frames_host(x1, md.radii, group, 3, want=ALL)
        j2 = b2.submit_group_pairs_frames_host(x2, md.radii, group, 3, want=ALL)   # two batches in flight at once
        with pytest.raises(SasaB200Error) as e:
            b1.submit_group_pairs_frames_host(x1, md.radii, group, 3, want=ALL)   # b1 already carries a run
        assert e.value.code == _lib.ERR_INVALID_ARGUMENT
        r1, r2 = j1.wait(), j2.wait()
        same(r1[0], ref[0])
        same(r1[1], ref[1])
        assert np.array_equal(bits(r1[2].pair_area), bits(ref[2].pair_area))
        assert np.array_equal(bits(r1[2].seg_pair_area), bits(ref[2].seg_pair_area))
        assert np.array_equal(bits(r2[2].pair_area), bits(ref[2].pair_area[::-1]))   # b2 ran the frames in reverse order
        assert np.array_equal(bits(r2[2].seg_pair_area.reshape(F, G, 3)), bits(ref[2].seg_pair_area.reshape(F, G, 3)[::-1]))
    b1.close()
    b2.close()


def test_trajectory_interface_pairs(eng, tmp_path):
    from rustsasa_b200 import trajectory_interface
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=30, n_atoms=1100, seed=8)
    F, N = md.xyz.shape[:2]
    G = len(md.seg_be)
    dense = sectors(md.xyz.mean(axis=0), 3)
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    _, _, ref = b.run_group_pairs_frames_host(md.xyz, md.radii, dense, 3, want=("protein", "seg"))
    b.close()
    mm = np.lib.format.open_memmap(str(tmp_path / "traj.npy"), mode="w+", dtype=np.float32, shape=md.xyz.shape)
    mm[:] = md.xyz
    mm.flush()
    mm = np.load(str(tmp_path / "traj.npy"), mmap_mode="r")
    labels = np.array([3, 10, 42], np.uint32)[dense]
    plain = trajectory_interface(md.xyz, md.radii, labels, md.seg_be, md.seg_polar, engine=eng)
    assert plain.pair_labels is None and plain.pair_area is None and plain.seg_pair_area is None
    for src, fpc in ((md.xyz, 1), (md.xyz, 7), (md.xyz, F), (mm, 7)):
        t = trajectory_interface(src, md.radii, labels, md.seg_be, md.seg_polar, frames_per_call=fpc, engine=eng, pairs=True)
        assert np.array_equal(t.pair_labels, [3, 10, 42])
        assert np.array_equal(bits(t.pair_area), bits(ref.pair_area)), fpc
        assert np.array_equal(bits(t.seg_pair_area), bits(ref.seg_pair_area.reshape(F, G, 3))), fpc
        for f in ("complex", "isolated", "buried", "complex_seg", "isolated_seg"):
            assert np.array_equal(bits(getattr(t, f)), bits(getattr(plain, f))), (f, fpc)
    t = trajectory_interface(mm, md.radii, labels, frames_per_call=4, engine=eng, pairs=True)
    assert t.seg_pair_area is None and np.array_equal(bits(t.pair_area), bits(ref.pair_area))
    with pytest.raises(ValueError):
        trajectory_interface(md.xyz, md.radii, np.arange(N, dtype=np.uint32) % 18, engine=eng, pairs=True)
