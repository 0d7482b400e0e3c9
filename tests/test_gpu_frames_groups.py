"""Grouped runs of MD frames (buried surface area along a trajectory): sasa_b200_batch_run_groups_frames_host / _submit_, and
the trajectory_interface front end.

The complex outputs must equal sasa_b200_batch_run_frames_host bit for bit, and the isolated outputs sasa_b200_batch_run_groups_host
on the same coordinates packed as float4 with the labels tiled over the frames.  The isolated values are also checked against the
CPU oracle run on each group's atoms of a frame alone.  Every path a grouped frames run takes is reached: the fused kernel reading
the 12-byte coordinates, frames above the grouped fused kernel's capacity (large-structure path, float4 packing on the device),
and n_points > 128, where every frame takes the large-structure path.
"""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PROBE = 1.4
ALL = ("counts", "atom", "seg", "protein")
FIELDS = ("counts", "atom_sasa", "seg_sasa", "protein")
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
                 'int main() { printf("%u %u\\n", sasa::max_atoms(1024, 1, 16384, false, true), '
                 'sasa::max_atoms(1024, 1, 16384, false, false)); return 0; }\n')
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-I",
                        os.path.join(ROOT, "rustsasa_b200", "csrc"), "-o", exe, src],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    assert r.returncode == 0, r.stdout
    grouped, plain = (int(x) for x in subprocess.run([exe], stdout=subprocess.PIPE, text=True, check=True).stdout.split())
    assert 0 < grouped < plain
    return grouped, plain


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


def plane_groups(xyz):
    """Two groups: the atoms on either side of a plane through the centroid of the base structure (the mean frame)."""
    base = xyz.astype(np.float64).mean(axis=0)
    return (((base - base.mean(axis=0)) @ np.array([0.6, -0.3, 0.74])) > 0.0).astype(np.uint32)


def random_groups(rng, n):
    return rng.integers(0, int(rng.choice([1, 2, 3, 5, 7])), size=n).astype(np.uint32)


def frames_batch(eng, F, N, seg_be=None, polar=None):
    off = (np.arange(F + 1) * N).astype(np.uint64)
    if seg_be is None:
        return eng.batch(off)
    G = len(seg_be)
    return eng.batch(off, np.tile(seg_be, (F, 1)), (np.arange(F + 1) * G).astype(np.uint64),
                     None if polar is None else np.tile(polar, F))


def float4_frames(xyz, radii):
    F, N = xyz.shape[:2]
    return np.concatenate([xyz.reshape(F * N, 3), np.tile(radii, F)[:, None]], axis=1).astype(np.float32)


def same(a, b, fields=FIELDS):
    for f in fields:
        x, y = getattr(a, f), getattr(b, f)
        assert (x is None) == (y is None), f
        if x is not None:
            assert np.array_equal(x, y, equal_nan=f != "counts"), f


def check_against_references(b, xyz, radii, group, n_points=100, lanes=8, want=ALL):
    """run_groups_frames_host against run_frames_host (complex) and run_groups_host on the float4 packing (isolated)."""
    F = xyz.shape[0]
    cpx, iso = b.run_groups_frames_host(xyz, radii, group, PROBE, n_points, lanes, want=want)
    plain = b.run_frames_host(xyz, radii, PROBE, n_points, lanes, want=want)
    ref_cpx, ref_iso = b.run_groups_host(float4_frames(xyz, radii), np.tile(group, F), None, PROBE, n_points, lanes, want=want)
    same(cpx, plain)
    same(cpx, ref_cpx)
    same(iso, ref_iso)
    if "counts" in want:
        assert np.all(iso.counts >= cpx.counts)
    return cpx, iso


@pytest.mark.parametrize("lanes", [4, 8])
@pytest.mark.parametrize("n_points", [100, 960])
@pytest.mark.parametrize("labels", ["plane", "random"])
def test_bit_equal_to_frames_and_grouped_runs(eng, n_points, lanes, labels):
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=6, n_atoms=1200, seed=11)
    F, N = md.xyz.shape[:2]
    group = plane_groups(md.xyz) if labels == "plane" else random_groups(np.random.default_rng(n_points + lanes), N)
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    cpx, iso = check_against_references(b, md.xyz, md.radii, group, n_points, lanes)
    if len(np.unique(group)) > 1:
        assert np.all(iso.protein[:, 0] > cpx.protein[:, 0])   # something is buried in every frame
    if n_points <= 128:
        assert cpx.stats["gpu_launches"] < F   # one fused launch (+ the label expansion) for the whole chunk
    else:
        assert cpx.stats["gpu_launches"] > F   # every frame on the large-structure path
    b.close()


@pytest.mark.parametrize("n_points", [100, 960])
def test_oracle_parity(eng, oracle, n_points):
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=3, n_atoms=900, seed=5)
    F, N = md.xyz.shape[:2]
    for group in (plane_groups(md.xyz), random_groups(np.random.default_rng(n_points), N)):
        b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
        _, iso = b.run_groups_frames_host(md.xyz, md.radii, group, n_points=n_points, want=ALL)
        G = len(md.seg_be)
        for f in range(F):
            xyzr = np.concatenate([md.xyz[f], md.radii[:, None]], axis=1).astype(np.float32)
            counts, sasa = iso_oracle(oracle, xyzr, group, n_points=n_points)
            assert np.array_equal(iso.counts[f * N:(f + 1) * N], counts), f
            assert np.array_equal(iso.atom_sasa[f * N:(f + 1) * N], sasa), f
            assert np.array_equal(iso.seg_sasa[f * G:(f + 1) * G], oracle.segment_sums(sasa, md.seg_be)), f
        b.close()


@pytest.mark.parametrize("n_points", [100, 128])
def test_frames_above_grouped_fused_capacity(eng, oracle, grouped_capacity, n_points):
    """Frames that fit the plain fused kernel but not the grouped one: the grouped run takes the large-structure path, which
    reads float4 atoms that pack_frames_kernel builds on the device, while run_frames_host stays on the fused kernel."""
    from rustsasa_b200 import workloads as W
    cap, plain_cap = grouped_capacity
    md = W.md_trajectory(n_frames=3, n_atoms=cap + 300, seed=21)
    F, N = md.xyz.shape[:2]
    assert cap < N <= plain_cap, (cap, N, plain_cap)
    group = plane_groups(md.xyz)
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    cpx, iso = check_against_references(b, md.xyz, md.radii, group, n_points)
    assert cpx.stats["gpu_launches"] > F
    xyzr = np.concatenate([md.xyz[1], md.radii[:, None]], axis=1).astype(np.float32)
    counts, sasa = iso_oracle(oracle, xyzr, group, n_points=n_points)
    assert np.array_equal(iso.counts[N:2 * N], counts) and np.array_equal(iso.atom_sasa[N:2 * N], sasa)
    # random labels
    check_against_references(b, md.xyz, md.radii, random_groups(np.random.default_rng(3), N), n_points, want=("counts", "protein"))
    b.close()


@pytest.mark.parametrize("n_points", [129, 960])
def test_more_than_128_points_every_frame_on_the_large_path(eng, oracle, n_points):
    """n_points > 128: a grouped run has no fused kernel, so every frame takes the large-structure path even though the frames
    fit the fused kernels; the coordinates must be packed to float4 first."""
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=4, n_atoms=700, seed=9)
    F, N = md.xyz.shape[:2]
    group = plane_groups(md.xyz)
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    cpx, iso = check_against_references(b, md.xyz, md.radii, group, n_points)
    assert cpx.stats["gpu_launches"] > F
    xyzr = np.concatenate([md.xyz[F - 1], md.radii[:, None]], axis=1).astype(np.float32)
    counts, sasa = iso_oracle(oracle, xyzr, group, n_points=n_points)
    assert np.array_equal(iso.counts[(F - 1) * N:], counts) and np.array_equal(iso.atom_sasa[(F - 1) * N:], sasa)
    b.close()


@pytest.mark.parametrize("n_points", [100, 960])
def test_invariants_and_label_values(eng, n_points):
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=4, n_atoms=800, seed=13)
    F, N = md.xyz.shape[:2]
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    plain = b.run_frames_host(md.xyz, md.radii, n_points=n_points, want=ALL)
    cpx, iso = b.run_groups_frames_host(md.xyz, md.radii, np.full(N, 0xFFFFFFFF, np.uint32), n_points=n_points, want=ALL)
    same(cpx, plain)
    same(iso, plain)
    _, iso = b.run_groups_frames_host(md.xyz, md.radii, np.arange(N, dtype=np.uint32), n_points=n_points, want=("counts",))
    assert np.all(iso.counts == n_points)
    dense = np.random.default_rng(17).integers(0, 3, size=N).astype(np.uint32)
    sparse = np.array([0xFFFFFFFF, 0x80000000, 12345], np.uint32)[dense]
    a = b.run_groups_frames_host(md.xyz, md.radii, dense, n_points=n_points, want=ALL)
    s = b.run_groups_frames_host(md.xyz, md.radii, sparse, n_points=n_points, want=ALL)
    for x, y in zip(a, s):
        same(x, y)
    b.close()


@pytest.mark.parametrize("n_points", [100, 960])
def test_non_finite_frame(eng, n_points):
    from rustsasa_b200 import _lib
    from rustsasa_b200.engine import BatchResult
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=5, n_atoms=900, seed=3)
    F, N = md.xyz.shape[:2]
    G = len(md.seg_be)
    group = plane_groups(md.xyz)
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    good = b.run_groups_frames_host(md.xyz, md.radii, group, n_points=n_points, want=ALL)
    bad = md.xyz.copy()
    bad[2, 17, 1] = np.nan
    res = []
    for _ in range(2):
        r = BatchResult(np.full(F * N, 7, np.uint32), np.zeros(F * N, np.float32), np.zeros(F * G, np.float32), np.zeros((F, 3), np.float32))
        res.append(r)
    outs = [_lib.Outputs(r.counts.ctypes.data, r.atom_sasa.ctypes.data, r.seg_sasa.ctypes.data, r.protein.ctypes.data) for r in res]
    prm = _lib.Params(PROBE, n_points, 8, -1, 0)
    rc = b._L.sasa_b200_batch_run_groups_frames_host(b._h, bad.ctypes.data, md.radii.ctypes.data, group.ctypes.data, C.byref(prm),
                                                     C.byref(outs[0]), C.byref(outs[1]), None)
    assert rc == _lib.ERR_NON_FINITE
    for r, g in zip(res, good):
        for f in range(F):
            a, s = slice(f * N, (f + 1) * N), slice(f * G, (f + 1) * G)
            if f == 2:
                assert not np.any(r.counts[a]) and np.all(np.isnan(r.atom_sasa[a]))
                assert np.all(np.isnan(r.seg_sasa[s])) and np.all(np.isnan(r.protein[f]))
            else:
                assert np.array_equal(r.counts[a], g.counts[a]) and np.array_equal(r.atom_sasa[a], g.atom_sasa[a]), f
                assert np.array_equal(r.seg_sasa[s], g.seg_sasa[s]) and np.array_equal(r.protein[f], g.protein[f]), f
    # the context stays usable
    again = b.run_groups_frames_host(md.xyz, md.radii, group, n_points=n_points, want=ALL)
    same(again[1], good[1])
    b.close()


def test_errors_and_empty_batch(eng):
    from rustsasa_b200 import _lib
    from rustsasa_b200.engine import SasaB200Error
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=2, n_atoms=300, seed=1)
    F, N = md.xyz.shape[:2]
    group = plane_groups(md.xyz)
    b = frames_batch(eng, F, N)
    L, h = b._L, b._h
    x, r, g = md.xyz.ctypes.data, md.radii.ctypes.data, group.ctypes.data
    outs = _lib.Outputs(None, None, None, None)
    prm = _lib.Params(PROBE, 100, 8, -1, 0)
    for args in ((None, r, g), (x, None, g), (x, r, None)):
        assert L.sasa_b200_batch_run_groups_frames_host(h, *args, C.byref(prm), C.byref(outs), C.byref(outs), None) \
            == _lib.ERR_INVALID_ARGUMENT, args
        job = C.c_void_p()
        assert L.sasa_b200_batch_submit_groups_frames_host(h, *args, C.byref(prm), C.byref(outs), C.byref(outs), C.byref(job)) \
            == _lib.ERR_INVALID_ARGUMENT, args
    assert L.sasa_b200_batch_run_groups_frames_host(h, x, r, g, C.byref(prm), C.byref(outs), None, None) == _lib.ERR_INVALID_ARGUMENT
    for flags in (_lib.FLAG_BOUNDARY_STATS, _lib.FLAG_FORCE_STREAMING):
        with pytest.raises(SasaB200Error) as e:
            b.run_groups_frames_host(md.xyz, md.radii, group, flags=flags)
        assert e.value.code == _lib.ERR_UNSUPPORTED
    b.close()
    # frames of unequal size
    u = eng.batch(np.array([0, N, 2 * N - 1], np.uint64))
    assert L.sasa_b200_batch_run_groups_frames_host(u._h, x, r, g, C.byref(prm), C.byref(outs), C.byref(outs), None) \
        == _lib.ERR_INVALID_ARGUMENT
    u.close()
    # a batch of no frames
    e0 = eng.batch([0])
    cpx, iso = e0.run_groups_frames_host(np.zeros((0, 0, 3), np.float32), np.zeros(0, np.float32), np.zeros(0, np.uint32), want=ALL)
    assert cpx.protein.shape == (0, 3) and iso.counts.shape == (0,)
    assert L.sasa_b200_batch_run_groups_frames_host(e0._h, None, None, None, C.byref(prm), C.byref(outs), C.byref(outs), None) == _lib.OK
    e0.close()


def test_submit_wait(eng):
    from rustsasa_b200 import _lib
    from rustsasa_b200.engine import SasaB200Error
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=8, n_atoms=1000, seed=4)
    F, N = md.xyz.shape[:2]
    group = plane_groups(md.xyz)
    b1 = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    b2 = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    ref = b1.run_groups_frames_host(md.xyz, md.radii, group, want=ALL)
    x1 = eng.pinned_empty(md.xyz.shape, np.float32)
    x1[:] = md.xyz
    x2 = eng.pinned_empty(md.xyz.shape, np.float32)
    x2[:] = md.xyz[::-1]
    j1 = b1.submit_groups_frames_host(x1, md.radii, group, want=ALL)
    j2 = b2.submit_groups_frames_host(x2, md.radii, group, want=ALL)   # two batches in flight at once
    with pytest.raises(SasaB200Error) as e:
        b1.submit_groups_frames_host(x1, md.radii, group, want=ALL)   # b1 already carries a run
    assert e.value.code == _lib.ERR_INVALID_ARGUMENT
    r1, r2 = j1.wait(), j2.wait()
    for r, rf in zip(r1, ref):
        same(r, rf)
    G = len(md.seg_be)
    for r, rf in zip(r2, ref):   # b2 ran the frames in reverse order
        assert np.array_equal(r.protein, rf.protein[::-1])
        assert np.array_equal(r.seg_sasa.reshape(F, G), rf.seg_sasa.reshape(F, G)[::-1])
        assert np.array_equal(r.counts.reshape(F, N), rf.counts.reshape(F, N)[::-1])
    # the batch takes a new run once the job is done
    same(b1.submit_groups_frames_host(x1, md.radii, group, want=ALL).wait()[1], ref[1])
    b1.close()
    b2.close()


def test_trajectory_interface(eng, tmp_path):
    from rustsasa_b200 import TrajectoryInterfaceResult, trajectory_interface
    from rustsasa_b200 import workloads as W
    md = W.md_trajectory(n_frames=30, n_atoms=1100, seed=8)
    F, N = md.xyz.shape[:2]
    G = len(md.seg_be)
    group = plane_groups(md.xyz)
    b = frames_batch(eng, F, N, md.seg_be, md.seg_polar)
    cpx, iso = b.run_groups_frames_host(md.xyz, md.radii, group, want=("protein", "seg"))
    b.close()
    mm = np.lib.format.open_memmap(str(tmp_path / "traj.npy"), mode="w+", dtype=np.float32, shape=md.xyz.shape)
    mm[:] = md.xyz
    mm.flush()
    mm = np.load(str(tmp_path / "traj.npy"), mmap_mode="r")
    for src, fpc in ((md.xyz, 1), (md.xyz, 7), (md.xyz, F), (md.xyz, None), (mm, 7)):
        t = trajectory_interface(src, md.radii, group, md.seg_be, md.seg_polar, frames_per_call=fpc, engine=eng)
        assert isinstance(t, TrajectoryInterfaceResult)
        assert np.array_equal(t.complex, cpx.protein) and np.array_equal(t.isolated, iso.protein), fpc
        assert np.array_equal(t.complex_seg, cpx.seg_sasa.reshape(F, G)), fpc
        assert np.array_equal(t.isolated_seg, iso.seg_sasa.reshape(F, G)), fpc
        assert np.array_equal(t.buried, iso.protein[:, 0] - cpx.protein[:, 0])
        assert np.all(t.buried > 0)
    t = trajectory_interface(mm, md.radii, group, frames_per_call=4, engine=eng)
    assert t.complex_seg is None and t.isolated_seg is None
    assert np.array_equal(t.complex[:, 0], cpx.protein[:, 0]) and np.array_equal(t.isolated[:, 0], iso.protein[:, 0])
