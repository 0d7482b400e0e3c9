#!/usr/bin/env python
"""Buried surface area along an MD trajectory: grouped runs through the frames form, end to end from page-locked host memory.

On the seeded cfg3 trajectory (10,000 frames x 5,000 atoms, ProteinLevel, 100 points), every frame cut in two by a plane through
the centroid of the mean frame, timed alternating in one process:
  (a) the plain frames run                                   (Batch.run_frames_host)
  (b) the grouped frames run: complex and isolated in one pass (Batch.run_groups_frames_host)
  (c) the route without it: run_frames_host on the complex plus one run_frames_host per group's sub-trajectory
End to end is a host clock around the call (it returns with the outputs in host memory); the device span is the library's
CUDA-event span of the pipelined run (sasa_b200_stats.kernel_ms), summed over the calls of (c).  Bytes on the wire are counted
from the shapes.  (b)'s complex is checked against (a) and (b)'s isolated per-atom areas against (c) scattered back, bit for bit
(from one atom-level run each).  Then one trajectory_interface pass with --frames-per-call frames per call, checked against (b).
With --atoms2 the same is repeated on a trajectory of that frame size (default 3,500 atoms: frames that fit the grouped fused
kernel).  Prints one JSON line.
usage: python tools/bench_frames_groups.py [--frames 10000] [--atoms 5000] [--atoms2 3500] [--reps 8] [--frames-per-call 1000]
                                           [--out path]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_interface import card  # noqa: E402


def plane_groups(xyz):
    base = xyz[: min(64, xyz.shape[0])].astype(np.float64).mean(axis=0)
    return (((base - base.mean(axis=0)) @ np.array([0.6, -0.3, 0.74])) > 0.0).astype(np.uint32)


def timed(runs, reps):
    """Median / range of the host-clock end-to-end time and of the device span (ms) of every run, alternating, after one
    warm-up call each.  A run returns its device span in ms."""
    for f in runs.values():
        f()
    e2e = {k: [] for k in runs}
    dev = {k: [] for k in runs}
    for _ in range(reps):
        for k, f in runs.items():
            t0 = time.perf_counter()
            span = f()
            e2e[k].append((time.perf_counter() - t0) * 1e3)
            dev[k].append(span)
    med = lambda d: {k: float(np.median(v)) for k, v in d.items()}   # noqa: E731
    rng = lambda d: {k: [float(min(v)), float(max(v))] for k, v in d.items()}   # noqa: E731
    return dict(e2e_ms=med(e2e), e2e_range_ms=rng(e2e), device_ms=med(dev), device_range_ms=rng(dev))


def measure(eng, F, n_atoms, reps, fpc):
    from rustsasa_b200 import BatchResult, trajectory_interface, workloads as W
    md = W.md_trajectory(n_frames=F, n_atoms=n_atoms)
    N = md.xyz.shape[1]
    G = len(md.seg_be)
    group = plane_groups(md.xyz)
    masks = [np.nonzero(group == g)[0] for g in np.unique(group)]

    def frames_batch(n, seg=True):
        off = np.arange(F + 1, dtype=np.uint64) * n
        if not seg:
            return eng.batch(off)
        return eng.batch(off, np.tile(md.seg_be, (F, 1)), np.arange(F + 1, dtype=np.uint64) * G, np.tile(md.seg_polar, F))

    b = frames_batch(N)
    h_xyz = eng.pinned_empty((F, N, 3), np.float32)
    h_xyz[...] = md.xyz
    subs = []
    for m in masks:   # the sub-trajectories of route (c), extracted before the timing (their extraction is not counted)
        x = eng.pinned_empty((F, m.size, 3), np.float32)
        x[...] = md.xyz[:, m, :]
        subs.append((frames_batch(m.size, seg=False), x, np.ascontiguousarray(md.radii[m]), BatchResult(protein=eng.pinned_empty((F, 3), np.float32))))
    res_a = BatchResult(protein=eng.pinned_empty((F, 3), np.float32))
    res_b = (BatchResult(protein=eng.pinned_empty((F, 3), np.float32)), BatchResult(protein=eng.pinned_empty((F, 3), np.float32)))
    res_c = BatchResult(protein=eng.pinned_empty((F, 3), np.float32))
    stats_b = {}

    def run_a():
        return b.run_frames_host(h_xyz, md.radii, want=("protein",), result=res_a).stats["kernel_ms"]

    def run_b():
        cpx, _ = b.run_groups_frames_host(h_xyz, md.radii, group, want=("protein",), result=res_b)
        stats_b.update(cpx.stats)
        return cpx.stats["kernel_ms"]

    def run_c():
        t = b.run_frames_host(h_xyz, md.radii, want=("protein",), result=res_c).stats["kernel_ms"]
        for bs, x, r, out in subs:
            t += bs.run_frames_host(x, r, want=("protein",), result=out).stats["kernel_ms"]
        return t

    times = timed({"a_frames": run_a, "b_groups_frames": run_b, "c_frames_per_group": run_c}, reps)
    launches_b = stats_b["gpu_launches"]

    # correctness, from one atom-level run each
    cpx, iso = b.run_groups_frames_host(h_xyz, md.radii, group, want=("atom", "protein"))
    plain = b.run_frames_host(h_xyz, md.radii, want=("atom", "protein"))
    split = np.empty((F, N), np.float32)
    for (bs, x, r, _), m in zip(subs, masks):
        split[:, m] = bs.run_frames_host(x, r, want=("atom",)).atom_sasa.reshape(F, m.size)
    complex_equal = bool(np.array_equal(cpx.atom_sasa, plain.atom_sasa) and np.array_equal(cpx.protein, plain.protein)
                         and np.array_equal(np.asarray(res_b[0].protein), np.asarray(res_a.protein)))
    isolated_equal = bool(np.array_equal(iso.atom_sasa.reshape(F, N), split))

    # the front end: pageable input staged block by block
    t0 = time.perf_counter()
    t = trajectory_interface(md.xyz, md.radii, group, md.seg_be, md.seg_polar, frames_per_call=fpc, engine=eng)
    front_ms = (time.perf_counter() - t0) * 1e3
    front_equal = bool(np.array_equal(t.complex, cpx.protein) and np.array_equal(t.isolated, iso.protein))
    buried = t.buried

    for bs, *_ in subs:
        bs.close()
    b.close()
    atoms = F * N
    wire = {
        "a_frames": dict(h2d=atoms * 12 + N * 4, d2h=F * 12),
        "b_groups_frames": dict(h2d=atoms * 12 + N * 8, d2h=2 * F * 12),
        "c_frames_per_group": dict(h2d=2 * atoms * 12 + 2 * N * 4, d2h=(1 + len(masks)) * F * 12),
        "float4_tiled_groups": dict(h2d=atoms * 20, d2h=2 * F * 12),
    }
    return dict(workload=f"{md.name}, two groups per frame (plane through the centroid), ProteinLevel, 100 points",
                frames=F, atoms_per_frame=N, group_sizes=[int(m.size) for m in masks], reps=reps, **times,
                atoms_per_s_e2e={k: atoms / (v * 1e-3) for k, v in times["e2e_ms"].items()},
                ratio_b_over_c_e2e=times["e2e_ms"]["b_groups_frames"] / times["e2e_ms"]["c_frames_per_group"],
                ratio_b_over_a_e2e=times["e2e_ms"]["b_groups_frames"] / times["e2e_ms"]["a_frames"],
                gpu_launches_b=launches_b, wire_bytes=wire,
                complex_equal_frames_run=complex_equal, isolated_equal_per_group_runs=isolated_equal,
                trajectory_interface=dict(frames_per_call=fpc, e2e_ms=front_ms, equal_direct_run=front_equal,
                                          buried_mean=float(np.mean(buried)), buried_min=float(np.min(buried))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=10000)
    ap.add_argument("--atoms", type=int, default=5000)
    ap.add_argument("--atoms2", type=int, default=3500, help="second frame size (0: skip)")
    ap.add_argument("--reps", type=int, default=8)
    ap.add_argument("--frames-per-call", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from rustsasa_b200 import Engine
    eng = Engine(0)
    out = dict(cfg3=measure(eng, args.frames, args.atoms, args.reps, args.frames_per_call))
    if args.atoms2:
        out["fits_grouped_fused"] = measure(eng, args.frames, args.atoms2, args.reps, args.frames_per_call)
    name, power = card()
    out.update(gpu=name, power_limit=power)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    eng.close()
    ok = all(r["complex_equal_frames_run"] and r["isolated_equal_per_group_runs"] and r["trajectory_interface"]["equal_direct_run"]
             for k, r in out.items() if isinstance(r, dict))
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
