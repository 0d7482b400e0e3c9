#!/usr/bin/env python
"""Pairwise buried area along an MD trajectory: per-frame group-pair and residue-partner areas summed on the device, end to end
from page-locked host memory.

Routes, timed alternating in one process (ProteinLevel outputs, 100 points):
  (a) the grouped frames run: complex and isolated totals only                 (Batch.run_groups_frames_host)
  (b) the pairwise frames run: (a) plus the per-frame L x L pair areas and the per-residue partner areas, summed on the device
                                                                                (Batch.run_group_pairs_frames_host)
  (c) today's route: the pairs run on float4 frames with the labels tiled over the frames (Batch.run_group_pairs_host, K =
      max(1, L - 1) slots per atom copied back), then group_pair_table and per-residue float64 atom-order sums (np.add.at) on
      the host.  The float4 packing and the tiled labels are built before the timing and not counted.
Trajectories: the seeded 3,500-atom trajectory (frames that fit the grouped fused kernel) cut in two by a plane through the
centroid of the mean frame and in four sectors about its centroid, and cfg3 (5,000 atoms, --cfg3-frames frames) cut in two.
End to end is a host clock around the call (it returns with the outputs in host memory); the device span is the library's
CUDA-event span of the pipelined run (sasa_b200_stats.kernel_ms).  Bytes on the wire are counted from the shapes.  (b)'s sums are
checked against (c)'s bit for bit, and (b)'s complex / isolated totals against (a)'s.
With --profile, the reduction kernels are timed in a separate torch.profiler run (CUDA activities) of one (b) call on each
trajectory, against the total kernel time of that call.  Prints one JSON line; exits 1 when a check fails.
usage: python tools/bench_frames_group_pairs.py [--frames 10000] [--atoms 3500] [--cfg3-frames 2000] [--reps 5] [--profile]
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

from bench_frames_groups import plane_groups, timed  # noqa: E402
from bench_interface import card  # noqa: E402


def sector_groups(xyz, n):
    base = xyz[: min(64, xyz.shape[0])].astype(np.float64).mean(axis=0)
    c = base - base.mean(axis=0)
    ang = np.arctan2(c[:, 1], c[:, 0]) + np.pi
    return np.minimum((ang / (2 * np.pi) * n).astype(np.uint32), n - 1)


def host_reduction(partner, area, tiled, F, N, L, seg_of_atom, G):
    """(c)'s host side: group_pair_table in dense form, and per residue the float64 sums of the slot areas in atom order."""
    from rustsasa_b200 import group_pair_table
    dense = np.zeros((F, L, L), np.float64)
    for s, rows in enumerate(group_pair_table(partner, area, tiled, np.arange(F + 1, dtype=np.int64) * N)):
        for g, h, gh, hg in rows:
            dense[s, g, h], dense[s, h, g] = gh, hg
    seg = np.zeros((F * G, L), np.float64)
    atom, slot = np.nonzero(partner < L)   # atom-major: np.add.at adds in atom order
    frame = atom // N
    np.add.at(seg, (frame * G + seg_of_atom[atom % N], partner[atom, slot].astype(np.int64)), area[atom, slot].astype(np.float64))
    return dense, seg


def measure(eng, name, md, group, reps, profile):
    from rustsasa_b200 import BatchResult, PairSums
    F, N = md.xyz.shape[:2]
    G = len(md.seg_be)
    L = int(group.max()) + 1
    K = max(1, L - 1)
    seg_of_atom = np.zeros(N, np.int64)
    for q, (b0, b1) in enumerate(md.seg_be):
        seg_of_atom[b0:b1] = q
    b = eng.batch(np.arange(F + 1, dtype=np.uint64) * N, np.tile(md.seg_be, (F, 1)), np.arange(F + 1, dtype=np.uint64) * G,
                  np.tile(md.seg_polar, F))
    h_xyz = eng.pinned_empty((F, N, 3), np.float32)
    h_xyz[...] = md.xyz
    h_xyzr = eng.pinned_empty((F * N, 4), np.float32)   # (c)'s input, packed before the timing
    h_xyzr[:, :3] = md.xyz.reshape(F * N, 3)
    h_xyzr[:, 3] = np.tile(md.radii, F)
    tiled = np.tile(group, F)
    pin = lambda shape, dt: eng.pinned_empty(shape, dt)   # noqa: E731
    res_a = (BatchResult(protein=pin((F, 3), np.float32)), BatchResult(protein=pin((F, 3), np.float32)))
    res_b = (BatchResult(protein=pin((F, 3), np.float32)), BatchResult(protein=pin((F, 3), np.float32)),
             PairSums(L, pin((F, L, L), np.float64), pin((F * G, L), np.float64)))
    out_c = {}
    stats = {}

    def run_a():
        cpx, _ = b.run_groups_frames_host(h_xyz, md.radii, group, want=("protein",), result=res_a)
        return cpx.stats["kernel_ms"]

    def run_b():
        cpx, _, _ = b.run_group_pairs_frames_host(h_xyz, md.radii, group, L, want=("protein",), result=res_b)
        stats["b"] = cpx.stats
        return cpx.stats["kernel_ms"]

    def run_c():
        cpx, _, pairs = b.run_group_pairs_host(h_xyzr, tiled, want=("protein",), max_partners=K)
        out_c["sums"] = host_reduction(pairs.partner, pairs.buried_area, tiled, F, N, L, seg_of_atom, G)
        stats["c"] = cpx.stats
        return cpx.stats["kernel_ms"]

    times = timed({"a_groups_frames": run_a, "b_group_pairs_frames": run_b, "c_pairs_run_host_reduction": run_c}, reps)
    dense, seg = out_c["sums"]
    sums_equal = bool(np.array_equal(np.asarray(res_b[2].pair_area).view(np.uint64), dense.view(np.uint64))
                      and np.array_equal(np.asarray(res_b[2].seg_pair_area).view(np.uint64), seg.view(np.uint64)))
    totals_equal = bool(np.array_equal(np.asarray(res_b[0].protein), np.asarray(res_a[0].protein))
                        and np.array_equal(np.asarray(res_b[1].protein), np.asarray(res_a[1].protein)))
    atoms = F * N
    wire = {
        "a_groups_frames": dict(h2d=atoms * 12 + N * 8, d2h=2 * F * 12),
        "b_group_pairs_frames": dict(h2d=atoms * 12 + N * 8, d2h=2 * F * 12 + F * L * L * 8 + F * G * L * 8),
        "c_pairs_run_host_reduction": dict(h2d=atoms * 20, d2h=2 * F * 12 + atoms * K * 8),
    }
    out = dict(workload=f"{md.name}, {name}, ProteinLevel, 100 points", frames=F, atoms_per_frame=N, segments_per_frame=G,
               n_labels=L, slots_per_atom=K, reps=reps, **times,
               ratio_b_over_a_e2e=times["e2e_ms"]["b_group_pairs_frames"] / times["e2e_ms"]["a_groups_frames"],
               ratio_b_over_c_e2e=times["e2e_ms"]["b_group_pairs_frames"] / times["e2e_ms"]["c_pairs_run_host_reduction"],
               gpu_launches_b=stats["b"]["gpu_launches"], gpu_launches_c=stats["c"]["gpu_launches"], wire_bytes=wire,
               sums_equal_host_route=sums_equal, totals_equal_grouped_frames_run=totals_equal,
               pair_area_frame_mean=np.asarray(res_b[2].pair_area).mean(axis=0).tolist())
    if profile:
        out["profile"] = profile_sums(b, h_xyz, md.radii, group, L, res_b)
    b.close()
    return out


def profile_sums(b, h_xyz, radii, group, L, res_b):
    """Device time of the reduction kernels against every kernel of one (b) call, from torch.profiler (CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    b.run_group_pairs_frames_host(h_xyz, radii, group, L, want=("protein",), result=res_b)   # warm-up
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        b.run_group_pairs_frames_host(h_xyz, radii, group, L, want=("protein",), result=res_b)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.key_averages():
        t = getattr(ev, "self_device_time_total", None)
        if t is None:
            t = getattr(ev, "self_cuda_time_total", 0.0)
        if t and "memcpy" not in ev.key.lower() and "memset" not in ev.key.lower():
            per[ev.key] = dict(us=float(t), calls=int(ev.count))
    total = sum(v["us"] for v in per.values())
    red = {k: v for k, v in per.items() if "pair_sums_kernel" in k}
    red_us = sum(v["us"] for v in red.values())
    return dict(kernels_us_total=total, reduction_kernels=red, reduction_us=red_us,
                reduction_share_of_kernel_time=red_us / total if total else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=10000)
    ap.add_argument("--atoms", type=int, default=3500)
    ap.add_argument("--cfg3-frames", type=int, default=2000, help="frames of the cfg3 trajectory (0: skip)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from rustsasa_b200 import Engine, workloads as W
    eng = Engine(0)
    name, power = card()
    out = dict(gpu=name, power_limit=power)
    md = W.md_trajectory(n_frames=args.frames, n_atoms=args.atoms)
    out["fits_grouped_fused_2"] = measure(eng, "two groups per frame (plane through the centroid)", md, plane_groups(md.xyz),
                                          args.reps, args.profile)
    out["fits_grouped_fused_4"] = measure(eng, "four sectors about the centroid", md, sector_groups(md.xyz, 4), args.reps,
                                          args.profile)
    del md
    if args.cfg3_frames:
        md = W.md_trajectory(n_frames=args.cfg3_frames, n_atoms=5000)
        out["cfg3_2"] = measure(eng, "two groups per frame (plane through the centroid)", md, plane_groups(md.xyz), args.reps,
                                args.profile)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    eng.close()
    ok = all(r["sums_equal_host_route"] and r["totals_equal_grouped_frames_run"] for r in out.values() if isinstance(r, dict))
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
