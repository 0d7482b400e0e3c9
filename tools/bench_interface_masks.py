#!/usr/bin/env python
"""Cost of interface patches (grouped runs with exposed-point masks), device-resident, CUDA events.

On the seeded cfg2 proteome batch, every structure cut into two groups by a random plane through its centroid (the groups of
tools/bench_interface.py), timed alternating in one process at 100 points:
  (a) the grouped run                                       (Batch.run_groups_device)
  (b) the grouped masked run: both mask sets in one pass     (Batch.run_groups_masks_device)
  (c) the two-run masked baseline: a masked run of the complex, plus a masked run of the batch rebuilt with every group as
      a structure of its own                                 (Batch.run_masks_device twice)
(b)'s masks are checked against (c)'s bit for bit after scattering back.  Then, on cfg4 (150 k atoms) cut in two by a plane
through its centroid at 960 points, where grouped runs take the large-structure path and a masked grouped run streams every
atom twice: the grouped run, the grouped masked run and the plain masked run.  Prints one JSON line.
usage: python tools/bench_interface_masks.py [--structures 4400] [--reps 10] [--reps960 3] [--out path]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_interface import card, plane_groups, split_order  # noqa: E402


def timed(runs, reps):
    """Median and range in ms of every run, alternating, after one warm-up call each."""
    import torch
    for f in runs.values():
        f()
    torch.cuda.synchronize()
    times = {k: [] for k in runs}
    for _ in range(reps):
        for k, f in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
    return {k: float(np.median(v)) for k, v in times.items()}, {k: [float(min(v)), float(max(v))] for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--structures", type=int, default=4400)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--reps960", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from rustsasa_b200 import Engine, workloads as W
    probe, n_points = 1.4, 100
    Wd = (n_points + 31) // 32
    d = W.proteome_batch(args.structures, seed=W.SEED)
    S, N = len(d.struct_off) - 1, d.n_atoms
    group = plane_groups(d.struct_off, d.xyzr, W.SEED + 17)
    perm, split_off = split_order(d.struct_off, group)

    eng = Engine(0)
    b = eng.batch(d.struct_off, d.seg_be, d.struct_seg_off, d.seg_polar)
    bs = eng.batch(split_off)
    dev = torch.device("cuda", 0)
    d_x = torch.from_numpy(d.xyzr).to(dev)
    d_g = torch.from_numpy(group.view(np.int32)).to(dev)
    d_xs = torch.from_numpy(np.ascontiguousarray(d.xyzr[perm])).to(dev)
    z = lambda shape, dt=torch.float32: torch.zeros(shape, dtype=dt, device=dev)   # noqa: E731
    m_cpx, m_iso = z((N, Wd), torch.int32), z((N, Wd), torch.int32)      # (b)
    c_cpx, c_split = z((N, Wd), torch.int32), z((N, Wd), torch.int32)    # (c)
    pc, pa, ps, pp = z(N, torch.int32), z(N), z(len(d.seg_be)), z((S, 3))
    sc, sa, sp = z(N, torch.int32), z(N), z((2 * S, 3))
    run_a = lambda: b.run_groups_device(d_x, d_g, probe_radius=probe, n_points=n_points)   # noqa: E731
    run_b = lambda: b.run_groups_masks_device(d_x, d_g, m_cpx, m_iso, probe_radius=probe, n_points=n_points)   # noqa: E731

    def run_c():
        b.run_masks_device(d_x, c_cpx, probe_radius=probe, n_points=n_points, counts=pc, atom_sasa=pa, seg_sasa=ps, protein=pp)
        bs.run_masks_device(d_xs, c_split, probe_radius=probe, n_points=n_points, counts=sc, atom_sasa=sa, protein=sp)

    med, spread = timed({"a_grouped": run_a, "b_grouped_masks": run_b, "c_two_run_masks": run_c}, args.reps)
    b.sync()
    bs.sync()
    # correctness on the timed inputs: (b) against (c), bit for bit after scattering (c)'s rebuilt batch back
    cpx, iso = run_b()
    run_c()
    torch.cuda.synchronize()
    b.sync()
    bs.sync()
    split = np.empty((N, Wd), np.uint32)
    split[perm] = c_split.cpu().numpy().view(np.uint32)
    masks_equal = bool(torch.equal(m_cpx, c_cpx)) and bool(np.array_equal(m_iso.cpu().numpy().view(np.uint32), split))
    counts_equal = bool(torch.equal(cpx.counts, pc))
    bs.close()
    b.close()

    # 960 points on cfg4 cut in two: the large-structure path, streaming both evaluations of every atom
    g4 = W.large_assembly(150000)
    x4 = g4.xyzr[:, :3].astype(np.float64)
    grp4 = ((x4 - x4.mean(axis=0)) @ np.array([0.6, -0.3, 0.74]) > 0.0).astype(np.uint32)
    b4 = eng.batch(g4.struct_off)
    N4, W4 = g4.n_atoms, (960 + 31) // 32
    d_x4 = torch.from_numpy(g4.xyzr).to(dev)
    d_g4 = torch.from_numpy(grp4.view(np.int32)).to(dev)
    e_cpx, e_iso, e_plain = z((N4, W4), torch.int32), z((N4, W4), torch.int32), z((N4, W4), torch.int32)
    med960, spread960 = timed({
        "grouped": lambda: b4.run_groups_device(d_x4, d_g4, n_points=960),
        "grouped_masks": lambda: b4.run_groups_masks_device(d_x4, d_g4, e_cpx, e_iso, n_points=960),
        "masks": lambda: b4.run_masks_device(d_x4, e_plain, n_points=960),
    }, args.reps960)
    b4.sync()
    b4.run_groups_masks_device(d_x4, d_g4, e_cpx, e_iso, n_points=960)
    torch.cuda.synchronize()
    st = b4.sync()   # statistics of this one run
    masks960_equal = bool(torch.equal(e_cpx, e_plain))
    b4.close()

    name, power = card()
    out = dict(workload=d.name + ", two groups per structure (random plane through the centroid)", atoms=N, structures=S,
               n_points=n_points, reps=args.reps, median_ms=med, spread_ms=spread,
               ratio_b_over_a=med["b_grouped_masks"] / med["a_grouped"], ratio_b_over_c=med["b_grouped_masks"] / med["c_two_run_masks"],
               masks_equal_two_run=masks_equal, complex_counts_equal=counts_equal,
               cfg4_960=dict(atoms=N4, reps=args.reps960, median_ms=med960, spread_ms=spread960,
                             ratio_grouped_masks_over_grouped=med960["grouped_masks"] / med960["grouped"],
                             streamed_atoms=st["streamed_atoms"], complex_masks_equal_masked_run=masks960_equal),
               gpu=name, power_limit=power)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    eng.close()
    if not (masks_equal and counts_equal and masks960_equal):
        sys.exit(1)


if __name__ == "__main__":
    main()
