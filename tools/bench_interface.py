#!/usr/bin/env python
"""Cost of a grouped run (buried surface area) on the seeded cfg2 proteome batch, device-resident, CUDA events.

Every structure is cut into two groups by a random plane through its centroid.  Timed, alternating, in one process:
  (a) the plain run                                          (Batch.run_device)
  (b) the grouped run: complex + isolated in one pass        (Batch.run_groups_device)
  (c) the two-run baseline: the plain run, plus the batch rebuilt with every group as a structure of its own
All runs produce counts, per-atom areas and protein totals; (a) and (b) also residue sums ((c)'s rebuilt batch has no
residues: they straddle the plane).  (b)'s isolated counts are checked against (c)'s count for count.  Prints one JSON line.
usage: python tools/bench_interface.py [--structures 4400] [--reps 10] [--out path]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return name, pl


def other_group_fraction(d, group, probe, n_sample):
    """Fraction of atoms with a neighbour (r_i + r_j + 2 probe) of the other group, over the first n_sample structures."""
    from scipy.spatial import cKDTree
    hit = tot = 0
    for s in range(min(n_sample, len(d.struct_off) - 1)):
        a0, a1 = int(d.struct_off[s]), int(d.struct_off[s + 1])
        x, g = d.xyzr[a0:a1], group[a0:a1]
        pairs = cKDTree(x[:, :3]).query_pairs(2.0 * float(x[:, 3].max()) + 2.0 * probe, output_type="ndarray")
        i, j = pairs[:, 0], pairs[:, 1]
        dist = np.linalg.norm(x[i, :3] - x[j, :3], axis=1)
        m = (dist <= x[i, 3] + x[j, 3] + 2.0 * probe) & (g[i] != g[j])
        flag = np.zeros(a1 - a0, bool)
        flag[i[m]] = True
        flag[j[m]] = True
        hit += int(flag.sum())
        tot += a1 - a0
    return hit / max(tot, 1)


def plane_groups(struct_off, xyzr, seed):
    """Two groups per structure: the sides of a random plane through its centroid."""
    rng = np.random.default_rng(seed)
    group = np.empty(xyzr.shape[0], np.uint32)
    for s in range(len(struct_off) - 1):
        a0, a1 = int(struct_off[s]), int(struct_off[s + 1])
        x = xyzr[a0:a1, :3].astype(np.float64)
        nrm = rng.normal(size=3)
        group[a0:a1] = ((x - x.mean(axis=0)) @ nrm > 0.0).astype(np.uint32)
    return group


def split_order(struct_off, group):
    """The two-run baseline's rebuilt batch: per structure the atoms of group 0, then those of group 1, each a structure of its
    own.  Returns (perm, split_off): rebuilt atom k is original atom perm[k]."""
    perm, split_off = [], [0]
    for s in range(len(struct_off) - 1):
        a0, a1 = int(struct_off[s]), int(struct_off[s + 1])
        for g in (0, 1):
            idx = a0 + np.nonzero(group[a0:a1] == g)[0]
            perm.append(idx)
            split_off.append(split_off[-1] + idx.size)
    return np.concatenate(perm), np.asarray(split_off, np.uint64)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--structures", type=int, default=4400)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--sample", type=int, default=200, help="structures used for the other-group-neighbour fraction")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from rustsasa_b200 import Engine, workloads as W
    probe, n_points = 1.4, 100
    d = W.proteome_batch(args.structures, seed=W.SEED)
    S, N = len(d.struct_off) - 1, d.n_atoms
    group = plane_groups(d.struct_off, d.xyzr, W.SEED + 17)
    perm, split_off = split_order(d.struct_off, group)   # (c)'s rebuilt batch

    eng = Engine(0)
    b = eng.batch(d.struct_off, d.seg_be, d.struct_seg_off, d.seg_polar)
    bs = eng.batch(split_off)
    dev = torch.device("cuda", 0)
    d_x = torch.from_numpy(d.xyzr).to(dev)
    d_g = torch.from_numpy(group.view(np.int32)).to(dev)
    d_xs = torch.from_numpy(np.ascontiguousarray(d.xyzr[perm])).to(dev)
    z = lambda n, dt=torch.float32: torch.zeros(n, dtype=dt, device=dev)   # noqa: E731
    pc, pa, ps, pp = z(N, torch.int32), z(N), z(len(d.seg_be)), z((S, 3))
    sc, sa, sp = z(N, torch.int32), z(N), z((2 * S, 3))
    run_a = lambda: b.run_device(d_x, probe_radius=probe, n_points=n_points, counts=pc, atom_sasa=pa, seg_sasa=ps, protein=pp)   # noqa: E731
    run_b = lambda: b.run_groups_device(d_x, d_g, probe_radius=probe, n_points=n_points)   # noqa: E731

    def run_c():
        run_a()
        bs.run_device(d_xs, probe_radius=probe, n_points=n_points, counts=sc, atom_sasa=sa, protein=sp)

    runs = {"a_plain": run_a, "b_grouped": run_b, "c_two_run": run_c}
    for f in runs.values():   # warm-up: modules, tables, workspaces
        f()
    torch.cuda.synchronize()
    b.sync()
    bs.sync()
    times = {k: [] for k in runs}
    for _ in range(args.reps):
        for k, f in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
    b.sync()
    bs.sync()
    # correctness on the timed inputs: (b) against (c), count for count
    cpx, iso = run_b()
    run_c()
    torch.cuda.synchronize()
    b.sync()
    bs.sync()
    iso_counts = iso.counts.cpu().numpy()
    split_counts = np.empty(N, np.int32)
    split_counts[perm] = sc.cpu().numpy()
    counts_equal = bool(np.array_equal(iso_counts, split_counts)) and bool(torch.equal(cpx.counts, pc))
    # one grouped run through the host entry point
    t0 = time.perf_counter()
    b.run_groups_host(d.xyzr, group, probe_radius=probe, n_points=n_points)
    host_ms = (time.perf_counter() - t0) * 1e3
    med = {k: float(np.median(v)) for k, v in times.items()}
    name, power = card()
    out = dict(workload=d.name + ", two groups per structure (random plane through the centroid)", atoms=N, structures=S,
               n_points=n_points, reps=args.reps, median_ms=med, spread_ms={k: [float(min(v)), float(max(v))] for k, v in times.items()},
               ratio_b_over_a=med["b_grouped"] / med["a_plain"], ratio_b_over_c=med["b_grouped"] / med["c_two_run"],
               grouped_host_ms=host_ms, other_group_neighbour_fraction=other_group_fraction(d, group, probe, args.sample),
               fraction_sample_structures=min(args.sample, S), isolated_counts_equal_two_run=counts_equal, gpu=name,
               power_limit=power)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    bs.close()
    b.close()
    eng.close()
    if not counts_equal:
        sys.exit(1)


if __name__ == "__main__":
    main()
