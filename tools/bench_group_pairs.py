#!/usr/bin/env python
"""Cost of the pairwise buried-area run, device-resident, CUDA events, alternated repetitions.

Workloads (100 points):
  cfg2 / 2   every structure of the seeded cfg2 proteome batch cut in two by a random plane through its centroid: the pairs run
             (Batch.run_group_pairs_device) against the grouped run (Batch.run_groups_device) -- the partner pass when it adds
             nothing the grouped run does not already give
  cfg2 / 4   every structure cut in four by two orthogonal planes through its centroid: the pairs run against today's route,
             the grouped run plus one plain run of the batch rebuilt with every pair g + h of a structure as a structure of its
             own (all six pairs: the quadrants meet along the cut axis)
  cfg4 / 12  the 150 k-atom cfg4 assembly cut into 12 sectors about an axis: the large-structure path with many partners,
             against the grouped run
Checks, bit for bit, on the timed inputs: the pairs run's complex and isolated outputs against the grouped run's, and on cfg2 / 4
every slot count against isolated - dimer count from the rebuilt batch (and no non-zero partner left out).  Prints one JSON line;
exits 1 when a check fails.
usage: python tools/bench_group_pairs.py [--structures 4400] [--reps 8] [--out path]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_interface import card, plane_groups  # noqa: E402

PROBE, NP = 1.4, 100


def quadrant_groups(struct_off, xyzr, seed):
    """Four groups per structure: the quadrants of two orthogonal random planes through its centroid."""
    rng = np.random.default_rng(seed)
    group = np.empty(xyzr.shape[0], np.uint32)
    for s in range(len(struct_off) - 1):
        a0, a1 = int(struct_off[s]), int(struct_off[s + 1])
        x = xyzr[a0:a1, :3].astype(np.float64)
        q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        c = x - x.mean(axis=0)
        group[a0:a1] = (c @ q[:, 0] > 0).astype(np.uint32) + 2 * (c @ q[:, 1] > 0).astype(np.uint32)
    return group


def sector_groups(xyzr, n):
    c = xyzr[:, :3].astype(np.float64) - xyzr[:, :3].astype(np.float64).mean(axis=0)
    ang = np.arctan2(c[:, 1], c[:, 0]) + np.pi
    return np.minimum((ang / (2 * np.pi) * n).astype(np.uint32), n - 1)


def dimer_order(struct_off, group, n_groups):
    """Today's route: per structure, the atoms of g + h for every pair g < h, each a structure of its own.  Returns (perm,
    off, owner): rebuilt atom k is original atom perm[k], and owner[k] is the partner group whose dimer it sits in."""
    perm, off, owner = [], [0], []
    for s in range(len(struct_off) - 1):
        a0, a1 = int(struct_off[s]), int(struct_off[s + 1])
        g = group[a0:a1]
        for a in range(n_groups):
            for b in range(a + 1, n_groups):
                idx = np.nonzero((g == a) | (g == b))[0]
                perm.append(a0 + idx)
                owner.append(np.where(g[idx] == a, b, a).astype(np.uint32))
                off.append(off[-1] + idx.size)
    return np.concatenate(perm), np.asarray(off, np.uint64), np.concatenate(owner)


def timed(runs, reps, syncs):
    import torch
    for f in runs.values():   # warm-up: modules, tables, workspaces
        f()
    torch.cuda.synchronize()
    for s in syncs:
        s.sync()
    times = {k: [] for k in runs}
    for _ in range(reps):
        for k, f in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
    for s in syncs:
        s.sync()
    return {k: float(np.median(v)) for k, v in times.items()}, {k: [float(min(v)), float(max(v))] for k, v in times.items()}


def same(a, b):
    import torch
    return bool(torch.equal(a.view(torch.int32), b.view(torch.int32)))


def outputs_equal(x, y):
    return all(same(getattr(u, f), getattr(v, f)) for u, v in zip(x[:2], y[:2]) for f in ("counts", "atom_sasa", "protein"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--structures", type=int, default=4400)
    ap.add_argument("--reps", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from rustsasa_b200 import Engine, workloads as W
    eng = Engine(0)
    dev = torch.device("cuda", 0)
    want = ("counts", "atom", "protein")
    out = {"n_points": NP, "reps": args.reps}
    ok = True

    d = W.proteome_batch(args.structures, seed=W.SEED)
    b = eng.batch(d.struct_off, d.seg_be, d.struct_seg_off, d.seg_polar)
    d_x = torch.from_numpy(d.xyzr).to(dev)
    # cfg2 cut in two
    g2 = torch.from_numpy(plane_groups(d.struct_off, d.xyzr, W.SEED + 17).view(np.int32)).to(dev)
    res = {}
    runs = {"grouped": lambda: res.__setitem__("g", b.run_groups_device(d_x, g2, probe_radius=PROBE, n_points=NP, want=want)),
            "pairs": lambda: res.__setitem__("p", b.run_group_pairs_device(d_x, g2, probe_radius=PROBE, n_points=NP, want=want,
                                                                           max_partners=1))}
    med, spread = timed(runs, args.reps, [b])
    torch.cuda.synchronize()
    c2 = outputs_equal(res["p"], res["g"])
    cpx, iso, pr = res["p"]
    c2 = c2 and same(pr.buried_counts[:, 0], iso.counts - cpx.counts)
    ok &= c2
    out["cfg2_two_groups"] = dict(atoms=d.n_atoms, structures=len(d.struct_off) - 1, median_ms=med, spread_ms=spread,
                                  ratio_pairs_over_grouped=med["pairs"] / med["grouped"], bit_identical=c2)

    # cfg2 cut in four
    group4 = quadrant_groups(d.struct_off, d.xyzr, W.SEED + 29)
    g4 = torch.from_numpy(group4.view(np.int32)).to(dev)
    perm, off, owner = dimer_order(d.struct_off, group4, 4)
    bd = eng.batch(off)
    d_xd = torch.from_numpy(np.ascontiguousarray(d.xyzr[perm])).to(dev)
    dcnt = torch.zeros(perm.shape[0], dtype=torch.int32, device=dev)
    dat, dpr = torch.zeros(perm.shape[0], device=dev), torch.zeros((len(off) - 1, 3), device=dev)

    def route():
        res["g4"] = b.run_groups_device(d_x, g4, probe_radius=PROBE, n_points=NP, want=want)
        bd.run_device(d_xd, probe_radius=PROBE, n_points=NP, counts=dcnt, atom_sasa=dat, protein=dpr)

    runs = {"grouped_plus_dimer_runs": route,
            "pairs": lambda: res.__setitem__("p4", b.run_group_pairs_device(d_x, g4, probe_radius=PROBE, n_points=NP, want=want,
                                                                            max_partners=3))}
    med, spread = timed(runs, args.reps, [b, bd])
    torch.cuda.synchronize()
    c4 = outputs_equal(res["p4"], res["g4"])
    _, iso4, p4 = res["p4"]
    part, bc = p4.partner.cpu().numpy().view(np.uint32), p4.buried_counts.cpu().numpy().view(np.uint32)
    dense = np.zeros((d.n_atoms, 4), np.int64)
    rows, cols = np.nonzero(bc > 0)
    dense[rows, part[rows, cols]] = bc[rows, cols]
    ref = np.zeros((d.n_atoms, 4), np.int64)
    ref[perm, owner] = iso4.counts.cpu().numpy()[perm].astype(np.int64) - dcnt.cpu().numpy()[:].astype(np.int64)
    c4 = c4 and bool(np.array_equal(dense, ref)) and int(p4.needed.cpu()[0]) <= 3
    ok &= c4
    out["cfg2_four_groups"] = dict(atoms=d.n_atoms, dimer_structures=len(off) - 1, dimer_atoms=int(perm.shape[0]), median_ms=med,
                                   spread_ms=spread, ratio_pairs_over_route=med["pairs"] / med["grouped_plus_dimer_runs"],
                                   partners_needed=int(p4.needed.cpu()[0]), bit_identical=c4)
    bd.close()
    b.close()

    # cfg4 in 12 sectors
    L = W.large_assembly()
    bl = eng.batch(L.struct_off)
    d_xl = torch.from_numpy(L.xyzr).to(dev)
    g12 = torch.from_numpy(sector_groups(L.xyzr, 12).view(np.int32)).to(dev)
    runs = {"grouped": lambda: res.__setitem__("gl", bl.run_groups_device(d_xl, g12, probe_radius=PROBE, n_points=NP, want=want)),
            "pairs": lambda: res.__setitem__("pl", bl.run_group_pairs_device(d_xl, g12, probe_radius=PROBE, n_points=NP, want=want,
                                                                             max_partners=16))}
    med, spread = timed(runs, args.reps, [bl])
    torch.cuda.synchronize()
    cl = outputs_equal(res["pl"], res["gl"])
    ok &= cl
    out["cfg4_twelve_sectors"] = dict(atoms=L.n_atoms, median_ms=med, spread_ms=spread,
                                      ratio_pairs_over_grouped=med["pairs"] / med["grouped"],
                                      partners_needed=int(res["pl"][2].needed.cpu()[0]), bit_identical=cl)
    bl.close()
    name, power = card()
    out.update(gpu=name, power_limit=power, all_checks_passed=bool(ok))
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    eng.close()
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
