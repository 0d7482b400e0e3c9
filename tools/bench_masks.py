#!/usr/bin/env python
"""Cost of exposed-point masks (Batch.run_masks_*) against the plain run, CUDA events, alternating repetitions in one process.

Device-resident, counts + per-atom areas + level sums (the same outputs for both runs; the masked run also writes the masks):
  cfg2  seeded proteome batch, 4,400 structures, 100 points (the fused kernels)
  cfg5  seeded capsid shell, 1 M atoms, 960 points (the large-structure path, chunked cap tables)
Host form on cfg2 (pageable numpy buffers for both runs, so both take the per-chunk pipeline): the masks add n_atoms * W * 4
bytes of copy-out (16 B per atom at 100 points, as much as the float4 input), timed by the host clock around each call.
The mask popcounts are checked against the plain counts.  Prints one JSON line.
usage: python tools/bench_masks.py [--reps 10] [--host-reps 5] [--out path]
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


def popcounts(m):
    return np.unpackbits(np.ascontiguousarray(m).view(np.uint8), axis=1).sum(axis=1)


def device_leg(eng, d, n_points, reps):
    import torch
    dev = torch.device("cuda", 0)
    N, S = d.n_atoms, len(d.struct_off) - 1
    W = (n_points + 31) // 32
    b = eng.batch(d.struct_off, d.seg_be, d.struct_seg_off, d.seg_polar)
    d_x = torch.from_numpy(d.xyzr).to(dev)
    z = lambda n, dt=torch.float32: torch.zeros(n, dtype=dt, device=dev)   # noqa: E731
    nseg = 0 if d.seg_be is None else len(d.seg_be)
    pc, pa, ps, pp = z(N, torch.int32), z(N), z(nseg), z((S, 3))
    mc, ma, ms, mp = z(N, torch.int32), z(N), z(nseg), z((S, 3))
    mask = z((N, W), torch.int32)
    segs = lambda t: t if nseg else None   # noqa: E731
    runs = {"plain": lambda: b.run_device(d_x, n_points=n_points, counts=pc, atom_sasa=pa, seg_sasa=segs(ps), protein=pp),
            "masked": lambda: b.run_masks_device(d_x, mask, n_points=n_points, counts=mc, atom_sasa=ma, seg_sasa=segs(ms), protein=mp)}
    for f in runs.values():   # warm-up: modules, tables, workspaces
        f()
    torch.cuda.synchronize()
    b.sync()
    times = {k: [] for k in runs}
    for _ in range(reps):
        for k, f in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
    b.sync()
    runs["masked"]()
    streamed = int(b.sync()["streamed_atoms"])   # atoms the masked run sent through the streaming routine
    same = all(bool(torch.equal(x, y)) for x, y in ((pc, mc), (pa, ma), (ps, ms), (pp, mp)))
    pc_ok = bool(np.array_equal(popcounts(mask.cpu().numpy()), pc.cpu().numpy()))
    b.close()
    med = {k: float(np.median(v)) for k, v in times.items()}
    return dict(workload=d.name, atoms=N, structures=S, n_points=n_points, reps=reps, median_ms=med,
                spread_ms={k: [float(min(v)), float(max(v))] for k, v in times.items()},
                ratio_masked_over_plain=med["masked"] / med["plain"], mask_bytes=N * W * 4, masked_streamed_atoms=streamed,
                outputs_equal_plain=same, popcounts_equal_counts=pc_ok)


def host_leg(eng, d, n_points, reps):
    b = eng.batch(d.struct_off, d.seg_be, d.struct_seg_off, d.seg_polar)
    runs = {"plain": lambda: b.run_host(d.xyzr, n_points=n_points), "masked": lambda: b.run_masks_host(d.xyzr, n_points=n_points)}
    for f in runs.values():
        f()
    wall = {k: [] for k in runs}
    span = {k: [] for k in runs}
    for _ in range(reps):
        for k, f in runs.items():
            t0 = time.perf_counter()
            r = f()
            wall[k].append((time.perf_counter() - t0) * 1e3)
            span[k].append(float(r.stats["kernel_ms"]))
    b.close()
    med = {k: float(np.median(v)) for k, v in wall.items()}
    return dict(workload=d.name, n_points=n_points, reps=reps, median_wall_ms=med,
                median_device_span_ms={k: float(np.median(v)) for k, v in span.items()},
                ratio_masked_over_plain=med["masked"] / med["plain"], input_bytes=d.n_atoms * 16,
                mask_bytes=d.n_atoms * ((n_points + 31) // 32) * 4, buffers="pageable numpy (per-chunk pipeline for both)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--host-reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from rustsasa_b200 import Engine, workloads as W
    eng = Engine(0)
    cfg2 = W.proteome_batch(4400, seed=W.SEED)
    out = dict(cfg2=device_leg(eng, cfg2, 100, args.reps), cfg5=device_leg(eng, W.capsid_shell(1000000), 960, args.reps),
               cfg2_host=host_leg(eng, cfg2, 100, args.host_reps))
    out["gpu"], out["power_limit"] = card()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    eng.close()
    ok = all(out[k]["outputs_equal_plain"] and out[k]["popcounts_equal_counts"] for k in ("cfg2", "cfg5"))
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
