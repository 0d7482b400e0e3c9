#!/usr/bin/env python
"""Small inputs through every kernel family, for compute-sanitizer (memcheck / racecheck / initcheck are 10-100x slower):
fused tight + generic kernels, large path at 100 and 960 points, atom-range split (plain and peer pointers to local vectors),
one-structure calls, frames, indexed wire format, level sums, submit / wait.  Results are checked against the oracle."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from oracle import load  # noqa: E402
from rustsasa_b200 import Engine, workloads as W  # noqa: E402
from rustsasa_b200.engine import index_radii  # noqa: E402

orc = load(fast=True)
eng = Engine(0)
ok = True


def check(name, cond):
    global ok
    print(("ok   " if cond else "FAIL ") + name, flush=True)
    ok = ok and bool(cond)


d = W.proteome_batch(6, seed=3)
b = eng.batch(d.struct_off, d.seg_be, d.struct_seg_off, d.seg_polar)
o = orc.run_batch(d.xyzr, d.struct_off, seg_be=d.seg_be, struct_seg_off=d.struct_seg_off)
r = b.run_host(d.xyzr)
check("fused tight kernel, all levels", np.array_equal(r.counts, o["counts"]) and np.array_equal(r.seg_sasa, o["seg"]))
pal, idx = index_radii(d.xyzr[:, 3])
r2 = b.run_indexed_host(d.xyzr[:, :3], idx, pal)
check("indexed wire format", np.array_equal(r2.counts, r.counts) and np.array_equal(r2.protein, r.protein))
j = b.submit_host(d.xyzr)
r3 = j.wait()
check("submit / wait", np.array_equal(np.asarray(r3.counts), r.counts))
# page-locked outputs: with more than one chunk in the plan (tools/gpu_sanitize.sh sets SASA_B200_CHUNK_ATOMS=4000) this is the
# gated single-launch pipeline -- one kernel, results stored straight into host memory
rp = b.run_host(d.xyzr, result=b._host_outputs(("counts", "atom", "seg", "protein"), "pinned"))
check(f"page-locked outputs ({rp.stats['gpu_launches']} launch(es)) == pageable outputs ({r.stats['gpu_launches']})",
      np.array_equal(np.asarray(rp.counts), r.counts) and np.array_equal(np.asarray(rp.seg_sasa), r.seg_sasa)
      and np.array_equal(np.asarray(rp.protein), r.protein) and np.array_equal(np.asarray(rp.atom_sasa), r.atom_sasa))
r4 = b.run_host(d.xyzr, n_points=300, want=("counts",))
o4 = orc.run_batch(d.xyzr, d.struct_off, 1.4, 300)
check("generic fused kernel with the chunked table (300 points)", np.array_equal(r4.counts, o4["counts"]))
r5 = b.run_host(d.xyzr, n_points=1500, want=("counts",))
o5 = orc.run_batch(d.xyzr, d.struct_off, 1.4, 1500)
check("generic fused kernel, point chunks (1500 points)", np.array_equal(r5.counts, o5["counts"]))
b.close()

a = W.large_assembly(7000)
for n in (100, 960):
    sasa, counts = eng.calculate_sasa_internal(a.xyzr, None, 1.4, n, -1, want_counts=True)
    oo = orc.calculate_sasa_internal(a.xyzr, 1.4, n, threads=-1)
    check(f"one-structure call, large path, {n} points", np.array_equal(counts, oo["counts"]) and np.array_equal(sasa, oo["sasa"]))
a17 = W.large_assembly(17000)   # >= kLargeTexAtoms (16,384) atoms: the texture-path instance of the 100-point cells kernel
sasa, counts = eng.calculate_sasa_internal(a17.xyzr, None, 1.4, 100, -1, want_counts=True)
oo17 = orc.calculate_sasa_internal(a17.xyzr, 1.4, 100, threads=-1)
check("one-structure call, large path with texture fetches, 100 points", np.array_equal(counts, oo17["counts"]) and np.array_equal(sasa, oo17["sasa"]))
b = eng.batch(a.struct_off, a.seg_be, a.struct_seg_off, a.seg_polar)
full = b.run_host(a.xyzr, n_points=960)
parts = [b.run_atom_range_host(a.xyzr, k, 3, n_points=960) for k in range(3)]
check("atom-range split (3 shares)", np.array_equal(parts[0].counts + parts[1].counts + parts[2].counts, full.counts))
check("large path level sums", np.array_equal(full.seg_sasa, orc.segment_sums(oo["sasa"], a.seg_be)))
d_x = torch.from_numpy(a.xyzr).cuda()
cnt = torch.zeros(a.n_atoms, dtype=torch.int32, device="cuda")
atm = torch.zeros(a.n_atoms, dtype=torch.float32, device="cuda")
for k in range(2):   # "peers" that are all the local vectors: every share writes the same complete vectors
    b.run_atom_range_peers_device(d_x, k, 2, [cnt.data_ptr()] * 2, [atm.data_ptr()] * 2, n_points=960)
torch.cuda.synchronize()
b.sync()
check("atom-range split with peer pointers", np.array_equal(cnt.cpu().numpy().view(np.uint32), full.counts))
b.close()

md = W.md_trajectory(n_frames=3, n_atoms=900)
F, N = md.xyz.shape[:2]
off = (np.arange(F + 1) * N).astype(np.uint64)
b = eng.batch(off, np.tile(md.seg_be, (F, 1)), (np.arange(F + 1) * len(md.seg_be)).astype(np.uint64), np.tile(md.seg_polar, F))
rf = b.run_frames_host(md.xyz, md.radii, want=("counts", "protein"))
xyzr = np.concatenate([md.xyz[0], md.radii[:, None]], axis=1)
of = orc.calculate_sasa_internal(xyzr, 1.4, 100)
check("frames entry point", np.array_equal(rf.counts[:N], of["counts"]))
b.close()
eng.close()
print("ALL OK" if ok else "FAILURES", flush=True)
sys.exit(0 if ok else 1)
