#!/usr/bin/env python
"""Latency of ONE structure through sasa_b200_calculate_sasa_internal (host buffers, synchronous) -- BASELINE config 1.
usage (GPU box): latency_single.py [names...]"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rustsasa_b200 import Engine  # noqa: E402
from tests.golden_data import Golden  # noqa: E402

g = Golden()
eng = Engine(0)
for name in sys.argv[1:] or ["151L_H3.pdb", "example.cif", "4xfj", "1hbn", "1jz8"]:
    s = g.structure(name)
    x = s["xyzr"]
    for _ in range(5):
        eng.calculate_sasa_internal(x, None, 1.4, 100, -1)
    t0 = time.perf_counter()
    reps = 50
    for _ in range(reps):
        eng.calculate_sasa_internal(x, None, 1.4, 100, -1)
    dt = (time.perf_counter() - t0) / reps
    print(f"{name:14s} {x.shape[0]:6d} atoms  {dt * 1e6:8.1f} us/call  "
          f"{x.shape[0] / dt / 1e6:7.2f} M atoms/s", flush=True)
