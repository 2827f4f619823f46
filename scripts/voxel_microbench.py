"""Voxel binning (+normalise) timing at several sizes."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cistaflow_b200 as cf
from cistaflow_b200 import synth

dev = torch.device("cuda", 0)
cases = [(8, 15000, 180, 240), (64, 15000, 180, 240), (64, 50000, 260, 346), (512, 50000, 260, 346), (8, 100000, 480, 640)]
for (B, n, H, W) in cases:
    reps = max(1, min(8, 64 // B))
    sets = []
    for r in range(2):
        ev, off = synth.event_windows(min(B, 16), n, H, W, seed=5 + r)
        k = B // min(B, 16)
        import numpy as np
        evs = np.concatenate([ev] * k)
        offs = np.concatenate([[0], np.cumsum(np.tile(np.diff(off), k))]).astype(np.int64)
        sets.append((torch.from_numpy(evs).to(dev), torch.from_numpy(offs).to(dev)))
    out = torch.empty((B, 5, H, W), device=dev)
    for mode_norm in ("std", None):
        def run(i):
            e, o = sets[i % 2]
            cf.events_to_voxel_grid_batched(e, o, 5, W, H, normalize=mode_norm, filter_hot_pixel=mode_norm is not None,
                                            flavour="numpy", mode="atomic", out=out)
        for i in range(3):
            run(i)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(10):
            run(i)
        b.record()
        torch.cuda.synchronize()
        us = a.elapsed_time(b) / 10 * 1e3
        nbytes = B * (32 * n + 4 * 5 * H * W)
        print(f"B={B:4d} n={n:6d} {H}x{W} norm={mode_norm}: {us:9.1f} us  {nbytes / us / 1e3:8.1f} GB/s "
              f"({nbytes / us / 1e3 / 6545 * 100:5.1f}% of HBM)  {B * n / us:8.1f} Mev/s")
