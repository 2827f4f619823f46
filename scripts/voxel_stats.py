"""Time of the window statistics with fp64 per-thread partials (voxel_stats_kernel) against a build of the library
that predates them, at the bench's headline shape (64 windows of 5 x 480x640, 100 000 events per window).

Both libraries are loaded side by side with ctypes (the same C ABI), and two calls are timed:
  preprocess_ms   cf_voxel_preprocess, std, hot-pixel threshold 25/5, out of place (statistics + normalise kernels)
  fused_ms        cf_voxel_bin, ATOMIC_L2, flavour numpy, fused std (zero -> scatter -> statistics -> normalise)
Times are CUDA events around --iters calls after --warmup calls, medians of --rounds rounds in which the two libraries
alternate.  Each call takes the next of two independent sets of inputs (2 x 393 MB grids, 2 x 205 MB events), so no
call reads what the previous one left in the 126 MB L2.  Outputs of the two libraries are compared at the same inputs.
The card name, power limit and maximum SM clock are read with a read-only `nvidia-smi --query-gpu` in the same
process; the result is DIR/voxel_stats.json.

    python scripts/voxel_stats.py --baseline OLD.so --out DIR [--iters 20] [--warmup 3] [--rounds 5]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

B, NB, H, W, EVENTS = 64, 5, 480, 640, 100_000
ATOMIC_L2, FLAVOUR_NUMPY, PRE_STD = 2, 1, 1


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "--id=0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit_w": float(power), "sm_max_mhz": float(clock)}
    except (OSError, ValueError, subprocess.TimeoutExpired):
        return {"name": None, "power_limit_w": None, "sm_max_mhz": None}


def bind(path):
    from cistaflow_b200 import _lib
    lib = ctypes.CDLL(path)
    for name in ("cf_voxel_preprocess", "cf_preprocess_workspace_bytes", "cf_voxel_bin", "cf_voxel_workspace_bytes",
                 "cf_last_error"):
        res, args = _lib.SYMBOLS[name]
        getattr(lib, name).restype, getattr(lib, name).argtypes = res, args
    return lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline", required=True, help="libcistaflow.so built from the parent commit")
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()

    import torch
    from cistaflow_b200 import _lib, synth
    assert torch.cuda.is_available(), "scripts/voxel_stats.py needs a CUDA device"
    dev = torch.device("cuda", 0)
    libs = {"fp32_partials": bind(os.path.abspath(a.baseline)), "fp64_partials": bind(_lib.LIB_PATH)}
    cells = NB * H * W
    thr = 25.0 / NB
    s = torch.cuda.current_stream().cuda_stream

    grids, events, offsets = [], [], []
    for k in range(2):
        g = torch.randn(B, cells, device=dev)
        grids.append(torch.where(torch.rand(B, cells, device=dev) < 0.2, g, torch.zeros_like(g)).contiguous())
        ev, off = synth.event_windows(B, EVENTS, H, W, seed=11 + k)
        events.append(torch.from_numpy(ev).to(dev))
        offsets.append(torch.from_numpy(off).to(dev))
    out = torch.empty(B, cells, device=dev)
    pws_bytes = libs["fp64_partials"].cf_preprocess_workspace_bytes(B, cells)
    pws = torch.empty(pws_bytes, dtype=torch.uint8, device=dev)
    vws_bytes = max(l.cf_voxel_workspace_bytes(B * EVENTS, B, NB, H, W, ATOMIC_L2, FLAVOUR_NUMPY, PRE_STD) for l in libs.values())
    vws = torch.empty(vws_bytes, dtype=torch.uint8, device=dev)

    def preprocess(lib, i):
        rc = lib.cf_voxel_preprocess(grids[i].data_ptr(), out.data_ptr(), B, cells, PRE_STD, thr, pws.data_ptr(),
                                     pws_bytes, s)
        assert rc == 0, lib.cf_last_error()

    def fused(lib, i):
        rc = lib.cf_voxel_bin(events[i].data_ptr(), offsets[i].data_ptr(), B * EVENTS, B, NB, H, W, ATOMIC_L2,
                              FLAVOUR_NUMPY, PRE_STD, thr, out.data_ptr(), vws.data_ptr(), vws_bytes, s)
        assert rc == 0, lib.cf_last_error()

    # the two libraries agree at the same inputs (the statistics differ in their last bits only)
    agree = {}
    for what, fn in (("preprocess", preprocess), ("fused", fused)):
        res = {}
        for name, lib in libs.items():
            fn(lib, 0)
            torch.cuda.synchronize()
            res[name] = out.clone()
        agree[what] = float((res["fp32_partials"] - res["fp64_partials"]).abs().max())

    def time_ms(fn, lib):
        for i in range(a.warmup):
            fn(lib, i & 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(a.iters):
            fn(lib, i & 1)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / a.iters

    times = {w: {n: [] for n in libs} for w in ("preprocess_ms", "fused_ms")}
    for _ in range(a.rounds):
        for name, lib in libs.items():
            times["preprocess_ms"][name].append(time_ms(preprocess, lib))
            times["fused_ms"][name].append(time_ms(fused, lib))
    result = {"card": card(), "shape": f"{B} x {NB}x{H}x{W}, {EVENTS} events per window",
              "max_abs_output_difference": agree,
              "median": {w: {n: statistics.median(v) for n, v in t.items()} for w, t in times.items()},
              "rounds": times}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "voxel_stats.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({k: result[k] for k in ("card", "shape", "max_abs_output_difference", "median")}, indent=1))


if __name__ == "__main__":
    main()
