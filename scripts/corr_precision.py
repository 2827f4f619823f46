"""Time, accuracy and useful rate of the correlation pyramid build for each precision.

For fp32, tf32, auto and 3xtf32 at the headline launch (64 x 256 x 60x80) and the config shapes, 4 levels:
  ms      CUDA events around --iters calls of build_pyramid after --warmup calls, into two output sets used in turn
          (level 0 alone is 5.9 GB at the headline: every launch writes past the L2); inputs stay the same
  err     normwise max|err| / max|ref| of level 0 against a float64 contraction, on 64 sampled query rows of the
          first and the last batch item
  tflops  useful rate 2*B*N^2*D / time (the three MMAs of 3xtf32 count once)
  kernels (--kernels) device time per kernel and call from a torch.profiler pass of its own, after the timed loop
The card name, power limit and maximum SM clock are read with a read-only `nvidia-smi --query-gpu`; the result is
written to DIR/corr_precision.json.

    python scripts/corr_precision.py --out DIR [--iters 20] [--warmup 3] [--shapes headline] [--kernels]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (batch, image height, image width): the feature maps are 1/8 of the x32-padded image, D = 256
SHAPES = {
    "headline": [(64, 480, 640)],
    "all": [(64, 480, 640), (8, 480, 640), (64, 180, 240), (64, 260, 346), (1, 624, 970), (2, 128, 192)],
}
PRECISIONS = ("fp32", "tf32", "auto", "3xtf32")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "--id=0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit_w": float(power), "sm_max_mhz": float(clock)}
    except (OSError, ValueError, subprocess.TimeoutExpired):
        return {"name": None, "power_limit_w": None, "sm_max_mhz": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", choices=sorted(SHAPES), default="all")
    ap.add_argument("--kernels", action="store_true")
    args = ap.parse_args()
    assert args.iters >= 20, "time at least 20 launches"

    import torch

    import cistaflow_b200 as cf
    from cistaflow_b200 import _lib, synth

    assert torch.cuda.is_available(), "corr_precision.py measures on the GPU"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    rows = []
    for (B, H, W) in SHAPES[args.shapes]:
        hp, wp = synth.padded_dims(H, W)
        h, w, D = hp // 8, wp // 8, 256
        N = h * w
        gen = torch.Generator(device=dev).manual_seed(B * 100003 + H)
        a = torch.randn(B, D, h, w, device=dev, generator=gen)
        b = torch.randn(B, D, h, w, device=dev, generator=gen)
        sample = torch.randint(0, N, (64,), device=dev, generator=gen)
        exact = {i: (a[i].reshape(D, N)[:, sample].double().T @ b[i].reshape(D, N).double()) / D ** 0.5 for i in (0, B - 1)}
        for prec in PRECISIONS:
            outs = [[torch.empty((B * N, 1, h >> l, w >> l), device=dev) for l in range(4)] for _ in range(2)]
            for k in range(args.warmup):
                cf.build_pyramid(a, b, 4, precision=prec, out=outs[k % 2])
            kernel = lib.cf_last_kernel().decode()
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for k in range(args.iters):
                cf.build_pyramid(a, b, 4, precision=prec, out=outs[k % 2])
            t1.record()
            torch.cuda.synchronize()
            ms = t0.elapsed_time(t1) / args.iters
            l0 = outs[(args.iters - 1) % 2][0].view(B, N, N)
            err = max(float((l0[i, sample].double() - ref).abs().max() / ref.abs().max()) for i, ref in exact.items())
            row = {"batch": B, "image": [H, W], "map": [h, w], "D": D, "precision": prec, "ms": ms,
                   "tflops": 2.0 * B * N * N * D / (ms * 1e-3) / 1e12, "err_vs_f64": err, "last_kernel": kernel}
            if args.kernels:
                calls = 5
                with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                    for k in range(calls):
                        cf.build_pyramid(a, b, 4, precision=prec, out=outs[k % 2])
                    torch.cuda.synchronize()
                row["kernels_ms"] = {e.key[:48]: e.self_device_time_total / calls / 1e3 for e in prof.key_averages()
                                     if e.self_device_time_total > 0}
            rows.append(row)
            print(f"{B:3d} x {h}x{w} {prec:7s} {ms:9.3f} ms {row['tflops']:7.1f} TFLOP/s  err {err:.2e}  ({kernel})", flush=True)
            for name, t in row.get("kernels_ms", {}).items():
                print(f"      {t:9.3f} ms  {name}", flush=True)
            del outs
            torch.cuda.empty_cache()
    speedup = {}
    for r in rows:
        if r["precision"] == "3xtf32":
            f = next(x for x in rows if x["precision"] == "fp32" and x["batch"] == r["batch"] and x["map"] == r["map"])
            speedup[f"{r['batch']}x{r['map'][0]}x{r['map'][1]}"] = f["ms"] / r["ms"]
    result = {"card": card(), "iters": args.iters, "warmup": args.warmup, "rows": rows, "speedup_3xtf32_over_fp32": speedup}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "corr_precision.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"card": result["card"], "speedup_3xtf32_over_fp32": speedup}))


if __name__ == "__main__":
    main()
