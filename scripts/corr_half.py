"""Time and memory of the fp16 correlation pyramid (storage="f16", cf_corr_build_half / cf_corr_lookup_half) against
the default fp32 pyramid, at the five config shapes (D = 256, 4 levels, radius 4, precision "auto").

For each shape and storage:
  build_ms    the pyramid build alone
  lookup_ms   one lookup, smooth coordinates (coords_grid + an affine field + N(0, 0.5^2))
  step_ms     build + 6 lookups (the flow network's use of one block)
  peak_mb     growth of torch.cuda.max_memory_allocated for one CorrBlock (pyramid + operand copies)
Times are CUDA events around --iters calls after --warmup calls, medians of --rounds rounds in which the two storages
alternate.  Each side cycles through as many independent sets of inputs and pyramids as it takes to exceed 256 MB,
twice the 126 MB L2, so no call reads what the previous one left in the L2.  The card name, power limit and maximum SM
clock are read with a read-only `nvidia-smi --query-gpu` in the same process; the result is DIR/corr_half.json.

    python scripts/corr_half.py --out DIR [--iters 10] [--warmup 3] [--rounds 5]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [(8, 24, 32), (64, 36, 44), (64, 60, 80), (1, 80, 124), (2, 92, 160)]   # (B, h, w), feature-map pixels
D, LEVELS, RADIUS = 256, 4, 4


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "--id=0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit_w": float(power), "sm_max_mhz": float(clock)}
    except (OSError, ValueError, subprocess.TimeoutExpired):
        return {"name": None, "power_limit_w": None, "sm_max_mhz": None}


def smooth_coords(B, h, w, dev, seed):
    import torch
    import cistaflow_b200 as cf
    g = torch.Generator(device=dev).manual_seed(seed)
    c = cf.coords_grid(B, h, w, device=dev)
    a = 0.05 * torch.randn(B, 2, 2, device=dev, generator=g)
    xy = c - torch.tensor([w / 2, h / 2], device=dev).view(1, 2, 1, 1)
    c = c + torch.einsum("bij,bjhw->bihw", a, xy) + 0.5 * torch.randn(B, 2, h, w, device=dev, generator=g)
    return c.contiguous()


def pyramid_bytes(B, h, w, elt):
    N = h * w
    return sum(B * N * (h >> l) * (w >> l) for l in range(LEVELS)) * elt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    import torch
    import cistaflow_b200 as cf
    assert torch.cuda.is_available(), "corr_half.py measures on the GPU"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    result = {"card": card(), "iters": args.iters, "warmup": args.warmup, "rounds": args.rounds, "shapes": []}
    for B, h, w in SHAPES:
        per_set = 2 * B * D * h * w * 4 + pyramid_bytes(B, h, w, 2)
        nsets = max(1, min(16, -(-(256 << 20) // per_set)))
        g = torch.Generator(device=dev).manual_seed(h * w)
        sets = [(torch.randn(B, D, h, w, device=dev, generator=g), torch.randn(B, D, h, w, device=dev, generator=g),
                 smooth_coords(B, h, w, dev, seed=k)) for k in range(nsets)]
        row = {"B": B, "h": h, "w": w, "sets": nsets}
        # peak memory of one block, each storage
        for st in ("f32", "f16"):
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            base = torch.cuda.memory_allocated(dev)
            torch.cuda.reset_peak_memory_stats(dev)
            with torch.no_grad():
                blk = cf.CorrBlock(sets[0][0], sets[0][1], LEVELS, RADIUS, storage=st)
            torch.cuda.synchronize()
            row[f"peak_mb_{st}"] = (torch.cuda.max_memory_allocated(dev) - base) / 2 ** 20
            del blk
        # the pyramids the timed calls write / read, one per set and storage
        torch.cuda.empty_cache()
        pyrs = {st: [[torch.empty(B * h * w, 1, h >> l, w >> l, dtype=dt, device=dev) for l in range(LEVELS)]
                     for _ in range(nsets)]
                for st, dt in (("f32", torch.float32), ("f16", torch.float16))}
        outs = torch.empty(B, LEVELS * (2 * RADIUS + 1) ** 2, h, w, device=dev)

        def build(st, k):
            f1, f2, _ = sets[k % nsets]
            cf.build_pyramid(f1, f2, LEVELS, out=pyrs[st][k % len(pyrs[st])], storage=st)

        def look(st, k):
            cf.corr_lookup(pyrs[st][k % len(pyrs[st])], sets[k % nsets][2], RADIUS, out=outs)

        def step(st, k):
            build(st, k)
            for _ in range(6):
                look(st, k)

        for st in ("f32", "f16"):   # every pyramid written once before the lookups read it
            for k in range(len(pyrs[st])):
                build(st, k)
        times = {}
        for what, fn in (("build", build), ("lookup", look), ("step", step)):
            for st in ("f32", "f16"):
                times[(what, st)] = []
            for _ in range(args.rounds):
                for st in ("f32", "f16"):
                    for k in range(args.warmup):
                        fn(st, k)
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    for k in range(args.iters):
                        fn(st, k)
                    b.record()
                    b.synchronize()
                    times[(what, st)].append(a.elapsed_time(b) / args.iters)
            for st in ("f32", "f16"):
                row[f"{what}_ms_{st}"] = statistics.median(times[(what, st)])
        result["shapes"].append(row)
        print(json.dumps(row), flush=True)
        del sets, pyrs, outs
        torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "corr_half.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
