"""Time and memory of the on-demand correlation lookup (AlternateCorrBlock) against the materialized pyramid.

For each feature-map shape (D = 256, 4 levels, radius 4):
  prepare_ms         cf_corr_alt_prepare (transpose + pooling of the feature maps)
  lookup_ms          one on-demand lookup: tensor cores ("auto") and the fp32 SIMT kernel ("fp32"), for smooth
                     coordinates (coords_grid + an affine field + N(0, 0.5^2)) and noise coordinates (+ N(0, 5^2))
  ab_ms              CorrBlock("auto") build + 6 / + 12 lookups against prepare + 6 / + 12 on-demand lookups, smooth
                     coordinates; the two sides alternate within one process, --rounds times, median reported
  peak_mb            growth of torch.cuda.max_memory_allocated for one block and one lookup, each side
Times are CUDA events around --iters calls after --warmup calls; the same state and coordinates are read every call.
The on-demand state (2.33 feature maps) fits the 126 MB L2 at 8 x 24x32 (15 MB), 1 x 80x124 (24 MB) and 2 x 92x160
(70 MB), so those lookups read it from L2; at 64 x 36x44 (243 MB) and 64 x 60x80 (733 MB) it does not.  Lookups of
about 0.1 ms or less (8 x 24x32, 1 x 80x124, 2 x 92x160) are bound by per-call overhead: the Python call, the host
encoding of 1 + L tensor maps and two kernel launches.  The card name, power limit and maximum SM clock are read with
a read-only `nvidia-smi --query-gpu` in the same process; the result is DIR/corr_alt.json.

--trace-fit (CPU only, no GPU needed) instead counts, with the host restatement of the lookup's per-tile predicate, the
16x8 tiles that the models' own coordinates send to the tensor cores: the last-iteration coordinates of the
tests/golden/trace3_* fixtures (three consecutive frames of each model at 180x240), 4 levels, radius 4.

    python scripts/corr_alt.py --out DIR [--iters 20] [--warmup 3] [--rounds 5]
    python scripts/corr_alt.py --trace-fit
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

SHAPES = [(8, 24, 32), (64, 36, 44), (64, 60, 80), (1, 80, 124), (2, 92, 160)]   # (B, h, w), feature-map pixels


def tile_fits(coords, levels, radius):
    """Host restatement of tile_box() in csrc/corr_alt.cu: per batch item and 16x8 query tile, True when every level's
    box of patch origins fits the tensor-core kernel (bw_l wide, 8 bands of bh_l = 256 / bw_l rows high)."""
    import numpy as np
    c = np.clip(np.asarray(coords, np.float32), -1.0e6, 1.0e6)   # NaN -> -1e6 as fminf(fmaxf(.)) does
    c = np.where(np.isnan(c), np.float32(-1.0e6), c)
    B, _, h, w = c.shape
    th, tw = -(-h // 8), -(-w // 16)
    fits = np.ones((B, th, tw), bool)
    for l in range(levels):
        need = (16 >> l) + 2 * radius + 4
        bw = 16 if need <= 16 else (32 if need <= 32 else 64)
        bh = 256 // bw
        base = np.floor(c / np.float32(2 ** l)).astype(np.int64) - radius       # [B, 2, h, w]
        for ty in range(th):
            for tx in range(tw):
                t = base[:, :, 8 * ty:8 * ty + 8, 16 * tx:16 * tx + 16].reshape(B, 2, -1)
                wd = t[:, 0].max(1) - t[:, 0].min(1) + 2 * radius + 2
                ht = t[:, 1].max(1) - t[:, 1].min(1) + 2 * radius + 2
                fits[:, ty, tx] &= (wd <= bw) & (ht <= 8 * bh)
    return fits


def trace_fit():
    import numpy as np
    for trace in ("trace3_eiflow", "trace3_eraft"):
        with np.load(os.path.join(ROOT, "tests", "golden", trace + ".npz")) as z:
            frames = int(z["meta"][3])
            for f in range(frames):
                n_lookup = int(z[f"f{f}/counts"][0])
                coords = z[f"f{f}/coords{n_lookup - 1}"]
                fits = tile_fits(coords, 4, 4)
                print(f"{trace} frame {f}: coords {tuple(coords.shape)}, {int(fits.sum())} of {fits.size} tiles "
                      f"({100.0 * fits.mean():.1f} %) on the tensor cores")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--trace-fit", action="store_true")
    args = ap.parse_args()
    if args.trace_fit:
        trace_fit()
        return
    assert args.out, "--out DIR"

    import torch

    import cistaflow_b200 as cf
    from corr_precision import card

    assert torch.cuda.is_available(), "corr_alt.py measures on the GPU"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def timed(fn, iters):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        t0, t1 = ev(), ev()
        t0.record()
        for _ in range(iters):
            fn()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / iters

    def peak_growth(fn):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        keep = fn()
        torch.cuda.synchronize()
        grown = torch.cuda.max_memory_allocated(dev) - base
        del keep
        torch.cuda.empty_cache()
        return grown / 2 ** 20

    rows = []
    with torch.no_grad():
        for (B, h, w) in SHAPES:
            D = 256
            gen = torch.Generator(device=dev).manual_seed(B * 1009 + h)
            f1 = torch.randn(B, D, h, w, device=dev, generator=gen)
            f2 = torch.randn(B, D, h, w, device=dev, generator=gen)
            grid = cf.coords_grid(B, h, w, device=dev)
            xs, ys = grid[:, 0] - w / 2, grid[:, 1] - h / 2
            flow = torch.stack([0.04 * xs - 0.03 * ys + 2.7, 0.02 * xs + 0.05 * ys - 1.6], 1)
            coords = {"smooth": grid + flow + 0.5 * torch.randn(B, 2, h, w, device=dev, generator=gen),
                      "noise": grid + 5.0 * torch.randn(B, 2, h, w, device=dev, generator=gen)}
            row = {"batch": B, "map": [h, w], "D": D, "levels": 4, "radius": 4}
            row["prepare_ms"] = timed(lambda: cf.AlternateCorrBlock(f1, f2), args.iters)
            row["lookup_ms"] = {}
            for prec, name in (("auto", "tc"), ("fp32", "simt")):
                blk = cf.AlternateCorrBlock(f1, f2, precision=prec)
                for kind, c in coords.items():
                    row["lookup_ms"][f"{name}_{kind}"] = timed(lambda: blk(c), args.iters)
                del blk
            ab = {}
            for n in (6, 12):
                def materialized():
                    blk = cf.CorrBlock(f1, f2, precision="auto")
                    for _ in range(n):
                        blk(coords["smooth"])

                def on_demand():
                    blk = cf.AlternateCorrBlock(f1, f2)
                    for _ in range(n):
                        blk(coords["smooth"])
                m, o = [], []
                for _ in range(args.rounds):   # alternate the two sides
                    m.append(timed(materialized, 3))
                    o.append(timed(on_demand, 3))
                ab[f"corrblock_build_plus_{n}"] = statistics.median(m)
                ab[f"alt_prepare_plus_{n}"] = statistics.median(o)
            row["ab_ms"] = ab
            row["peak_mb"] = {
                "corrblock": peak_growth(lambda: (lambda b: (b, b(coords["smooth"])))(cf.CorrBlock(f1, f2, precision="auto"))),
                "alt": peak_growth(lambda: (lambda b: (b, b(coords["smooth"])))(cf.AlternateCorrBlock(f1, f2))),
            }
            rows.append(row)
            lk = row["lookup_ms"]
            print(f"{B:3d} x {h}x{w}: prepare {row['prepare_ms']:.3f} ms | lookup tc {lk['tc_smooth']:.3f} / {lk['tc_noise']:.3f}"
                  f" simt {lk['simt_smooth']:.3f} / {lk['simt_noise']:.3f} ms (smooth / noise) | "
                  f"+6: {ab['corrblock_build_plus_6']:.3f} vs {ab['alt_prepare_plus_6']:.3f} ms, "
                  f"+12: {ab['corrblock_build_plus_12']:.3f} vs {ab['alt_prepare_plus_12']:.3f} ms (CorrBlock vs on-demand) | "
                  f"peak {row['peak_mb']['corrblock']:.0f} vs {row['peak_mb']['alt']:.0f} MB", flush=True)
            del f1, f2, coords, grid, flow
            torch.cuda.empty_cache()
    result = {"card": card(), "iters": args.iters, "warmup": args.warmup, "rounds": args.rounds, "rows": rows}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "corr_alt.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
