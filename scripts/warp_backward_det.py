"""Time the deterministic warp adjoint (cf_warp_backward_det) against the atomic one (cf_warp_backward).

The training step's two warps, each with both gradients (image and flow) requested:
  frame   C = 1 at the full resolution, flow of the same size
  codes   C = 128 at half the resolution, the full-resolution flow down-sampled x0.5 inside the kernels
at 8 x 180x240 (the training crop) and 64 x 480x640, with smooth flow (synth.warp_inputs 'smooth', what a flow network
produces) and noise flow (N(0, 5^2) px per pixel + the affine component).

The C entry points are called directly on preallocated outputs and workspace.  Each side is timed with CUDA events
over --iters calls after --warmup calls; the two sides alternate within one process, --rounds times, and the median
of the rounds is reported.  Calls rotate over enough input sets that the sets together exceed the 126 MB L2 at least
three times, so every call reads its inputs from HBM.  The largest difference between the two sides' gradients,
relative to the largest gradient, is recorded as a check.  The card name, power limit and maximum SM clock are read
with a read-only `nvidia-smi --query-gpu`; the result is DIR/warp_backward_det.json and DIR/warp_backward_det.txt.
--kernels instead runs torch.profiler (CUDA activities) over --iters calls of the deterministic path at each shape
(smooth flow) and writes the device time per kernel and call to DIR/warp_backward_det_kernels.txt.

    python scripts/warp_backward_det.py --out DIR [--iters 10] [--warmup 2] [--rounds 5] [--small] [--kernels]
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

L2_BYTES = 126 << 20
# (name, B, C, H, W, flowH, flowW)
SHAPES = [("frame", 8, 1, 180, 240, 180, 240), ("codes", 8, 128, 90, 120, 180, 240),
          ("frame", 64, 1, 480, 640, 480, 640), ("codes", 64, 128, 240, 320, 480, 640)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "--id=0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit_w": float(power), "sm_max_mhz": float(clock)}
    except (OSError, ValueError, subprocess.TimeoutExpired):
        return {"name": None, "power_limit_w": None, "sm_max_mhz": None}


def input_sets(torch, synth, dev, B, C, H, W, fH, fW, kind, seed):
    set_bytes = 4 * B * (3 * C * H * W + 4 * fH * fW)   # grad_out, img, grad_img, flow, grad_flow
    n_sets = max(2, -(-3 * L2_BYTES // set_bytes))
    gen = torch.Generator(device=dev).manual_seed(seed)
    sets = []
    for k in range(n_sets):
        flow = torch.from_numpy(synth.warp_inputs(B, fH, fW, seed=seed + k, code_channels=1, flow_kind=kind)[2]).to(dev)
        img = torch.randn(B, C, H, W, generator=gen, device=dev)
        gout = torch.randn(B, C, H, W, generator=gen, device=dev)
        sets.append((gout, img, flow, torch.empty_like(img), torch.empty_like(flow)))
    return sets


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--small", action="store_true", help="only the 8 x 180x240 shapes")
    ap.add_argument("--kernels", action="store_true", help="per-kernel device times of the deterministic path")
    args = ap.parse_args()

    import torch
    import cistaflow_b200 as cf
    from cistaflow_b200 import _lib, synth
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = cf.load_library()
    stream = torch.cuda.current_stream(dev).cuda_stream
    rows, kernel_lines = [], []
    for name, B, C, H, W, fH, fW in SHAPES:
        if args.small and B != 8:
            continue
        for kind in (("smooth",) if args.kernels else ("smooth", "noise")):
            sets = input_sets(torch, synth, dev, B, C, H, W, fH, fW, kind, seed=100)
            ws_bytes = lib.cf_warp_backward_det_workspace_bytes(B, C, H, W, fH, fW)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)

            def atomic(s):
                go, im, fl, gi, gf = s
                _lib.check(lib.cf_warp_backward(go.data_ptr(), im.data_ptr(), fl.data_ptr(), gi.data_ptr(), gf.data_ptr(),
                                                B, C, H, W, fH, fW, -1.0, stream), "cf_warp_backward")

            def det(s):
                go, im, fl, gi, gf = s
                _lib.check(lib.cf_warp_backward_det(go.data_ptr(), im.data_ptr(), fl.data_ptr(), gi.data_ptr(),
                                                    gf.data_ptr(), B, C, H, W, fH, fW, -1.0, ws.data_ptr(), ws_bytes,
                                                    stream), "cf_warp_backward_det")

            if args.kernels:
                from torch.profiler import ProfilerActivity, profile
                for k in range(args.warmup):
                    det(sets[k % len(sets)])
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for k in range(args.iters):
                        det(sets[k % len(sets)])
                    torch.cuda.synchronize()
                per = {}
                for e in prof.events():
                    if e.device_type.name == "CUDA":
                        per[e.name] = per.get(e.name, 0.0) + e.device_time / 1e3 / args.iters
                kernel_lines.append(f"{name} {B} x {H}x{W} ({kind} flow): ms per call, {sum(per.values()):.3f} in all")
                for kname, ms in sorted(per.items(), key=lambda kv: -kv[1]):
                    kernel_lines.append(f"  {ms:9.3f}  {kname[:110]}")
                print("\n".join(kernel_lines[-len(per) - 1:]), flush=True)
                del sets, ws
                torch.cuda.empty_cache()
                continue
            # agreement of the two sides on the first input set
            atomic(sets[0])
            gi_a, gf_a = sets[0][3].clone(), sets[0][4].clone()
            det(sets[0])
            gi_d, gf_d = sets[0][3], sets[0][4]
            diff_img = ((gi_d - gi_a).abs().max() / gi_a.abs().max().clamp_min(1e-30)).item()
            diff_flow = ((gf_d - gf_a).abs().max() / gf_a.abs().max().clamp_min(1e-30)).item()
            del gi_a, gf_a

            def timed(fn):
                for k in range(args.warmup):
                    fn(sets[k % len(sets)])
                start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                start.record()
                for k in range(args.iters):
                    fn(sets[k % len(sets)])
                end.record()
                end.synchronize()
                return start.elapsed_time(end) / args.iters

            t_atomic, t_det = [], []
            for _ in range(args.rounds):
                t_atomic.append(timed(atomic))
                t_det.append(timed(det))
            row = {"warp": name, "batch": B, "channels": C, "image": [H, W], "flow": [fH, fW], "flow_kind": kind,
                   "input_sets": len(sets), "workspace_mb": ws_bytes / 1e6,
                   "atomic_ms": statistics.median(t_atomic), "det_ms": statistics.median(t_det),
                   "atomic_ms_rounds": t_atomic, "det_ms_rounds": t_det,
                   "max_rel_diff_grad_img": diff_img, "max_rel_diff_grad_flow": diff_flow}
            row["det_over_atomic"] = row["det_ms"] / row["atomic_ms"]
            rows.append(row)
            print(json.dumps({k: row[k] for k in ("warp", "batch", "image", "flow_kind", "atomic_ms", "det_ms",
                                                  "det_over_atomic")}), flush=True)
            del sets, ws
            torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    if args.kernels:
        c = card()
        with open(os.path.join(args.out, "warp_backward_det_kernels.txt"), "w") as fh:
            fh.write(f"{c['name']}, power limit {c['power_limit_w']} W; torch.profiler over {args.iters} calls after "
                     f"{args.warmup} warm-up calls\n" + "\n".join(kernel_lines) + "\n")
        return
    result = {"card": card(), "iters": args.iters, "warmup": args.warmup, "rounds": args.rounds, "rows": rows}
    with open(os.path.join(args.out, "warp_backward_det.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    c = result["card"]
    lines = [f"{c['name']}, power limit {c['power_limit_w']} W, SM clock max {c['sm_max_mhz']} MHz; "
             f"median of {args.rounds} alternating rounds of {args.iters} calls (after {args.warmup} warm-up calls)",
             f"{'warp':6} {'batch x image':>16} {'flow':>7} {'atomic ms':>10} {'det ms':>9} {'det/atomic':>10} "
             f"{'ws MB':>8} {'rel diff img':>13} {'rel diff flow':>13}"]
    for r in rows:
        lines.append(f"{r['warp']:6} {r['batch']:>4} x {r['image'][0]:>3}x{r['image'][1]:<4} {r['flow_kind']:>7} "
                     f"{r['atomic_ms']:>10.3f} {r['det_ms']:>9.3f} {r['det_over_atomic']:>10.2f} {r['workspace_mb']:>8.1f} "
                     f"{r['max_rel_diff_grad_img']:>13.2e} {r['max_rel_diff_grad_flow']:>13.2e}")
    with open(os.path.join(args.out, "warp_backward_det.txt"), "w") as fh:
        fh.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
