#!/usr/bin/env python
"""Benchmark of the CISTA-Flow motion-compensation hot path (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Headline workload = BASELINE.json configs[4]: 64 independent 480x640 event sequences, cista-eiflow
shape, STRONG-scaled over the N GPUs of one box (64/N streams per rank, no data-path collective).
A *step* is one pass of the hot path over this rank's streams = exactly the hot-path calls of one
reconstructed frame per stream (SURVEY.md section 3.1; reference loop test_wo_flow.py:109-149,
DCEIFlow/DCEIFlow.py:209-227, e2v/e2v_model.py:184-191):
  1. event windows -> voxel grids + fused normalisation      (B x 100 000 events, 5 bins)
  2. correlation pyramid build                                (fmaps [B,256,60,80], 4 levels)
  3. 6 pyramid lookups (DCEIFlow's 6 refinement iterations, radius 4)
  4. flow-guided warp of the previous frame [B,1,480,640] and the sparse codes [B,128,240,320]
     (flow x0.5 down-sampling fused)
metric = reconstructed frames/s of the hot path (whole job, no network runs); Mevents/s beside it.

value      inputs resident in HBM, the step replayed as one CUDA graph, timed with CUDA events on the
           launching stream; max over ranks.  Inputs + outputs of a step are ~17 GB at N=1 (>> 126 MB L2).
e2e        same step through the public Python API from pinned HOST buffers: H2D of every input and
           D2H of every result inside the timed region (three streams, two buffer sets).
roofline   the dominant kernel of the step (correlation pyramid build), timed alone with CUDA events in
           this run; algorithmic bytes / measured HBM peak, tensor-pipe figure beside it.
cpu_baseline / --impl reference   the oracle port of the reference's own CPU path (the same NumPy/torch
           CPU calls the reference makes) on a bounded sample of the same workload, all host threads.
other_configs   (N=1 only) configs[0] B=1 latency, configs[1] (round 1's headline), configs[2] the
           260x346 voxel+warp microbench at x1/x64/x1024 windows, configs[3] 624x970 / 1 M events.
--dump-outputs DIR   after the timed steps, what the last timed step returned (voxel grids, every lookup output, warped
           frame and codes; rank 0) as DIR/<name>.npy, float32, a fixed sample of each output (see dump_outputs).  The
           inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

# the tree may be read-only: no __pycache__ next to the sources
sys.dont_write_bytecode = True

# torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU reference arm (rank 0) must get all host cores
if os.environ.get("OMP_NUM_THREADS") == "1" and os.environ.get("RANK", "0") == "0":
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)

import numpy as np  # noqa: E402
import torch  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TOTAL_STREAMS = 64
# ---- workloads: BASELINE.json configs ------------------------------------------------------------------
WORKLOADS = {
    "configs[4]": dict(
        workload="configs[4]: 64 independent 480x640 sequences, cista-eiflow hot path (100000 ev/window, 5 bins, "
                 "fmaps [B,256,60,80], CorrBlock 4 levels radius 4, 6 lookups/frame, codes [B,128,240,320]), "
                 "64/N streams per GPU",
        H=480, W=640, streams=TOTAL_STREAMS, events=100000, lookups=6),
    "configs[0]": dict(workload="configs[0]: cista-eiflow hot path, 180x240, 15000 ev/frame, batch 1, 6 lookups/frame",
                       H=180, W=240, streams=1, events=15000, lookups=6),
    "configs[1]": dict(workload="configs[1]: cista-eraft hot path, 180x240, 15000 ev/frame, batch 8, 12 lookups/frame",
                       H=180, W=240, streams=8, events=15000, lookups=12),
    "configs[3]": dict(workload="configs[3]: cista-eiflow hot path, 624x970 (HS-ERGB scale), 1000000 ev/window, batch 1, "
                                "6 lookups/frame", H=624, W=970, streams=1, events=1000000, lookups=6),
}
COMMON = dict(bins=5, levels=4, radius=4, code_channels=128, warp_mode="forward", flow_kind="smooth")
DISTINCT = 4   # distinct synthetic streams generated on the host; a rank's batch tiles them (cheap host side)


def make_cfg(name):
    cfg = dict(WORKLOADS[name])
    cfg.update(COMMON)
    return cfg


def public_config(cfg, world):
    """The `config` object of the JSON line: identical for both arms (ours / reference)."""
    per_rank = cfg["streams"] // world
    return {"workload": cfg["workload"], "H": cfg["H"], "W": cfg["W"], "streams_total": cfg["streams"],
            "streams_per_gpu": per_rank, "events_per_window": cfg["events"], "bins": cfg["bins"],
            "lookups": cfg["lookups"], "corr_levels": cfg["levels"], "corr_radius": cfg["radius"],
            "code_channels": cfg["code_channels"], "warp_mode": cfg["warp_mode"], "flow_kind": cfg["flow_kind"],
            "parallelism": f"{world} x {per_rank} independent streams (strong scaling of a fixed {cfg['streams']}-stream "
                           f"job), no data-path collective",
            "l2": "inputs + outputs of one step exceed the 126 MB L2 (no flush needed); two rotating buffer sets"}


def make_host_streams(cfg, seed0, n):
    """n distinct synthetic streams (NumPy, SURVEY.md 8d recipe): one frame's hot-path inputs each."""
    from cistaflow_b200 import synth
    H, W = cfg["H"], cfg["W"]
    ev, off = synth.event_windows(n, cfg["events"], H, W, seed0)
    img, codes, flow = synth.warp_inputs(n, H, W, seed0 + 1, cfg["code_channels"], flow_kind=cfg["flow_kind"])
    _, _, flow_noise = synth.warp_inputs(1, H, W, seed0 + 5, 1, flow_kind="noise")
    f1, f2, c0 = synth.corr_inputs(n, H, W, seed0 + 2)
    rng = np.random.default_rng(seed0 + 3)
    coords = [c0] + [(c0 + 0.5 * rng.standard_normal(c0.shape)).astype(np.float32) for _ in range(cfg["lookups"] - 1)]
    return dict(events=ev, offsets=off, img=img, codes=codes, flow=flow, flow_noise=flow_noise, fmap1=f1, fmap2=f2,
                coords=coords)


def tile_rows(a, B):
    """[n, ...] -> [B, ...] by repetition (torch tensor, any device)."""
    n = a.shape[0]
    if n == B:
        return a
    rep = -(-B // n)
    return a.repeat((rep,) + (1,) * (a.dim() - 1))[:B].contiguous()


def tile_events(ev, off, B):
    """n windows -> B windows by repetition: (events [sum,4], offsets [B+1]) as torch tensors on ev's device."""
    n = off.numel() - 1
    counts = (off[1:] - off[:-1])
    idx = torch.arange(B) % n
    parts = [ev[int(off[i]):int(off[i + 1])] for i in idx.tolist()]
    new_off = torch.zeros(B + 1, dtype=torch.int64)
    new_off[1:] = torch.cumsum(counts[idx], 0)
    return torch.cat(parts, 0).contiguous(), new_off


def bytes_model(cfg, B):
    """Algorithmic bytes / flops per step for B streams (SURVEY.md section 8d)."""
    H, W = cfg["H"], cfg["W"]
    hp, wp = -(-H // 32) * 32, -(-W // 32) * 32
    h, w = hp // 8, wp // 8
    N = h * w
    k = 2 * cfg["radius"] + 1
    lvl_cells = sum((h >> l) * (w >> l) for l in range(cfg["levels"]))
    return dict(
        voxel=B * (32 * cfg["events"] + 4 * cfg["bins"] * H * W),
        warp=B * (8 * H * W + 8 * H * W + (H // 2) * (W // 2) * 8 * cfg["code_channels"]),
        corr_build_bytes=4 * B * (2 * 256 * N + N * lvl_cells),
        corr_build_flops=2 * B * N * N * 256,
        lookup=B * N * (4 * cfg["levels"] * k * k + 8 + 4 * cfg["levels"] * (k + 1) ** 2),
        N=N, h=h, w=w)


# ---- clocks -------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, watts, reasons, capped = [], [], [], set(), 0
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            try:
                watts.append(float(parts[2]))
            except ValueError:
                pass
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
                    capped += n == "sw_power_cap"
        # median over the samples taken under load (the upper half: idle samples sit at the idle clock)
        load = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "sm_min_mhz_under_load": min(load) if load else None, "power_w_max": max(watts) if watts else None,
                "sw_power_cap_share_of_samples": capped / len(sm) if sm else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def ncu_traffic(kernel_prefix):
    """DRAM bytes of one launch of `kernel_prefix` from the committed ncu --set full summary of THIS workload
    (profiles/r02/headline_kernels_ncu_full.txt; None when absent)."""
    path = os.path.join(ROOT, "profiles", "r02", "headline_kernels_ncu_full.txt")
    try:
        lines = open(path).read().splitlines()
    except OSError:
        return None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for i, line in enumerate(lines):
        if line.startswith("---") and kernel_prefix in line:
            tot = 0.0
            for l2 in lines[i + 1:i + 8]:
                parts = l2.split()
                if parts and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(parts[1]) * unit.get(parts[2], 1.0)
            return tot
    return None


def numa_pin(local_rank):
    """Bind this rank (and therefore its pinned host buffers, first-touch) to the NUMA node of its GPU.
    Returns a short description for the JSON line.  Best effort: any failure leaves the affinity alone."""
    try:
        props = torch.cuda.get_device_properties(local_rank)
        bus = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return f"gpu {bus}: no NUMA node reported"
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = set(os.sched_getaffinity(0))
        cpus = [c for c in cpus if c in allowed]
        if not cpus:
            return f"gpu {bus}: node {node} has no allowed cpu"
        os.sched_setaffinity(0, cpus)
        return f"gpu {bus} -> NUMA node {node} ({len(cpus)} cpus)"
    except Exception as e:  # noqa: BLE001
        return f"not pinned ({type(e).__name__})"


# ---- CPU reference arm ----------------------------------------------------------------------------------
def cpu_step(cfg, host, ids):
    """The hot path of one frame for the streams `ids` of `host` on the CPU, through the oracle port (the same
    NumPy / torch CPU calls the reference makes, SURVEY.md section 3.1)."""
    from oracle import ref_port
    ev, off = host["events"], host["offsets"]
    grids = []
    for b in ids:
        g = ref_port.voxel_grid_numpy(ev[off[b]:off[b + 1]], cfg["bins"], cfg["W"], cfg["H"])
        grids.append(ref_port.preprocess_numpy(g, "std", True))
    sel = np.asarray(ids)
    with torch.no_grad():
        pyr = ref_port.corr_pyramid(torch.from_numpy(host["fmap1"][sel]), torch.from_numpy(host["fmap2"][sel]), cfg["levels"])
        outs = [ref_port.corr_lookup(pyr, torch.from_numpy(c[sel]), cfg["radius"]) for c in host["coords"]]
        wi, wz = ref_port.warp_frame_and_codes(torch.from_numpy(host["img"][sel]), torch.from_numpy(host["codes"][sel]),
                                               torch.from_numpy(host["flow"][sel]), cfg["warp_mode"])
    return grids, outs, wi, wz


def time_cpu(cfg, host, sample, steps, warmup):
    """(seconds per step, host threads, what the last step returned)"""
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
    except OSError:
        pass
    torch.set_num_threads(len(os.sched_getaffinity(0)))
    n = len(host["offsets"]) - 1
    ids = [i % n for i in range(sample)]
    for _ in range(warmup):
        cpu_step(cfg, host, ids)
    t0 = time.perf_counter()
    for _ in range(steps):
        last = cpu_step(cfg, host, ids)
    dt = time.perf_counter() - t0
    return dt / steps, torch.get_num_threads(), last


DUMP_BYTES = 48 << 20   # all files --dump-outputs writes, together


def dump_outputs(out_dir, grids, outs, wi, wz):
    """One step's results (voxel grids, lookup outputs, warped frame, warped codes) as out_dir/<name>.npy, float32.
    An output larger than its share of DUMP_BYTES is stored as its elements at a fixed sample of flat indices (sorted,
    NumPy default_rng(0)): the same positions on every run of the same workload."""
    arrays = {"voxel": torch.as_tensor(np.stack(grids)) if isinstance(grids, list) else grids,
              **{f"lookup{k}": o for k, o in enumerate(outs)}, "warped_frame": wi, "warped_codes": wz}
    cap = DUMP_BYTES // 4 // len(arrays)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.reshape(-1)
        if t.numel() > cap:
            idx = np.sort(np.random.default_rng(0).integers(0, t.numel(), cap))
            t = t[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return  # the CPU arm runs on rank 0 only
    sample = 4  # streams per step: a bounded sample of the 64-stream job (one 480x640 stream-frame is ~0.25 s on 8 cores)
    host = make_host_streams(cfg, 1234 + 1000 * 4, sample)
    sec, cores, last = time_cpu(cfg, host, sample, args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last)
    fps = sample / sec
    desc = (f"each step = the full hot path of {sample} of the 64 streams (480x640, 100000 events, 6 lookups) through "
            f"oracle/ref_port.py (the reference's own NumPy/torch CPU calls), {args.steps} steps after {args.warmup} "
            f"warm-up, all host threads")
    line = {
        "impl": "reference", "metric": "recon_frames_per_s", "value": fps, "unit": "frames/s",
        "mevents_per_s": sample * cfg["events"] / sec / 1e6,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 (f64 event time, tf32 correlation)", "data": "synthetic",
        "config": public_config(cfg, world),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---- our arm ----------------------------------------------------------------------------------------------
class HotPath:
    """Device-resident inputs of one rank for one workload + the step through the public API."""

    def __init__(self, cfg, B, dev, seed, n_sets=2, distinct=DISTINCT):
        import cistaflow_b200 as cf
        self.cf, self.cfg, self.B, self.dev = cf, cfg, B, dev
        self.host = [make_host_streams(cfg, seed + 101 * s, min(distinct, B)) for s in range(n_sets)]
        self.sets = [self._to_dev(h) for h in self.host]
        self.side = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]

    def _to_dev(self, h):
        B, dev = self.B, self.dev
        ev, off = tile_events(torch.from_numpy(h["events"]), torch.from_numpy(h["offsets"]), B)
        d = dict(events=ev.to(dev), offsets=off.to(dev))
        for k in ("img", "codes", "flow", "fmap1", "fmap2"):
            d[k] = tile_rows(torch.from_numpy(h[k]).to(dev), B)
        d["flow_noise"] = tile_rows(torch.from_numpy(h["flow_noise"]).to(dev), B)
        d["coords"] = [tile_rows(torch.from_numpy(c).to(dev), B) for c in h["coords"]]
        return d

    def voxel(self, d, out=None):
        c = self.cfg
        return self.cf.events_to_voxel_grid_batched(d["events"], d["offsets"], c["bins"], c["W"], c["H"], normalize="std",
                                                    filter_hot_pixel=True, flavour="numpy", mode="atomic", out=out)

    def step(self, d):
        """The hot path of one frame for B streams, through the public API (one chain of launches)."""
        c, cf = self.cfg, self.cf
        vox = self.voxel(d)
        blk = cf.CorrBlock(d["fmap1"], d["fmap2"], num_levels=c["levels"], radius=c["radius"])
        outs = [blk(x) for x in d["coords"]]
        wi, wz = cf.warp_frame_and_codes(d["img"], d["codes"], d["flow"], c["warp_mode"])
        return vox, outs, wi, wz

    def step_branched(self, d, cur):
        """The same calls; the three sub-paths that do not depend on each other inside one frame (voxel grids |
        pyramid build -> dependent lookups | frame + codes warp) are issued on three streams, i.e. captured as
        parallel branches of the step's CUDA graph (fills launch ramps and tails)."""
        c, cf = self.cfg, self.cf
        for s_ in self.side:
            s_.wait_stream(cur)
        with torch.cuda.stream(self.side[0]):
            vox = self.voxel(d)
        with torch.cuda.stream(self.side[1]):
            wi, wz = cf.warp_frame_and_codes(d["img"], d["codes"], d["flow"], c["warp_mode"])
        blk = cf.CorrBlock(d["fmap1"], d["fmap2"], num_levels=c["levels"], radius=c["radius"])
        outs = [blk(x) for x in d["coords"]]
        for s_ in self.side:
            cur.wait_stream(s_)
        return vox, outs, wi, wz


_WC_KEEP = []


def pinned_write_combined(t):
    """Host copy of device tensor `t` in cudaHostAllocWriteCombined | Portable memory (falls back to ordinary pinned
    memory when the runtime call is unavailable).  The buffer lives for the rest of the process."""
    import ctypes
    nbytes = t.numel() * t.element_size()
    try:
        rt = ctypes.CDLL("libcudart.so.12")
        ptr = ctypes.c_void_p()
        err = rt.cudaHostAlloc(ctypes.byref(ptr), ctypes.c_size_t(max(nbytes, 16)), ctypes.c_uint(0x01 | 0x04))
        if err != 0 or not ptr.value:
            raise OSError(f"cudaHostAlloc failed: {err}")
        buf = (ctypes.c_uint8 * max(nbytes, 16)).from_address(ptr.value)
        host = torch.frombuffer(buf, dtype=t.dtype, count=t.numel()).view(t.shape)
        _WC_KEEP.append(buf)
        staged = torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t)
        host.copy_(staged)          # sequential CPU writes into the write-combined buffer
        if not host.is_pinned():
            raise OSError("not recognised as pinned")
        return host
    except (OSError, AttributeError, RuntimeError):
        return torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t)


def capture(stream, fn):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        keep = fn()
    return g, keep


def time_graphs(graphs, stream, steps, warmup, barrier=None):
    """ms per replay: W untimed + K timed replays rotating over `graphs`, CUDA events on `stream`."""
    for i in range(warmup):
        graphs[i % len(graphs)].replay()
    (barrier or torch.cuda.synchronize)()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(steps):
        graphs[i % len(graphs)].replay()
    e1.record(stream)
    (barrier or torch.cuda.synchronize)()
    return e0.elapsed_time(e1) / steps


def kernel_times(hp, stream, model, hbm, tf32_peak, noise_flow=True):
    """Each of the four kernels alone: `inner` launches back to back inside a CUDA graph (no host gaps), rotating
    over the buffer sets, CUDA events on `stream`."""
    cf, cfg, dev = hp.cf, hp.cfg, hp.dev
    sets = hp.sets
    blocks = [cf.CorrBlock(d["fmap1"], d["fmap2"], num_levels=cfg["levels"], radius=cfg["radius"]) for d in sets]
    lookup_out = [cf.corr_lookup(blocks[i].corr_pyramid, d["coords"][0], cfg["radius"]) for i, d in enumerate(sets)]
    vox_out = [hp.voxel(d) for d in sets]
    warp_out = [cf.warp_frame_and_codes(d["img"], d["codes"], d["flow"], cfg["warp_mode"]) for d in sets]
    pyr_out = [b.corr_pyramid for b in blocks]

    def graph_time(fn, inner, reps=5):
        for i in range(len(sets)):
            fn(i)
        torch.cuda.synchronize()
        g, _ = capture(stream, lambda: [fn(k % len(sets)) for k in range(inner)])
        return time_graphs([g], stream, reps, 2) / inner * 1e-3

    small = model["corr_build_bytes"] < 2e8
    t = dict(
        lookup=graph_time(lambda i: cf.corr_lookup(pyr_out[i], sets[i]["coords"][0], cfg["radius"], out=lookup_out[i]),
                          12 if small else 4),
        voxel=graph_time(lambda i: hp.voxel(sets[i], out=vox_out[i]), 8 if small else 4),
        warp=graph_time(lambda i: cf.warp_frame_and_codes(sets[i]["img"], sets[i]["codes"], sets[i]["flow"], cfg["warp_mode"],
                                                          out=warp_out[i]), 8 if small else 4),
        build=graph_time(lambda i: cf.build_pyramid(sets[i]["fmap1"], sets[i]["fmap2"], cfg["levels"], out=pyr_out[i]),
                         8 if small else 2))
    if noise_flow:   # (headline workload only) the same build with TF32 operands forced: documents what CF_CORR_AUTO chose against
        t["build_tf32"] = graph_time(lambda i: cf.build_pyramid(sets[i]["fmap1"], sets[i]["fmap2"], cfg["levels"], precision="tf32",
                                                                out=pyr_out[i]), 8 if small else 2)
        t["warp_noise"] = graph_time(lambda i: cf.warp_frame_and_codes(sets[i]["img"], sets[i]["codes"], sets[i]["flow_noise"],
                                                                       cfg["warp_mode"], out=warp_out[i]), 8 if small else 4)

    def hbm_roof(nbytes, sec):
        return {"bound": "hbm", "achieved": nbytes / sec / 1e9, "peak": hbm, "unit": "GB/s",
                "frac": nbytes / sec / 1e9 / hbm, "ms_per_launch": sec * 1e3, "algorithmic_bytes": nbytes}

    kernels = {
        "corr_build": {**hbm_roof(model["corr_build_bytes"], t["build"]),
                       "tensor": {"achieved": model["corr_build_flops"] / t["build"] / 1e12, "peak": tf32_peak,
                                  "unit": "TFLOP/s (tf32)", "frac": model["corr_build_flops"] / t["build"] / 1e12 / tf32_peak}},
        "corr_lookup": hbm_roof(model["lookup"], t["lookup"]),
        "voxel_bin+normalise": {**hbm_roof(model["voxel"], t["voxel"]),
                                "mevents_per_s": hp.B * cfg["events"] / t["voxel"] / 1e6},
        "warp_frame_and_codes": hbm_roof(model["warp"], t["warp"]),
    }
    if noise_flow:
        kernels["corr_build"]["precision"] = "auto (fp16 operand copies on this shape; TF32 operands forced: %.4f ms)" % (t["build_tf32"] * 1e3) \
            if model["N"] % 64 == 0 and model["N"] >= 2048 and hp.B * model["N"] >= 19200 else "auto (TF32 operands on this shape)"
        kernels["warp_frame_and_codes[noise_flow]"] = {
            **hbm_roof(model["warp"], t["warp_noise"]),
            "note": "flow ~ N(0,5^2) px per pixel (SURVEY 8d adversarial variant: every tap of a warp in a different line)"}
    del blocks, lookup_out, vox_out, warp_out, pyr_out
    return kernels


def measure_tf32_peak(dev):
    """cuBLAS TF32 8192^3, best of 10 (the denominator of the tensor-pipe fraction, measured in this run)."""
    a = torch.randn(8192, 8192, device=dev)
    b = torch.randn(8192, 8192, device=dev)
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        for _ in range(3):
            torch.matmul(a, b)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    return 2 * 8192 ** 3 / (best * 1e-3) / 1e12


def other_config_line(name, dev, stream, hbm, tf32_peak, steps):
    """A secondary BASELINE config on one GPU: step time (branched CUDA graph) + the four kernels."""
    cfg = make_cfg(name)
    B = cfg["streams"]
    hp = HotPath(cfg, B, dev, 1234 + 1000 * int(name[8]), n_sets=2 if B * cfg["H"] * cfg["W"] < 4e6 else 1)
    for d in hp.sets:
        hp.step(d)
    torch.cuda.synchronize()
    graphs = [capture(stream, lambda d=d: hp.step_branched(d, stream))[0] for d in hp.sets]
    ms = time_graphs(graphs, stream, steps, 5)
    model = bytes_model(cfg, B)
    kern = kernel_times(hp, stream, model, hbm, tf32_peak, noise_flow=False)
    out = {"workload": cfg["workload"], "ms_per_step": ms, "frames_per_s": B / (ms * 1e-3),
           "mevents_per_s": B * cfg["events"] / (ms * 1e-3) / 1e6,
           "kernels": {k: {kk: v[kk] for kk in ("ms_per_launch", "achieved", "frac")} |
                       ({"tensor_frac": v["tensor"]["frac"]} if "tensor" in v else {}) for k, v in kern.items()}}
    del hp, graphs
    torch.cuda.empty_cache()
    return out


def stock_torch_line(cfg, B, dev):
    """SURVEY.md 8(d): the reference's own torch op sequences for this path on the same GPU (stock PyTorch CUDA kernels,
    eager), timed beside the library on the headline workload -- scripts/stock_torch_gpu.py.  A comparator, not a path
    of the library; a failure here must not lose the bench line."""
    try:
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import stock_torch_gpu
        hp = HotPath(cfg, B, dev, 1234 + 1000 * 4, n_sets=1)
        d, cf = hp.sets[0], hp.cf
        vox = cf.events_to_voxel_grid_batched(d["events"], d["offsets"], cfg["bins"], cfg["W"], cfg["H"], normalize="std",
                                              filter_hot_pixel=True, flavour="torch", mode="atomic")
        ours = (vox, cf.CorrBlock(d["fmap1"], d["fmap2"], num_levels=cfg["levels"], radius=cfg["radius"])(d["coords"][0]),
                *cf.warp_frame_and_codes(d["img"], d["codes"], d["flow"], cfg["warp_mode"]))
        out = stock_torch_gpu.measure(d, cfg, ours=ours)
        del hp, d, ours, vox
        torch.cuda.empty_cache()
        return out
    except Exception as e:  # noqa: BLE001
        torch.cuda.empty_cache()
        return {"unavailable": f"{type(e).__name__}: {e}"[:300]}


def microbench_config2(dev, stream, hbm):
    """configs[2]: voxel-binning + forward-splat warp microbench at 346x260, 5 bins, 50k events/window,
    batched x1 / x64 / x1024 windows (separates launch latency from bandwidth)."""
    import cistaflow_b200 as cf
    cfg = dict(workload="configs[2]: voxel-binning + forward-splat warp microbench, 260x346, 5 bins, 50000 ev/window",
               H=260, W=346, streams=1, events=50000, lookups=1, **COMMON)
    host = make_host_streams(cfg, 1234 + 1000 * 2, DISTINCT)
    rows = {}
    for B in (1, 64, 1024):
        model = bytes_model(cfg, B)
        ev, off = tile_events(torch.from_numpy(host["events"]), torch.from_numpy(host["offsets"]), B)
        ev, off = ev.to(dev), off.to(dev)
        img, codes, flow = (tile_rows(torch.from_numpy(host[k]).to(dev), B) for k in ("img", "codes", "flow"))
        vox = torch.empty((B, 5, cfg["H"], cfg["W"]), device=dev)
        wout = (torch.empty_like(img), torch.empty_like(codes))

        def f_vox():
            cf.events_to_voxel_grid_batched(ev, off, 5, cfg["W"], cfg["H"], normalize="std", filter_hot_pixel=True,
                                            flavour="numpy", mode="atomic", out=vox)

        def f_warp():
            cf.warp_frame_and_codes(img, codes, flow, "forward", out=wout)

        res = {}
        for label, fn, nbytes in (("voxel_bin+normalise", f_vox, model["voxel"]), ("warp_frame_and_codes", f_warp, model["warp"])):
            fn()
            torch.cuda.synchronize()
            inner = 16 if B == 1 else (4 if B == 64 else 1)
            g, _ = capture(stream, lambda: [fn() for _ in range(inner)])
            sec = time_graphs([g], stream, 5, 2) / inner * 1e-3
            res[label] = {"ms_per_launch": sec * 1e3, "achieved": nbytes / sec / 1e9, "frac": nbytes / sec / 1e9 / hbm}
        res["voxel_bin+normalise"]["mevents_per_s"] = B * cfg["events"] / (res["voxel_bin+normalise"]["ms_per_launch"] * 1e-3) / 1e6
        rows[f"x{B}"] = res
        del ev, off, img, codes, flow, vox, wout
        torch.cuda.empty_cache()
    return {"workload": cfg["workload"], "windows": rows,
            "note": "x1 re-runs the same L2-resident buffers (latency row); x64 / x1024 exceed the L2"}


def run_ours(args, cfg):
    import torch.distributed as dist
    from cistaflow_b200 import _lib, sharding

    rank, local_rank, world = sharding.env_rank_world()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm"
    assert cfg["streams"] % world == 0, "the 64-stream job must divide over the ranks"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    numa = numa_pin(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    assert lib.cf_device_check() == 0, lib.cf_last_error().decode()

    B = cfg["streams"] // world                       # this rank's streams (stream s lives on rank s % world)
    model = bytes_model(cfg, B)
    hp = HotPath(cfg, B, dev, 1234 + 1000 * 4 + 7 * rank)
    stream = torch.cuda.Stream(dev, priority=-1)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        for d in hp.sets:
            hp.step(d)  # warm: module load, smem opt-in attributes, allocator
        torch.cuda.synchronize()
        # -- step graph: the frame's three independent sub-paths either as parallel graph branches or as one chain.
        #    Branches fill launch ramps and tails when the kernels are short (small per-rank batches); at 64 streams
        #    every kernel fills the machine and the branches only fight over L2 and HBM.  Calibrated here, on set 0:
        #    3 untimed + 10 timed replays of each form, the faster one is THE step (both times are reported).
        def capture_step(d, branched):
            n0 = lib.cf_launch_count()
            g, k = capture(stream, (lambda: hp.step_branched(d, stream)) if branched else (lambda: hp.step(d)))
            return g, k, lib.cf_launch_count() - n0

        cal = {}
        for form in (True, False):
            g, k, _ = capture_step(hp.sets[0], form)
            cal[form] = time_graphs([g], stream, 10, 3)
            del g, k
        torch.cuda.empty_cache()
        branched = cal[True] < 0.98 * cal[False]      # ties go to the chain (run-to-run noise is ~2 %)
        graphs, keep = [], []
        for d in hp.sets:
            g, k, launches_per_step = capture_step(d, branched)
            graphs.append(g)
            keep.append(k)
        sampler = ClockSampler(local_rank) if rank == 0 else None
        step_ms_local = time_graphs(graphs, stream, args.steps, args.warmup, barrier)
        other_form_ms_local = cal[not branched]
        if args.dump_outputs and rank == 0:     # replay i used graphs[i % n]: keep[(steps - 1) % n] holds the last step
            dump_outputs(args.dump_outputs, *keep[(args.steps - 1) % len(keep)])

        # -- e2e: pinned host buffers -> H2D -> public API (the captured graph) -> D2H, every step.  Three streams
        #    (upload / compute / read-back) over the two device buffer sets, so the PCIe transfers of neighbouring
        #    steps overlap (full duplex); every step uploads all of its inputs and reads back all of its results.
        in_keys = ("events", "offsets", "img", "codes", "flow", "fmap1", "fmap2")

        def flat_inputs(d):
            return [d[k] for k in in_keys] + list(d["coords"])

        def flat_outputs(k):
            vox, outs, wi, wz = k
            return [vox, *outs, wi, wz]

        # upload sources: write-combined pinned memory (the GPU only reads it: no cache snooping on the host side);
        # download targets: ordinary pinned memory (the host reads them)
        pinned_in = [pinned_write_combined(t) for t in flat_inputs(hp.sets[0])]
        pinned_out = [[torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in flat_outputs(k)] for k in keep]
        torch.cuda.synchronize()
        h2d = sum(t.numel() * t.element_size() for t in pinned_in)
        d2h = sum(t.numel() * t.element_size() for t in pinned_out[0])
        s_h2d, s_d2h = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        ev_h2d = [torch.cuda.Event() for _ in range(2)]
        ev_comp = [torch.cuda.Event() for _ in range(2)]
        ev_d2h = [torch.cuda.Event() for _ in range(2)]
        n_sets = len(hp.sets)

        def e2e_step(i):
            k = i % n_sets
            if i >= n_sets:
                s_h2d.wait_event(ev_comp[k])      # step i-2 has consumed this input set
            with torch.cuda.stream(s_h2d):
                for dst, src in zip(flat_inputs(hp.sets[k]), pinned_in):
                    dst.copy_(src, non_blocking=True)
                ev_h2d[k].record(s_h2d)
            stream.wait_event(ev_h2d[k])
            if i >= n_sets:
                stream.wait_event(ev_d2h[k])      # step i-2's results have left this output set
            graphs[k].replay()
            ev_comp[k].record(stream)
            s_d2h.wait_event(ev_comp[k])
            with torch.cuda.stream(s_d2h):   # (the read-back split over two streams measured the same 49.5 GB/s)
                for dst, src in zip(pinned_out[k], flat_outputs(keep[k])):
                    dst.copy_(src, non_blocking=True)
                ev_d2h[k].record(s_d2h)

        e2e_steps = args.steps
        for i in range(max(3, n_sets)):
            e2e_step(i)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(s_h2d)
        for i in range(e2e_steps):
            e2e_step(i)
        s_d2h.wait_stream(stream)
        f1.record(s_d2h)
        barrier()
        e2e_ms_local = f0.elapsed_time(f1) / e2e_steps
        clocks = sampler.stop() if sampler else None

        # -- event ingest alone (SURVEY 8f rank 3): host events -> H2D -> voxel grids + normalisation on the device (where
        #    the network consumes them; the reference bins on the host and uploads the grid).  Two host formats: the
        #    reference's fp64 rows (32 B/event) and the packed records (8 B/event, packed by the reader on the host).
        d0 = hp.sets[0]
        packed_host = torch.from_numpy(hp.cf.pack_events_host(d0["events"].cpu().numpy(), d0["offsets"].cpu().numpy()).view(np.int64))
        packed_pin = pinned_write_combined(packed_host.to(dev))
        packed_dev = torch.empty_like(packed_host, device=dev)
        vox_buf = torch.empty_like(keep[0][0])
        ingest = {}
        for label, host_t, dev_t_, fn in (
                ("fp64_rows", pinned_in[0], d0["events"], lambda: hp.voxel(d0, out=vox_buf)),
                ("packed_8B", packed_pin, packed_dev, lambda: hp.cf.events_to_voxel_grid_packed(
                    packed_dev, d0["offsets"], cfg["bins"], cfg["W"], cfg["H"], normalize="std", filter_hot_pixel=True, out=vox_buf))):
            dev_t_.copy_(host_t, non_blocking=True)
            fn()
            torch.cuda.synchronize()
            g_in, _ = capture(stream, fn)
            t0_, t1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 5
            t0_.record(stream)
            for _ in range(reps):
                dev_t_.copy_(host_t, non_blocking=True)
                g_in.replay()
            t1_.record(stream)
            torch.cuda.synchronize()
            ms = t0_.elapsed_time(t1_) / reps
            ingest[label] = {"ms_per_step": ms, "mevents_per_s_per_rank": B * cfg["events"] / (ms * 1e-3) / 1e6,
                             "h2d_bytes_per_step": host_t.numel() * host_t.element_size()}
            del g_in
        del pinned_in, pinned_out, packed_pin, packed_dev, vox_buf

        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peaks = json.load(open(peaks_path))
            hbm, bf16, peak_src = peaks["hbm_gbs"], peaks["bf16_tflops"], "measured (MEASURED_PEAKS.json, burst)"
        else:
            hbm, bf16, peak_src = 6650.0, 1590.0, "fallback (B200_PROFILING.md)"
        tf32_peak = measure_tf32_peak(dev)
        kernels = kernel_times(hp, stream, model, hbm, tf32_peak)

    # -- reduce over ranks (max), gather the per-rank table (the only collective)
    step_ms = sharding.max_over_ranks(step_ms_local, dev)
    e2e_step_ms = sharding.max_over_ranks(e2e_ms_local, dev)
    other_form_ms = sharding.max_over_ranks(other_form_ms_local, dev)
    rows = torch.tensor([[step_ms_local, e2e_ms_local]], dtype=torch.float64, device=dev)
    table = sharding.gather_stream_metrics([rank], rows, world)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return

    # -- single-GPU extras: the other BASELINE configs and the CPU baseline (rank 0 of a 1-GPU run only)
    other, cpu, stock = None, None, None
    if world == 1:
        del graphs, keep, hp
        torch.cuda.empty_cache()
        if not args.no_extra:
            stock = stock_torch_line(cfg, B, dev)
            other = {}
            with torch.cuda.stream(stream):
                for name in ("configs[0]", "configs[1]", "configs[3]"):
                    other[name] = other_config_line(name, dev, stream, hbm, tf32_peak, steps=args.steps)
                other["configs[2]"] = microbench_config2(dev, stream, hbm)
        sample = 4
        host = make_host_streams(cfg, 1234 + 1000 * 4, sample)
        sec, cores, _ = time_cpu(cfg, host, sample, steps=3, warmup=1)
        cpu = {"value": sample / sec, "unit": "frames/s", "cores": cores, "kind": "port", "ms_per_step": sec * 1e3,
               "sample": f"3 steps after 1 warm-up, each the full hot path of {sample} of the 64 streams (480x640, 100000 "
                         f"events, 6 lookups), oracle/ref_port.py (the reference's own NumPy/torch CPU calls), all host threads"}

    share = {k: v["ms_per_launch"] * (cfg["lookups"] if k == "corr_lookup" else 1)
             for k, v in kernels.items() if "noise" not in k}
    dominant = max(share, key=share.get)
    kname = {"corr_build": "corr_tc_kernel", "corr_lookup": "corr_lookup_r4l4_kernel",
             "voxel_bin+normalise": "voxel", "warp_frame_and_codes": "warp_tma_kernel"}[dominant]
    roof = {k: v for k, v in kernels[dominant].items()}
    roof.update({"kernel": kname, "traffic": ncu_traffic(kname), "peak_source": peak_src,
                 "share_of_step": share[dominant] / sum(share.values()),
                 "note": "dominant kernel of the step, timed alone (back-to-back launches inside a CUDA graph over rotating "
                         "buffer sets, CUDA events on the launching stream); traffic = dram read+write bytes of one launch "
                         "from the committed ncu --set full capture of this workload (profiles/r02/)"})
    if "tensor" in roof:
        roof["tensor"]["peak_source"] = "cuBLAS TF32 8192^3 measured in this run (best of 10)"

    frames = B * world
    gbs = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9  # noqa: E731
    line = {
        "metric": "recon_frames_per_s", "value": frames / (step_ms * 1e-3), "unit": "frames/s",
        "metric_note": "frames/s of the motion-compensation hot path (voxel + correlation + lookups + warp per frame); "
                       "no network runs (out of scope, SURVEY 8)",
        "mevents_per_s": frames * cfg["events"] / (step_ms * 1e-3) / 1e6,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
        "step_graph_form": "branched" if branched else "chain",
        "ms_per_step_other_form": other_form_ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 (f64 event time, tf32 correlation)", "data": "synthetic",
        "config": public_config(cfg, world),
        "timing": f"step = 1 CUDA-graph replay of this rank's {B} streams ({int(launches_per_step)} launches); the frame's three "
                  f"independent sub-paths (voxel | pyramid build -> {cfg['lookups']} lookups | warp) run as parallel graph "
                  f"branches or as one chain, whichever a 10-replay calibration on this rank found faster (branches must win by 2 %) (step_graph_form; "
                  f"ms_per_step_other_form = the calibration time of the other form); "
                  f"~{(sum(model[k] for k in ('voxel', 'warp', 'corr_build_bytes')) + cfg['lookups'] * model['lookup']) / 1e6:.0f} MB "
                  f"algorithmic traffic per step and rank",
        "e2e": {"value": frames / (e2e_step_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": e2e_step_ms, "steps": e2e_steps,
                "mevents_per_s": frames * cfg["events"] / (e2e_step_ms * 1e-3) / 1e6,
                "pcie_gbs_per_rank": {"h2d": gbs(h2d, e2e_step_ms), "d2h": gbs(d2h, e2e_step_ms)},
                "numa": numa,
                "path": "pinned host tensors -> H2D (fp64 event rows, feature maps, coords, frame, codes, flow) -> "
                        "cistaflow_b200 public API (captured once as a CUDA graph) -> D2H of voxel grids, all lookup outputs, "
                        "warped frame + codes; upload / compute / read-back on three streams, two device buffer sets; "
                        "bytes are per rank"},
        "ingest_per_rank": {**ingest, "note": "events in pinned host memory -> H2D -> voxel grids + std normalisation left on the "
                            "device (serialised copy + kernel on one stream, rank 0's figures); fp64_rows = the reference's [N,4] float64 "
                            "rows through cf_voxel_bin, packed_8B = host-packed records through cf_voxel_bin_packed"},
        "gpu_launches": int(launches_per_step * args.steps),
        "gpu_launches_per_step": int(launches_per_step),
        "roofline": roof,
        "kernels": kernels,
        "tf32_peak_measured_tflops": tf32_peak,
        "other_configs": other,
        "stock_torch_gpu": stock,
        "cpu_baseline": cpu,
        "clocks": clocks,
        "per_rank_ms": {"step": table[:, 0].tolist(), "e2e_step": table[:, 1].tolist()},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-extra", action="store_true", help="skip the other BASELINE configs (N=1 extras)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    cfg = make_cfg("configs[4]")
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if args.gpus != world and world == 1 and args.gpus > 1:
            # convenience: re-exec under torchrun when called as plain `python bench.py --gpus N`
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__),
                   "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup", str(args.warmup)]
            if args.no_extra:
                cmd.append("--no-extra")
            if args.dump_outputs:
                cmd += ["--dump-outputs", args.dump_outputs]
            sys.exit(subprocess.call(cmd))
        run_ours(args, cfg)


if __name__ == "__main__":
    main()
