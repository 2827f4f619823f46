"""Round-2 parity cases (GPU only): oracle comparisons at the FULL BASELINE sizes (not only properties),
the order-agnostic deterministic walk, and the pieces added this round (fused upflow8 + unpad + warp,
device-side windowing by N events).  Tolerances as in tests/test_gpu_parity.py (BASELINE.json north_star)."""
import numpy as np
import pytest
import torch

import cistaflow_b200 as cf
from cistaflow_b200 import synth
from oracle import explicit, ref_port

from test_gpu_parity import assert_voxel_close, bits, dev_t, last_kernel

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------ voxel ---
@pytest.mark.parametrize("flavour", ["torch", "numpy"])
def test_voxel_deterministic_unsorted_timestamps(cuda_device, flavour):
    """The reference's scatter-adds do not depend on the stamps being sorted; the deterministic mode must not either
    (round-1 ADVICE: the per-pixel walk assumed non-decreasing bins and silently dropped events).  Stamps are
    shuffled inside each window, first/last rows kept (they define t0 and dT), so every t* stays in [0, nb-1]."""
    h, w, n, batch = 48, 64, 6000, 3
    ev, off = synth.event_windows(batch, n, h, w, seed=123)
    rng = np.random.default_rng(5)
    for b in range(batch):
        s, e = off[b] + 1, off[b + 1] - 1
        ev[s:e, 0] = ev[s:e, 0][rng.permutation(e - s)]
    fl = explicit.FLAVOUR_TORCH if flavour == "torch" else explicit.FLAVOUR_NUMPY
    ref = np.stack([explicit.voxel_grid_sequential(ev[off[b]:off[b + 1]], 5, w, h, fl) for b in range(batch)])
    ev_d, off_d = dev_t(ev, cuda_device), dev_t(off, cuda_device)
    det = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, w, h, flavour=flavour, mode="deterministic").cpu().numpy()
    assert np.array_equal(bits(det), bits(ref))
    pos = ev.copy()
    pos[:, 3] = 1.0
    mag = np.stack([explicit.voxel_grid_sequential(pos[off[b]:off[b + 1]], 5, w, h, fl) for b in range(batch)])
    atom = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, w, h, flavour=flavour, mode="atomic").cpu().numpy()
    assert_voxel_close(atom, ref, mag)


def test_voxel_mvsec_deterministic_unsorted_timestamps(cuda_device):
    """Same for the second voxeliser (one index_put_ per bin: left and right weights interleave in event order)."""
    h, w, n = 40, 56, 5000
    ev = synth.events(n, h, w, seed=321)
    rng = np.random.default_rng(6)
    ev[1:-1, 0] = ev[1:-1, 0][rng.permutation(n - 2)]
    ev[:, 3] = np.where(ev[:, 3] == 0, -1.0, 1.0)
    xytp = ev[:, [1, 2, 0, 3]]
    ref = ref_port.mvsec_voxel_torch(torch.from_numpy(xytp[:, 0]), torch.from_numpy(xytp[:, 1]), torch.from_numpy(xytp[:, 2]),
                                     torch.from_numpy(xytp[:, 3]), 5, h, w).numpy()
    off = torch.tensor([0, n], dtype=torch.int64, device=cuda_device)
    got = cf.events_to_voxel_grid_batched(dev_t(ev, cuda_device), off, 5, w, h, flavour="mvsec", mode="deterministic")[0]
    assert np.array_equal(bits(got.cpu().numpy()), bits(ref))


def test_voxel_full_size_vs_sequential_oracle(cuda_device, parity_report):
    """configs[3] at full size: 1 M events at 624x970 against the plain-C sequential oracle -- deterministic mode
    bit-exact (both flavours), atomic mode within tolerance, fused normalisation against the explicit oracle."""
    n, h, w = 1_000_000, 624, 970
    ev = synth.events(n, h, w, seed=synth.seed_for(3))
    ev_d = dev_t(ev, cuda_device)
    off = torch.tensor([0, n], dtype=torch.int64, device=cuda_device)
    pos = ev.copy()
    pos[:, 3] = 1.0
    for flavour, fl in (("torch", explicit.FLAVOUR_TORCH), ("numpy", explicit.FLAVOUR_NUMPY)):
        ref = explicit.voxel_grid_sequential(ev, 5, w, h, fl)
        mag = explicit.voxel_grid_sequential(pos, 5, w, h, fl)
        det = cf.events_to_voxel_grid_batched(ev_d, off, 5, w, h, flavour=flavour, mode="deterministic")[0].cpu().numpy()
        assert np.array_equal(bits(det), bits(ref)), flavour
        atom = cf.events_to_voxel_grid_batched(ev_d, off, 5, w, h, flavour=flavour, mode="atomic")[0].cpu().numpy()
        frac = assert_voxel_close(atom, ref, mag)
        parity_report.add("voxel_full_size_624x970_1M", flavour=flavour, deterministic_bit_exact=True,
                          atomic_fraction_within_literal_tol=frac, atomic_max_abs_err=float(np.abs(atom - ref).max()))
    thr = 25.0 / 5
    fused = cf.events_to_voxel_grid_batched(ev_d, off, 5, w, h, normalize="std", filter_hot_pixel=True, flavour="numpy",
                                            mode="atomic")[0].cpu().numpy()
    np.testing.assert_allclose(fused, explicit.preprocess(ref, "std", thr), rtol=1e-4, atol=1e-4)


# ------------------------------------------------------------------- warp ---
@pytest.mark.parametrize("h,w", [(480, 640), (624, 970)])
@pytest.mark.parametrize("flow_kind", ["smooth", "noise"])
def test_warp_codes_full_size_vs_oracle(cuda_device, parity_report, h, w, flow_kind):
    """configs[3]/[4] at full size with the model's 128 code channels: frame [1,1,H,W] + codes [1,128,H/2,W/2]
    against the reference's grid_sample path (oracle port) -- |err| <= 1e-4 on every element."""
    img, codes, flow = synth.warp_inputs(1, h, w, seed=17, code_channels=128, flow_kind=flow_kind)
    ri, rz = ref_port.warp_frame_and_codes(torch.from_numpy(img), torch.from_numpy(codes), torch.from_numpy(flow), "forward")
    wi, wz = cf.warp_frame_and_codes(dev_t(img, cuda_device), dev_t(codes, cuda_device), dev_t(flow, cuda_device), "forward")
    ei, ez = (wi.cpu() - ri).abs(), (wz.cpu() - rz).abs()
    parity_report.add("warp_full_size", H=h, W=w, flow_kind=flow_kind, max_err_frame=ei.max().item(), max_err_codes=ez.max().item(),
                      fraction_within_tol=float(((ez <= 1e-4).float().mean() + (ei <= 1e-4).float().mean()) / 2))
    assert ei.max().item() <= 1e-4 and ez.max().item() <= 1e-4
    bi, bz = ref_port.warp_frame_and_codes(torch.from_numpy(img), torch.from_numpy(codes), torch.from_numpy(flow), "backward")
    vi, vz = cf.warp_frame_and_codes(dev_t(img, cuda_device), dev_t(codes, cuda_device), dev_t(flow, cuda_device), "backward")
    assert (vi.cpu() - bi).abs().max().item() <= 1e-4 and (vz.cpu() - bz).abs().max().item() <= 1e-4


# ------------------------------------------------------- batched, 64 streams ---
def test_voxel_64_streams_480x640_vs_oracle(cuda_device, parity_report):
    """The bench's own voxel launch (64 windows of 100 000 events at 480x640, fused std normalisation, hot-pixel
    filter): 4 distinct windows tiled to 64 like bench.py; every window against the sequential oracle + preprocess."""
    h, w, n, B = 480, 640, 100000, 64
    ev4, off4 = synth.event_windows(4, n, h, w, seed=4321)
    ev = np.concatenate([ev4] * (B // 4))
    off = np.arange(B + 1, dtype=np.int64) * n
    raw = cf.events_to_voxel_grid_batched(dev_t(ev, cuda_device), dev_t(off, cuda_device), 5, w, h, flavour="numpy",
                                          mode="atomic").cpu().numpy()
    fused = cf.events_to_voxel_grid_batched(dev_t(ev, cuda_device), dev_t(off, cuda_device), 5, w, h, normalize="std",
                                            filter_hot_pixel=True, flavour="numpy", mode="atomic").cpu().numpy()
    fr = []
    for b in range(4):
        win = ev4[off4[b]:off4[b + 1]]
        ref = explicit.voxel_grid_sequential(win, 5, w, h, explicit.FLAVOUR_NUMPY)
        pos = win.copy()
        pos[:, 3] = 1.0
        mag = explicit.voxel_grid_sequential(pos, 5, w, h, explicit.FLAVOUR_NUMPY)
        ref_n = explicit.preprocess(ref, "std", 5.0)
        for k in range(b, B, 4):
            fr.append(assert_voxel_close(raw[k], ref, mag))
            np.testing.assert_allclose(fused[k], ref_n, rtol=1e-4, atol=1e-4)
    parity_report.add("voxel_64x480x640_bench_launch", windows=B, min_fraction_within_literal_tol=min(fr))


# ------------------------------------------------ multi-frame model traces ---
@pytest.mark.parametrize("trace", ["trace3_eiflow", "trace3_eraft"])
def test_multi_frame_trace_replay(golden, cuda_device, parity_report, trace):
    """Three CONSECUTIVE recurrent frames (4th-6th) of the default-size reference models (180x240, base_channels 64,
    tests/golden/make_golden.py make_trace_multi): every frame's hot-path calls replayed through the CUDA path on the
    tensors the reference model actually produced, against the reference's own outputs."""
    from test_oracle_golden import trace3_events
    from test_gpu_parity import corr_err
    g = golden(trace)
    H, W, nev, frames, dsub, csub = (int(v) for v in g["meta"])
    frame_warp = cf.FrameWarp("forward")
    worst = {"lookup": 0.0, "warp": 0.0, "voxel": 0.0}
    for f in range(frames):
        n_lookup, n_warp = (int(v) for v in g[f"f{f}/counts"])
        ev = trace3_events(g, f)
        ref_grid = explicit.voxel_grid_sequential(ev, 5, W, H, explicit.FLAVOUR_NUMPY)
        grid = cf.events_to_voxel_grid(ev, 5, W, H, mode="deterministic")
        assert np.array_equal(bits(grid), bits(ref_grid))
        ref_norm = ref_port.preprocess_numpy(ref_grid, "std", True)
        fused = cf.events_to_voxel_grid_batched(dev_t(ev, cuda_device), torch.tensor([0, len(ev)], device=cuda_device), 5, W, H,
                                                normalize="std", filter_hot_pixel=True, flavour="numpy", mode="atomic")[0]
        worst["voxel"] = max(worst["voxel"], float(np.abs(fused.cpu().numpy() - ref_norm).max()))
        np.testing.assert_allclose(fused.cpu().numpy(), ref_norm, rtol=1e-4, atol=1e-4)
        blk = cf.CorrBlock(dev_t(g[f"f{f}/fmap1"], cuda_device), dev_t(g[f"f{f}/fmap2"], cuda_device), num_levels=4, radius=4)
        out = blk(dev_t(g[f"f{f}/coords{n_lookup - 1}"], cuda_device))
        e = corr_err(*g.pick(f"f{f}/lookup_last", out[:, ::4].cpu().numpy()))
        worst["lookup"] = max(worst["lookup"], e)
        assert e <= 1e-3
        flow = dev_t(g[f"f{f}/flow_final"], cuda_device)
        wi, wz = cf.warp_frame_and_codes(dev_t(g[f"f{f}/warp0_in"], cuda_device), dev_t(g[f"f{f}/warp1_in"], cuda_device), flow, "forward")
        ei = float(np.abs(np.subtract(*g.pick(f"f{f}/warp0_out", wi.cpu().numpy()))).max())
        ez = float(np.abs(np.subtract(*g.pick(f"f{f}/warp1_out", wz.cpu().numpy()))).max())
        worst["warp"] = max(worst["warp"], ei, ez)
        assert ei <= 1e-4 and ez <= 1e-4
        sep = frame_warp.warp_frame(dev_t(g[f"f{f}/warp0_in"], cuda_device), flow)
        np.testing.assert_allclose(*g.pick(f"f{f}/warp0_out", sep.cpu().numpy()), rtol=0, atol=1e-4)
    parity_report.add("multi_frame_trace_replay", trace=trace, frames=frames, max_lookup_err_over_max=worst["lookup"],
                      max_warp_abs_err=worst["warp"], max_fused_voxel_abs_err=worst["voxel"])


# ------------------------------------------------ fused upflow8 + unpad + warp ---
def test_upflow8_unpad_warp_golden(golden, cuda_device):
    """One launch for upflow8 + ImagePadder.unpad + frame warp + x0.5 flow + codes warp, against the reference's own
    outputs (tests/golden/warp.npz up8/*: DCEIFlow/utils/sample_utils.py:66-68, utils/image_process.py:103-107)."""
    g = golden("warp")
    pad = tuple(int(v) for v in g["up8/pad"])
    n0 = cf.load_library().cf_launch_count()
    wi, wz, flow = cf.warp_frame_and_codes_upflow8(dev_t(g["step/img"], cuda_device), dev_t(g["step/codes"], cuda_device),
                                                   dev_t(g["up8/flow_lr"], cuda_device), "forward", pad=pad)
    assert cf.load_library().cf_launch_count() - n0 == 1
    np.testing.assert_allclose(flow.cpu().numpy(), g["up8/flow_final"], rtol=0, atol=1e-5)
    np.testing.assert_allclose(wi.cpu().numpy(), g["up8/img_warped"], rtol=0, atol=1e-4)
    np.testing.assert_allclose(wz.cpu().numpy(), g["up8/codes_warped"], rtol=0, atol=1e-4)


@pytest.mark.parametrize("h,w,batch,channels", [(180, 240, 2, 128), (260, 346, 1, 128), (480, 640, 1, 128), (36, 44, 3, 6)])
@pytest.mark.parametrize("mode", ["forward", "backward"])
def test_upflow8_unpad_warp_vs_oracle(cuda_device, h, w, batch, channels, mode):
    """Config shapes (x32 padding on the top/left like ImagePadder): staged (TMA) and direct kernels, both warp modes."""
    img, codes, _ = synth.warp_inputs(batch, h, w, seed=31, code_channels=channels, flow_kind="smooth")
    hp, wp = synth.padded_dims(h, w)
    pad = (hp - h, wp - w)
    rng = np.random.default_rng(32)
    lr = synth.smooth_field(rng, batch, 2, hp // 8, wp // 8, 0.35, cell=4)      # x8 -> a few px, like the model's flow
    ri, rz, rf = ref_port.warp_frame_and_codes_upflow8(torch.from_numpy(img), torch.from_numpy(codes), torch.from_numpy(lr),
                                                       pad[0], pad[1], mode)
    wi, wz, wf = cf.warp_frame_and_codes_upflow8(dev_t(img, cuda_device), dev_t(codes, cuda_device), dev_t(lr, cuda_device),
                                                 mode, pad=pad)
    assert (wf.cpu() - rf).abs().max().item() <= 1e-5
    assert (wi.cpu() - ri).abs().max().item() <= 1e-4 and (wz.cpu() - rz).abs().max().item() <= 1e-4
    # ... and identical to the unfused calls on the up-sampled flow
    ui, uz = cf.warp_frame_and_codes(dev_t(img, cuda_device), dev_t(codes, cuda_device), wf, mode)
    assert (ui - wi).abs().max().item() <= 1e-6 and (uz - wz).abs().max().item() <= 1e-6
    with pytest.raises(ValueError):
        cf.warp_frame_and_codes_upflow8(dev_t(img, cuda_device), dev_t(codes, cuda_device), dev_t(lr, cuda_device), mode,
                                        pad=(pad[0] + 8, pad[1]))


# ------------------------------------------------------- device-side windowing ---
@pytest.mark.parametrize("n,limit", [(100000, 30000), (100001, 33334), (5, 30000), (0, 1000), (45000, 30000), (75000, 30000)])
def test_device_windowing_matches_the_reference_reader(cuda_device, n, limit):
    """video_readers.py:208-232 on the device: the x < W / y < H filter (stable compaction), np.array_split into
    round(n / limit) windows (round-half-even), then the voxel grids of those windows -- against the same steps in NumPy
    + the sequential oracle.  No read-back between the steps."""
    h, w = 60, 80
    ev = synth.events(n, h, w, seed=55) if n else np.zeros((0, 4))
    if n:
        rng = np.random.default_rng(2)
        bad = rng.random(n) < 0.03                      # sensor rows the reader drops: x == W, y >= H
        ev[bad, 1] = np.where(rng.random(bad.sum()) < 0.5, w, ev[bad, 1])
        ev[bad, 2] = np.where(ev[bad, 1] < w, h + 1, ev[bad, 2])
    ref = ev[ev[:, 1] < w]
    ref = ref[ref[:, 2] < h]
    k = round(ref.shape[0] / limit) or 1
    parts = np.array_split(ref, k, axis=0)
    out, kept = cf.filter_events(dev_t(ev, cuda_device), w, h)
    max_windows = 8
    offs, n_win = cf.window_offsets(kept, limit, max_windows, policy="split")
    assert kept.item() == ref.shape[0] and n_win.item() == min(k, max_windows)
    assert np.array_equal(out[: ref.shape[0]].cpu().numpy(), ref)
    sizes = np.diff(offs.cpu().numpy())
    assert list(sizes[:k]) == [len(p) for p in parts] and (sizes[k:] == 0).all()
    grids = cf.events_to_voxel_grid_batched(out, offs, 5, w, h, flavour="numpy", mode="deterministic").cpu().numpy()
    for i, part in enumerate(parts):
        if len(part):
            assert np.array_equal(bits(grids[i]), bits(explicit.voxel_grid_sequential(part, 5, w, h, explicit.FLAVOUR_NUMPY)))
    assert not grids[k:].any()
    # fixed-size windows (FixedSizeEventReader): the last window keeps the remainder
    offs_f, n_f = cf.window_offsets(kept, 30000, max_windows, policy="fixed")
    m = ref.shape[0]
    want = [min(i * 30000, m) for i in range(max_windows + 1)]
    assert offs_f.cpu().tolist() == want and n_f.item() == -(-m // 30000)


def test_out_of_grid_events_are_dropped_where_the_reference_wraps(cuda_device):
    """Round-1 ADVICE: the exact divergence on unfiltered input.  An event with x == W: the reference's NumPy voxeliser
    wraps it onto column 0 of the next row (flat index x + y*W + ti*W*H, utils/event_process.py:61-66); this library
    drops it -- i.e. equals the reference on the reader-filtered stream (video_readers.py:208-209)."""
    h, w = 24, 32
    ev = synth.events(3000, h, w, seed=9)
    ev[100:140, 1] = w                                # x == W, rows 100..139 (never the first / last row: t0, dT unchanged)
    ev[100:140, 2] = np.minimum(ev[100:140, 2], h - 2)
    ev[100:140, 3] = 1.0
    kept = ev[ev[:, 1] < w]
    ours = cf.events_to_voxel_grid(ev, 5, w, h, mode="deterministic")
    assert np.array_equal(bits(ours), bits(ref_port.voxel_grid_numpy(kept, 5, w, h)))
    wrapped = ref_port.voxel_grid_numpy(ev, 5, w, h)  # what the reference returns on the unfiltered stream
    assert not np.array_equal(wrapped, ours)
    assert abs(float(wrapped.sum()) - float(ours.sum())) > 1.0   # the wrapped events' polarity mass is in the reference grid only


@pytest.mark.parametrize("mode", ["atomic", "atomic_l2"])
def test_voxel_l2_path_over_several_chunks(cuda_device, mode):
    """The L2-atomic path splits the batch into chunks of windows whose grids and events fit a 96 MB L2 budget, and the
    statistics of a chunk go to its own slice of the workspace.  80 windows at 180x240 need two chunks: every window
    against the sequential oracle, raw and with fused normalisation, with empty and ragged windows on both sides of
    each flavour's chunk boundary."""
    h, w, nb, B = 180, 240, 5, 80
    specials = [0, 4099, 0, 3]                                   # per boundary: windows c-2, c-1 | c, c+1
    counts = [15000] * (B - 2 * len(specials)) + 2 * specials
    total = sum(counts)
    bounds = {}
    for flavour, planes in (("numpy", 1), ("pol", 2)):
        per_window = nb * planes * h * w * 4 + (total // B + 1) * 32   # bytes per window of the chunk budget
        chunk = (96 << 20) // per_window
        assert -(-B // chunk) >= 2, (flavour, chunk)
        bounds[flavour] = chunk
    assert abs(bounds["numpy"] - bounds["pol"]) >= 2 * len(specials) and max(bounds.values()) + 2 <= B
    special_at = {c + k: n for c in bounds.values() for k, n in zip((-2, -1, 0, 1), specials)}
    counts = [special_at.get(i, 15000) for i in range(B)]
    assert sum(counts) == total
    wins = [synth.events(n, h, w, seed=900 + i) if n else np.zeros((0, 4)) for i, n in enumerate(counts)]
    ev = np.concatenate(wins, axis=0)
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    ev_d, off_d = dev_t(ev, cuda_device), dev_t(off, cuda_device)
    for flavour, fl in (("numpy", explicit.FLAVOUR_NUMPY), ("pol", explicit.FLAVOUR_POL)):
        raw = cf.events_to_voxel_grid_batched(ev_d, off_d, nb, w, h, flavour=flavour, mode=mode).cpu().numpy()
        assert last_kernel() == "voxel_scatter_atomic_kernel"
        fused = {}
        for norm in ("std", "maxmin"):
            fused[norm] = cf.events_to_voxel_grid_batched(ev_d, off_d, nb, w, h, normalize=norm, filter_hot_pixel=True,
                                                          flavour=flavour, mode=mode).cpu().numpy()
            assert last_kernel() == "voxel_normalise_kernel"
        for b, win in enumerate(wins):
            ref = explicit.voxel_grid_sequential(win, nb, w, h, fl)
            mag = None
            if flavour == "numpy":                                # the pol grid holds positive weights: |ref| is M
                pos = win.copy()
                pos[:, 3] = 1.0
                mag = explicit.voxel_grid_sequential(pos, nb, w, h, fl)
            assert_voxel_close(raw[b], ref, mag)
            for norm, got in fused.items():
                np.testing.assert_allclose(got[b], explicit.preprocess(ref, norm, 25.0 / nb), rtol=1e-4, atol=1e-4)


# ------------------------------------------------- experiment paths stay correct ---
def _run_with_env(code, env_extra):
    import os
    import subprocess
    import sys
    env = dict(os.environ, **env_extra)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=env,
                         cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    return res


def test_corr_two_pass_conversion_and_lsu_stores_subprocess(cuda_device):
    """CF_TC_FLAGS bit16 (two-pass fp16 conversion) and bit5 (fp16 kernel: level-0 rows through the LSU): experiment paths of
    the fp16-operand pyramid build, against the fp32 SIMT kernel."""
    code = """
import torch
import cistaflow_b200 as cf
from cistaflow_b200 import synth
dev = torch.device('cuda', 0)
for (H, W, B) in ((480, 640, 2), (192, 256, 2), (512, 512, 2)):
    f1, f2, _ = synth.corr_inputs(B, H, W, 6)
    a, b = torch.from_numpy(f1).to(dev), torch.from_numpy(f2).to(dev)
    ref = cf.build_pyramid(a, b, 4, precision='fp32')
    got = cf.build_pyramid(a, b, 4, precision='f16')
    for l in range(4):
        err = (got[l] - ref[l]).abs().max().item() / ref[l].abs().max().item()
        assert err <= 1e-3, (H, W, l, err)
print('F16_OK')
"""
    # bit17: the fmap2 slice in 128-byte-swizzled boxes (the default where tiles are 160 columns wide is the 64-byte swizzle);
    # bit19: one level-0 store box per lane quarter and tile
    # bit25: level 3 pooled in the epilogue out of quads of tiles (tile indices padded to groups of four)
    # bit26: level 0 straight from registers in the tcgen05.ld.16x256b fragment layout (no staging, no TMA store)
    for flags in ("65536", "32", "128", str(1 << 17), str(1 << 19), str(1 << 25), str(1 << 26)):
        res = _run_with_env(code, {"CF_TC_FLAGS": flags})
        assert res.returncode == 0 and "F16_OK" in res.stdout, flags + res.stdout + res.stderr
