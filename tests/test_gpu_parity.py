"""Parity of the CUDA path (libcistaflow.so through the Python mirror) with the
oracle and with the reference-generated golden fixtures.  GPU only.

Tolerances (BASELINE.json north_star):
  voxel   bit-exact in deterministic mode; |err| <= 1e-5*(|ref|+1) in atomic mode
  warp    |err| <= 1e-4 absolute
  corr    1e-3 relative, measured normwise: max|err| <= 1e-3 * max|ref|
          (element-wise relative error is meaningless for near-zero correlations,
          SURVEY.md H3); the fp32 SIMT path is held to 1e-5 * max|ref|
  lookup  on an identical pyramid: |err| <= 1e-4 * max|ref| (same gather, fp32)
"""
import numpy as np
import pytest
import torch

import cistaflow_b200 as cf
from cistaflow_b200 import synth
from oracle import explicit, ref_port

pytestmark = pytest.mark.gpu


def dev_t(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_voxel_close(got, ref, mag=None):
    """Atomic mode: |err| <= 1e-5 * (M + 1) per cell.  M = sum of |weights| accumulated in the cell when the
    caller can supply it (the polarity-split grid holds exactly that), else |ref|.  fp32 sums taken in a
    different order differ by ~sqrt(n) ulp of the PARTIAL sums, so for a cell where +/- events cancel the
    error is relative to the magnitudes added, not to the (near-zero) result: with M = |ref| the atomic
    tests failed about one run in ten on the dense hot-pixel fixture (2.3e-5 on a cancelling cell)."""
    err = np.abs(got.astype(np.float64) - ref.astype(np.float64))
    m = np.abs(ref.astype(np.float64)) if mag is None else np.maximum(mag.astype(np.float64), np.abs(ref.astype(np.float64)))
    tol = 1e-5 * (m + 1.0)
    assert (err <= tol).all(), f"max err {err.max():.3e}"
    # ... and to the letter of north_star: the fraction of cells inside 1e-5 * (|ref| + 1) must be >= 95 %
    frac = float((err <= 1e-5 * (np.abs(ref.astype(np.float64)) + 1.0)).mean()) if err.size else 1.0
    assert frac >= 0.95, f"only {frac:.4f} of the cells within 1e-5*(|ref|+1)"
    VOXEL_FRACTIONS.append(frac)
    return frac


VOXEL_FRACTIONS = []   # literal-tolerance agreement of every atomic-mode comparison of this session


# ------------------------------------------------------------------ voxel ---
VOXEL_CASES = ["base", "dense_hot", "single", "two_same_t", "empty"]


@pytest.mark.parametrize("case", VOXEL_CASES)
def test_voxel_golden_deterministic_bit_exact(golden, cuda_device, case):
    g = golden("voxel")
    ev = g[f"{case}/events"]
    nb, w, h = (int(v) for v in g[f"{case}/dims"])
    got_t = cf.events_to_voxel_grid_pytorch(dev_t(ev, cuda_device), nb, w, h, mode="deterministic")
    assert got_t.device.type == "cuda" and got_t.dtype == torch.float32 and got_t.shape == (nb, h, w)
    assert np.array_equal(bits(got_t.cpu().numpy()), bits(g[f"{case}/torch"]))
    got_n = cf.events_to_voxel_grid(ev.copy(), nb, w, h, mode="deterministic")
    assert isinstance(got_n, np.ndarray) and got_n.dtype == np.float32
    assert np.array_equal(bits(got_n), bits(g[f"{case}/numpy"]))
    got_p = cf.events_to_voxel_grid_pol(ev.copy(), nb, w, h, mode="deterministic")
    assert got_p.shape == (nb, 2, h, w)
    assert np.array_equal(bits(got_p), bits(g[f"{case}/pol"]))


@pytest.mark.parametrize("case", VOXEL_CASES)
def test_voxel_golden_atomic(golden, cuda_device, case):
    g = golden("voxel")
    ev = g[f"{case}/events"]
    nb, w, h = (int(v) for v in g[f"{case}/dims"])
    keep = ev.copy()
    mag = g[f"{case}/pol"].sum(axis=1)   # sum of |weights| per cell
    assert_voxel_close(cf.events_to_voxel_grid(ev, nb, w, h, mode="atomic"), g[f"{case}/numpy"], mag)
    assert np.array_equal(ev, keep), "inputs must not be mutated"
    assert_voxel_close(cf.events_to_voxel_grid_pytorch(dev_t(ev, cuda_device), nb, w, h, mode="atomic").cpu().numpy(),
                       g[f"{case}/torch"], mag)
    assert_voxel_close(cf.events_to_voxel_grid_pol(ev, nb, w, h, mode="atomic"), g[f"{case}/pol"])


def test_voxel_cpu_tensor_round_trips_to_cpu(golden, cuda_device):
    g = golden("voxel")
    ev = torch.from_numpy(g["base/events"].copy())
    out = cf.events_to_voxel_grid_pytorch(ev, 5, 40, 30, mode="deterministic")
    assert out.device.type == "cpu"
    assert np.array_equal(bits(out.numpy()), bits(g["base/torch"]))


@pytest.mark.parametrize("case", ["base", "dense_hot", "empty"])
@pytest.mark.parametrize("mode", ["std", "maxmin"])
@pytest.mark.parametrize("hot", [False, True])
def test_preprocess_golden(golden, cuda_device, case, mode, hot):
    g = golden("voxel")
    got = cf.event_preprocess(g[f"{case}/numpy"].copy(), mode, hot)
    assert got.dtype == np.float32
    np.testing.assert_allclose(got, g[f"{case}/pre_numpy_{mode}_{int(hot)}"], rtol=1e-5, atol=1e-5)
    got_t = cf.event_preprocess_pytorch(dev_t(g[f"{case}/torch"], cuda_device), mode, hot)
    np.testing.assert_allclose(got_t.cpu().numpy(), g[f"{case}/pre_torch_{mode}_{int(hot)}"], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("n,h,w,batch", [(15000, 180, 240, 3), (50000, 260, 346, 2), (4097, 33, 47, 5)])
@pytest.mark.parametrize("flavour", ["torch", "numpy"])
def test_voxel_batched_vs_sequential_oracle(cuda_device, n, h, w, batch, flavour):
    """Config-size windows: deterministic mode bit-exact vs the plain-C sequential
    oracle; atomic mode within 1e-5; fused normalisation vs the explicit oracle."""
    ev, off = synth.event_windows(batch, n, h, w, seed=77)
    ev[off[1] + 10:off[1] + 15, 1:3] = [[-1, 0], [w, 0], [0, h], [0, -2], [w + 5, h + 5]]  # out of grid -> dropped
    ev_d, off_d = dev_t(ev, cuda_device), dev_t(off, cuda_device)
    fl = explicit.FLAVOUR_TORCH if flavour == "torch" else explicit.FLAVOUR_NUMPY
    ref, mag = [], []
    for b in range(batch):
        win = ev[off[b]:off[b + 1]]
        ok = (win[:, 1] >= 0) & (win[:, 1] < w) & (win[:, 2] >= 0) & (win[:, 2] < h)
        assert ok[0] and ok[-1]  # t0 / dT come from the window's first/last row: keep them in-grid
        ref.append(explicit.voxel_grid_sequential(win[ok], 5, w, h, fl))
        pos = win[ok].copy()
        pos[:, 3] = 1.0
        mag.append(explicit.voxel_grid_sequential(pos, 5, w, h, fl))   # sum of |weights| per cell
    ref, mag = np.stack(ref), np.stack(mag)
    det = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, w, h, flavour=flavour, mode="deterministic").cpu().numpy()
    assert np.array_equal(bits(det), bits(ref))
    det2 = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, w, h, flavour=flavour, mode="deterministic").cpu().numpy()
    assert np.array_equal(bits(det), bits(det2)), "deterministic mode must be run-to-run identical"
    for path, kernel in (("atomic_l2", ("voxel_scatter_atomic_kernel",)), ("atomic_tiled", ("voxel_tile_kernel",)),
                         ("atomic", None)):
        atom = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, w, h, flavour=flavour, mode=path).cpu().numpy()
        assert kernel is None or last_kernel() in kernel
        assert_voxel_close(atom, ref, mag)
        # ... and with the statistics + normalisation fused
        for norm in ("std", "maxmin"):
            thr_ = (20.0 if flavour == "torch" else 25.0) / 5
            fz = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, w, h, normalize=norm, filter_hot_pixel=True,
                                                 flavour=flavour, mode=path).cpu().numpy()
            for b in range(batch):
                np.testing.assert_allclose(fz[b], explicit.preprocess(ref[b], norm, thr_), rtol=1e-4, atol=1e-4)
    # fused std normalisation + hot-pixel filter
    thr = (20.0 if flavour == "torch" else 25.0) / 5
    fused = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, w, h, normalize="std", filter_hot_pixel=True,
                                            flavour=flavour, mode="deterministic").cpu().numpy()
    for b in range(batch):
        np.testing.assert_allclose(fused[b], explicit.preprocess(ref[b], "std", thr), rtol=1e-5, atol=1e-5)


def last_kernel():
    from cistaflow_b200 import _lib
    return _lib.load().cf_last_kernel().decode()


@pytest.mark.parametrize("h,w,counts", [
    (180, 240, [15000, 0, 7000, 15000, 1, 4096, 8192, 3, 15000, 0, 15000, 15000]),   # empty / tiny / chunk-sized windows
    (480, 640, [30000] * 11),                                                        # 3 waves of 4 windows (37 tiles each)
    (624, 970, [200000]),                                                            # one window over all 148 SMs
    (31, 45, [5000, 300]),                                                           # H*W % 4 != 0: scalar stores
])
@pytest.mark.parametrize("path", ["atomic_tiled", "atomic_l2"])
def test_voxel_atomic_paths_ragged_batches(cuda_device, h, w, counts, path):
    """Both data paths of the atomic mode (partition + shared-memory tiles; L2 atomics) on ragged batches: every window against the plain-C
    sequential oracle (atomic tolerance), raw and with fused std normalisation; polarity flavour too."""
    wins = [synth.events(n, h, w, seed=300 + i) if n else np.zeros((0, 4)) for i, n in enumerate(counts)]
    ev = np.concatenate(wins, axis=0)
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    ev_d, off_d = dev_t(ev, cuda_device), dev_t(off, cuda_device)
    raw = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, w, h, flavour="numpy", mode=path).cpu().numpy()
    assert last_kernel() in (("voxel_tile_kernel",) if path == "atomic_tiled" else ("voxel_scatter_atomic_kernel",))
    fused = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, w, h, normalize="std", filter_hot_pixel=True,
                                            flavour="numpy", mode=path).cpu().numpy()
    pol = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, w, h, flavour="pol", mode=path).cpu().numpy()
    for b, win in enumerate(wins):
        if len(win) == 0:
            assert not raw[b].any() and not fused[b].any() and not pol[b].any()
            continue
        ref = explicit.voxel_grid_sequential(win, 5, w, h, explicit.FLAVOUR_NUMPY)
        pos = win.copy()
        pos[:, 3] = 1.0
        mag = explicit.voxel_grid_sequential(pos, 5, w, h, explicit.FLAVOUR_NUMPY)
        assert_voxel_close(raw[b], ref, mag)
        np.testing.assert_allclose(fused[b], explicit.preprocess(ref, "std", 5.0), rtol=1e-4, atol=1e-4)
        assert_voxel_close(pol[b].sum(axis=1), mag, mag)               # |w| of both polarities = magnitude grid
        assert_voxel_close(pol[b][:, 1] - pol[b][:, 0], ref, mag)       # signed recombination = plain grid


@pytest.mark.parametrize("h,w,counts", [(180, 240, [15000, 0, 7000, 1, 15000]), (480, 640, [100000, 60000])])
def test_voxel_packed_events(cuda_device, h, w, counts):
    """Packed 8-byte events (SURVEY 8f rank 3): host and device packers agree bit for bit; the packed voxel kernel
    stays within the atomic-mode tolerance of the fp64 oracle, raw and with fused normalisation."""
    wins = [synth.events(n, h, w, seed=500 + i) if n else np.zeros((0, 4)) for i, n in enumerate(counts)]
    ev = np.concatenate(wins, axis=0)
    ev[7, 1:3] = [-3.0, 5.0]          # out of grid -> dropped by both paths
    wins[0][7, 1:3] = [-3.0, 5.0]
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    host = cf.pack_events_host(ev, off)
    ev_d, off_d = dev_t(ev, cuda_device), dev_t(off, cuda_device)
    packed = cf.pack_events(ev_d, off_d)
    assert last_kernel() == "events_pack_kernel"
    assert np.array_equal(packed.cpu().numpy().view(np.uint64), host)
    up = torch.from_numpy(host.view(np.int64)).to(cuda_device)       # the ingest path: pack on the host, upload 8 B/event
    raw = cf.events_to_voxel_grid_packed(up, off_d, 5, w, h).cpu().numpy()
    assert last_kernel() == "voxel_scatter_packed_kernel"
    fused = cf.events_to_voxel_grid_packed(up, off_d, 5, w, h, normalize="std", filter_hot_pixel=True).cpu().numpy()
    for b, win in enumerate(wins):
        if len(win) == 0:
            assert not raw[b].any() and not fused[b].any()
            continue
        ok = (win[:, 1] >= 0) & (win[:, 1] < w) & (win[:, 2] >= 0) & (win[:, 2] < h)
        ref = explicit.voxel_grid_sequential(win[ok], 5, w, h, explicit.FLAVOUR_NUMPY)
        pos = win[ok].copy()
        pos[:, 3] = 1.0
        mag = explicit.voxel_grid_sequential(pos, 5, w, h, explicit.FLAVOUR_NUMPY)
        assert_voxel_close(raw[b], ref, mag)
        np.testing.assert_allclose(fused[b], explicit.preprocess(ref, "std", 5.0), rtol=1e-4, atol=1e-4)


def test_voxel_is_reverse(cuda_device):
    ev = synth.events(2000, 20, 24, 5)
    got = cf.events_to_voxel_grid(ev, 5, 24, 20, is_reverse=True, mode="deterministic")
    rev = ev[::-1].copy()
    rev[:, 3] = -1.0
    ref = explicit.voxel_grid_sequential(rev, 5, 24, 20, explicit.FLAVOUR_NUMPY)
    assert np.array_equal(bits(got), bits(ref))


def test_voxel_full_size_properties(cuda_device):
    """HS-ERGB scale (config 4): 1 M events at 624x970 -- properties that do not
    need the sequential oracle: polarity sum is conserved, and atomic ~ deterministic."""
    n, h, w = 1_000_000, 624, 970
    ev = synth.events(n, h, w, seed=synth.seed_for(4))
    ev_d = dev_t(ev, cuda_device)
    off = torch.tensor([0, n], dtype=torch.int64, device=cuda_device)
    det = cf.events_to_voxel_grid_batched(ev_d, off, 5, w, h, flavour="torch", mode="deterministic")
    atom = cf.events_to_voxel_grid_batched(ev_d, off, 5, w, h, flavour="torch", mode="atomic")
    pol = np.where(ev[:, 3] == 0, -1.0, 1.0).sum()
    assert abs(det.double().sum().item() - pol) < 1e-2 * np.sqrt(n)   # each event deposits exactly its polarity
    assert_voxel_close(atom.cpu().numpy(), det.cpu().numpy())
    norm = cf.events_to_voxel_grid_batched(ev_d, off, 5, w, h, normalize="std", flavour="torch", mode="atomic")
    nz = norm[norm != 0].double()
    assert abs(nz.mean().item()) < 1e-3 and abs(nz.std(unbiased=False).item() - 1.0) < 1e-3


def test_voxel_error_paths(cuda_device):
    ev = dev_t(synth.events(10, 8, 8, 1), cuda_device)
    with pytest.raises(AssertionError):
        cf.events_to_voxel_grid_pytorch(ev[:, :3], 5, 8, 8)
    with pytest.raises(AssertionError):
        cf.events_to_voxel_grid_pytorch(ev, 0, 8, 8)
    with pytest.raises(RuntimeError):
        cf.events_to_voxel_grid_batched(ev.cpu(), torch.tensor([0, 10]), 5, 8, 8)


# ------------------------------------------------------------------- warp ---
def test_warp_golden(golden, cuda_device):
    g = golden("warp")
    img, flow = dev_t(g["img"], cuda_device), dev_t(g["flow"], cuda_device)
    fw, bw = cf.forwardWarp(22, 18), cf.backWarp(22, 18)
    np.testing.assert_allclose(fw(img, flow).cpu().numpy(), g["forward"], rtol=0, atol=1e-4)
    np.testing.assert_allclose(bw(img, flow).cpu().numpy(), g["backward"], rtol=0, atol=1e-4)
    np.testing.assert_allclose(fw(img, torch.zeros_like(flow)).cpu().numpy(), g["zero_flow_forward"], rtol=0, atol=1e-4)


def test_warp_frame_and_codes_golden(golden, cuda_device):
    g = golden("warp")
    img, codes, flow = (dev_t(g[f"step/{k}"], cuda_device) for k in ("img", "codes", "flow"))
    frame = cf.FrameWarp("forward")
    np.testing.assert_allclose(frame.warp_frame(img, flow).cpu().numpy(), g["step/img_warped"], rtol=0, atol=1e-4)
    half = dev_t(g["step/flow_half"], cuda_device)
    np.testing.assert_allclose(frame.warp_frame(codes, half).cpu().numpy(), g["step/codes_warped"], rtol=0, atol=1e-4)
    # fused x0.5 down-sampling: pass the full-resolution flow with the half-resolution codes
    np.testing.assert_allclose(cf.warp(codes, flow, -1.0).cpu().numpy(), g["step/codes_warped"], rtol=0, atol=1e-4)
    wi, wz = cf.warp_frame_and_codes(img, codes, flow, "forward")
    np.testing.assert_allclose(wi.cpu().numpy(), g["step/img_warped"], rtol=0, atol=1e-4)
    np.testing.assert_allclose(wz.cpu().numpy(), g["step/codes_warped"], rtol=0, atol=1e-4)
    _, wzb = cf.FrameWarp("backward").warp_frame_and_codes(img, codes, flow)
    np.testing.assert_allclose(wzb.cpu().numpy(), g["step/codes_warped_backward"], rtol=0, atol=1e-4)


@pytest.mark.parametrize("h,w,batch,channels", [(180, 240, 2, 128), (260, 346, 1, 128), (90, 120, 3, 5), (17, 23, 2, 1)])
@pytest.mark.parametrize("mode", ["forward", "backward"])
def test_warp_vs_oracle_config_shapes(cuda_device, h, w, batch, channels, mode):
    """Codes-shaped inputs (C=128 at H/2 x W/2) and image-shaped ones against the
    library-call oracle (F.grid_sample on CPU)."""
    img, codes, flow = synth.warp_inputs(batch, h, w, seed=5, code_channels=channels, flow_sigma=6.0)
    ref_i, ref_z = ref_port.warp_frame_and_codes(torch.from_numpy(img), torch.from_numpy(codes), torch.from_numpy(flow), mode)
    wi, wz = cf.warp_frame_and_codes(dev_t(img, cuda_device), dev_t(codes, cuda_device), dev_t(flow, cuda_device), mode)
    assert (wi.cpu() - ref_i).abs().max().item() <= 1e-4
    assert (wz.cpu() - ref_z).abs().max().item() <= 1e-4
    frame = cf.FrameWarp(mode)
    assert (frame.warp_frame(dev_t(img, cuda_device), dev_t(flow, cuda_device)).cpu() - ref_i).abs().max().item() <= 1e-4




@pytest.mark.parametrize("h,w,batch,channels,kernel", [
    (180, 240, 2, 128, "persist"),    # configs[1]: 90x120 codes, row pitch % 16 B == 0 -> TMA tensor boxes
    (260, 346, 1, 128, "persist"),     # configs[2]: 130x173 codes, odd width: no 16-byte row pitch -> quad-row tensor map
    (624, 970, 1, 32, "persist"),      # configs[3] shape (312x485 codes, odd width, H % 4 == 0), fewer channels to bound the CPU oracle
    (64, 96, 3, 13, "persist"),       # 13 channels: last chunk is partial (TMA zero-fills the missing channels)
    (66, 102, 2, 11, "direct"),        # 33x51 codes: odd width and 11 channels (the quad-row view needs C % 32 == 0)
    (66, 102, 2, 32, "persist"),       # 33x51 codes: odd width, odd height (channel stride 4 per stage), plane % 4 != 0
    (70, 44, 3, 64, "persist"),        # 35x22 codes: rows of 88 bytes (8-byte pitch), box wider than the image
    (36, 40, 1, 8, "persist"),        # tile larger than the image
])
@pytest.mark.parametrize("mode", ["forward", "backward"])
def test_warp_staged_paths_smooth_flow(cuda_device, monkeypatch, h, w, batch, channels, kernel, mode):
    """Network-like (smooth) flow: the taps of a tile fit the staging box, so the TMA-staged
    kernel does the work (asserted through cf_last_kernel), not the direct gather."""
    if kernel == "persist" and (w // 2) % 4:
        monkeypatch.setenv("CF_WARP_QUAD", "1")   # odd pitch: staged at any size (by default only from one full wave of CTAs)
    img, codes, flow = synth.warp_inputs(batch, h, w, seed=9, code_channels=channels, flow_kind="smooth")
    ref_i, ref_z = ref_port.warp_frame_and_codes(torch.from_numpy(img), torch.from_numpy(codes), torch.from_numpy(flow), mode)
    wi, wz = cf.warp_frame_and_codes(dev_t(img, cuda_device), dev_t(codes, cuda_device), dev_t(flow, cuda_device), mode)
    names = {"persist": ("warp_tma_kernel", "warp_tma_kernel"),
             "direct": ("warp_frame_and_codes_kernel", "warp_gather_kernel")}[kernel]
    assert last_kernel() == names[0]
    assert (wi.cpu() - ref_i).abs().max().item() <= 1e-4
    assert (wz.cpu() - ref_z).abs().max().item() <= 1e-4
    # the generic entry point (no image part, flow already at the codes' resolution)
    half = torch.nn.functional.interpolate(torch.from_numpy(flow), scale_factor=0.5, mode="bilinear", align_corners=True)
    got = cf.warp(dev_t(codes, cuda_device), half.to(cuda_device), -1.0 if mode == "forward" else 1.0)
    assert last_kernel() == names[1]
    assert (got.cpu() - ref_z).abs().max().item() <= 1e-4


def test_warp_image_rides_in_the_codes_tiles(cuda_device):
    """Many codes tiles (several waves of CTAs): the image blocks are warped by the first channel group's CTA of each
    codes tile instead of CTAs of their own.  24 streams of 192x256 with 128-channel codes = 1152 codes CTAs; both
    outputs against the oracle, including a frame whose flow has a discontinuity (direct-gather fallback tiles) and
    the gated all-zero-flow copy."""
    B, C, H, W = 24, 128, 192, 256
    img, codes, flow = synth.warp_inputs(B, H, W, seed=21, code_channels=C, flow_kind="smooth")
    flow[3, :, 50:120, 80:170] += 41.0
    ref_i, ref_z = ref_port.warp_frame_and_codes(torch.from_numpy(img), torch.from_numpy(codes), torch.from_numpy(flow), "forward")
    di, dz, df = dev_t(img, cuda_device), dev_t(codes, cuda_device), dev_t(flow, cuda_device)
    wi, wz = cf.warp_frame_and_codes(di, dz, df, "forward")
    assert last_kernel() == "warp_tma_kernel"
    assert (wi.cpu() - ref_i).abs().max().item() <= 1e-4
    assert (wz.cpu() - ref_z).abs().max().item() <= 1e-4
    gi, gz = cf.warp_frame_and_codes(di, dz, torch.zeros_like(df), "forward", skip_zero_flow=True)
    assert torch.equal(gi, di) and torch.equal(gz, dz)


@pytest.mark.parametrize("mode", ["forward", "backward"])
def test_warp_quad_row_view_mixed_tiles(cuda_device, mode):
    """Odd-width codes (130x173 of a 260x346 sensor) are staged through the quad-row tensor map (four source rows per
    map row, four boxes per channel, residue-major rows in shared memory).  Smooth flow with a discontinuity: ring tiles
    and direct-gather tiles in one launch, several streams (the global source-row index crosses stream boundaries), the
    last rows/columns of the plane (boxes run past the row end and past the channel end), and the gated copy."""
    B, C, H, W = 5, 128, 260, 346   # 540 codes CTAs: above the one-wave threshold of the odd-pitch path
    img, codes, flow = synth.warp_inputs(B, H, W, seed=31, code_channels=C, flow_kind="smooth")
    flow[1, :, 60:150, 200:300] += 33.0
    ref_i, ref_z = ref_port.warp_frame_and_codes(torch.from_numpy(img), torch.from_numpy(codes), torch.from_numpy(flow), mode)
    di, dz, df = dev_t(img, cuda_device), dev_t(codes, cuda_device), dev_t(flow, cuda_device)
    wi, wz = cf.warp_frame_and_codes(di, dz, df, mode)
    assert last_kernel() == "warp_tma_kernel"
    assert (wi.cpu() - ref_i).abs().max().item() <= 1e-4
    assert (wz.cpu() - ref_z).abs().max().item() <= 1e-4
    gi, gz = cf.warp_frame_and_codes(di, dz, torch.zeros_like(df), mode, skip_zero_flow=True)
    assert torch.equal(gi, di) and torch.equal(gz, dz)


def test_warp_staged_misaligned_base_and_mixed_tiles(cuda_device):
    """(a) a codes tensor whose base address is only 4-byte aligned (a view into a larger buffer) cannot
    be described by a tensor map and takes the direct gather; (b) smooth flow with one discontinuity: tiles
    that fit use the ring, the others the in-kernel direct gather, in the same launch."""
    B, C, H, W = 2, 16, 128, 192
    img, codes, flow = synth.warp_inputs(B, H, W, seed=4, code_channels=C, flow_kind="smooth")
    flow[:, :, 40:90, 60:130] += 37.0   # a moving object: taps of the tiles on its border span > 48 px
    ref_i, ref_z = ref_port.warp_frame_and_codes(torch.from_numpy(img), torch.from_numpy(codes), torch.from_numpy(flow), "forward")
    for shift in (0, 1, 3):
        buf = torch.zeros(codes.size + 8, device=cuda_device)
        view = buf[shift:shift + codes.size].view(codes.shape)
        view.copy_(torch.from_numpy(codes))
        assert view.data_ptr() % 16 == 4 * shift
        wi, wz = cf.warp_frame_and_codes(dev_t(img, cuda_device), view, dev_t(flow, cuda_device), "forward")
        assert last_kernel() == ("warp_tma_kernel" if shift == 0 else "warp_frame_and_codes_kernel")
        assert (wi.cpu() - ref_i).abs().max().item() <= 1e-4
        assert (wz.cpu() - ref_z).abs().max().item() <= 1e-4


def test_warp_full_size_properties(cuda_device):
    """480x640 codes (config 5): constant image stays constant (weights sum to 1);
    linearity warp(a*x + y) = a*warp(x) + warp(y); forward(flow) == backward(-flow)."""
    B, C, H, W = 2, 128, 240, 320
    gen = torch.Generator(device="cpu").manual_seed(3)
    x = torch.randn(B, C, H, W, generator=gen).to(cuda_device)
    y = torch.randn(B, C, H, W, generator=gen).to(cuda_device)
    flow = (7.0 * torch.randn(B, 2, 2 * H, 2 * W, generator=gen)).to(cuda_device)
    const = torch.full_like(x, 3.25)
    assert (cf.warp(const, flow, -1.0) - 3.25).abs().max().item() <= 1e-5
    lhs = cf.warp(2.5 * x + y, flow, -1.0)
    rhs = 2.5 * cf.warp(x, flow, -1.0) + cf.warp(y, flow, -1.0)
    assert (lhs - rhs).abs().max().item() <= 1e-4
    assert torch.equal(cf.warp(x, flow, -1.0), cf.warp(x, -flow, +1.0))


@pytest.mark.parametrize("mode", ["forward", "backward"])
@pytest.mark.parametrize("shape,flow_kind", [((2, 3, 18, 22), "noise"), ((1, 128, 90, 120), "smooth"), ((2, 5, 31, 45), "smooth")])
def test_warp_backward_matches_autograd_of_the_reference_ops(cuda_device, parity_report, mode, shape, flow_kind):
    """SURVEY 8f rank 2: gradients of forwardWarp / backWarp w.r.t. image (the bilinear splat) and flow against
    torch.autograd through the oracle port (F.grid_sample, reflection padding) on CPU."""
    B, C, H, W = shape
    rng = np.random.default_rng(5)
    img = rng.standard_normal(shape).astype(np.float32)
    _, _, flow = synth.warp_inputs(B, H, W, seed=8, code_channels=8, flow_kind=flow_kind)
    flow[0, :, 0, 0] = [-3.0 * W, 2.5 * H]      # far outside: reflected several times
    gout = rng.standard_normal(shape).astype(np.float32)
    ri, rf = torch.from_numpy(img).requires_grad_(), torch.from_numpy(flow).requires_grad_()
    ref_port.warp(ri, rf, mode).backward(torch.from_numpy(gout))
    di, df = dev_t(img, cuda_device).requires_grad_(), dev_t(flow, cuda_device).requires_grad_()
    mod = cf.forwardWarp(W, H) if mode == "forward" else cf.backWarp(W, H)
    out = mod(di, df)
    assert out.requires_grad
    out.backward(dev_t(gout, cuda_device))
    assert last_kernel() == "warp_backward_kernel"
    scale_i = max(1.0, float(ri.grad.abs().max()))
    scale_f = max(1.0, float(rf.grad.abs().max()))
    assert (di.grad.cpu() - ri.grad).abs().max().item() <= 1e-4 * scale_i
    # the flow gradient is discontinuous where a sample sits exactly on a pixel boundary: compare away from those
    err = (df.grad.cpu() - rf.grad).abs()
    assert err.max().item() <= 2e-3 * scale_f, err.max().item()
    assert (err > 1e-4 * scale_f).float().mean().item() < 1e-3
    parity_report.add("warp_backward_flow_gradient", mode=mode, shape=list(shape), flow_kind=flow_kind, elements=err.numel(),
                      above_1e4th_of_scale=int((err > 1e-4 * scale_f).sum()), max_err_over_scale=err.max().item() / scale_f)


def test_warp_backward_fused_half_resolution_flow(cuda_device, parity_report):
    """Codes at half resolution warped with the full-resolution flow (e2v_model.py:190): the kernel also applies the
    adjoint of the x0.5 bilinear down-sampling.  Oracle: autograd through F.interpolate + grid_sample."""
    B, C, H, W = 2, 16, 36, 48
    rng = np.random.default_rng(6)
    codes = rng.standard_normal((B, C, H // 2, W // 2)).astype(np.float32)
    _, _, flow = synth.warp_inputs(B, H, W, seed=9, code_channels=8, flow_kind="smooth")
    gout = rng.standard_normal(codes.shape).astype(np.float32)
    rz, rf = torch.from_numpy(codes).requires_grad_(), torch.from_numpy(flow).requires_grad_()
    ref_port.warp(rz, ref_port.downsample_flow(rf), "forward").backward(torch.from_numpy(gout))
    dz, df = dev_t(codes, cuda_device).requires_grad_(), dev_t(flow, cuda_device).requires_grad_()
    cf.warp(dz, df, -1.0).backward(dev_t(gout, cuda_device))
    assert (dz.grad.cpu() - rz.grad).abs().max().item() <= 1e-4 * max(1.0, float(rz.grad.abs().max()))
    err = (df.grad.cpu() - rf.grad).abs()
    scale = max(1.0, float(rf.grad.abs().max()))
    assert err.max().item() <= 2e-3 * scale and (err > 1e-4 * scale).float().mean().item() < 1e-3
    parity_report.add("warp_backward_flow_gradient_half_res", elements=err.numel(), above_1e4th_of_scale=int((err > 1e-4 * scale).sum()),
                      max_err_over_scale=err.max().item() / scale)


def test_warp_rejects_cpu_and_grad(cuda_device):
    img = torch.zeros(1, 1, 8, 8)
    with pytest.raises(RuntimeError):
        cf.forwardWarp(8, 8)(img, torch.zeros(1, 2, 8, 8))
    g = torch.zeros(1, 1, 8, 8, device=cuda_device, requires_grad=True)
    with pytest.raises(RuntimeError):   # the fused per-frame step is inference-only (warp() itself is differentiable)
        cf.warp_frame_and_codes(g, torch.zeros(1, 4, 4, 4, device=cuda_device), torch.zeros(1, 2, 8, 8, device=cuda_device))
    with pytest.raises(ValueError):
        cf.warp(torch.zeros(1, 1, 8, 8, device=cuda_device), torch.zeros(1, 2, 5, 5, device=cuda_device), -1.0)


# ---------------------------------------------------------- second voxeliser ---
@pytest.mark.parametrize("case", ["base", "binary", "dense", "two"])
def test_mvsec_voxeliser_golden(golden, cuda_device, case):
    """eventsToVoxel / events_to_voxel_torch (data_readers/MVSEC_utils.py, SURVEY 8f rank 4) = CF_FLAVOUR_MVSEC:
    deterministic mode bit-exact against the reference's own outputs (its per-bin index_put_ is sequential at these
    sizes), atomic mode within the voxel tolerance; both the signed grid and the positive / negative split."""
    g = golden("mvsec")
    ev = g[f"{case}/events_xytp"]
    nb, h, w = (int(v) for v in g[f"{case}/dims"])
    for pol, key in ((False, "voxel"), (True, "voxel_pol")):
        det = cf.eventsToVoxel(ev.copy(), num_bins=nb, height=h, width=w, event_polarity=pol, mode="deterministic")
        assert isinstance(det, np.ndarray) and det.dtype == np.float32 and det.shape == g[f"{case}/{key}"].shape
        assert np.array_equal(bits(det), bits(g[f"{case}/{key}"]))
        fast = cf.eventsToVoxelTorch(ev.copy(), nb, h, w, pol, mode="atomic")
        assert fast.device.type == "cpu"            # comes back where the input lived, like the reference
        assert_voxel_close(fast.numpy(), g[f"{case}/{key}"])
    xs, ys, ts, ps = (torch.from_numpy(np.ascontiguousarray(ev[:, k])) for k in (0, 1, 2, 3))
    direct = cf.events_to_voxel_torch(xs.int(), ys.int(), (ts - ts[0]) / (ts[-1] - ts[0]), ps.int(), nb, sensor_size=(h, w),
                                      device=cuda_device, mode="deterministic")
    assert direct.device.type == "cuda" and np.array_equal(bits(direct.cpu().numpy()), bits(g[f"{case}/direct"]))
    naive = cf.events_to_voxel_torch(xs.int(), ys.int(), (ts - ts[0]) / (ts[-1] - ts[0]), ps.int(), nb, sensor_size=(h, w),
                                     device=cuda_device, temporal_bilinear=False, mode="deterministic")
    assert np.array_equal(bits(naive.cpu().numpy()), bits(g[f"{case}/naive"]))   # MVSEC_utils.py:292-300


def test_mvsec_voxeliser_config_shape(cuda_device):
    """100 000 events at 480x640 (config 5): against the oracle port; conservation -- every event with a time stamp
    inside the window spreads exactly its polarity over two bins."""
    ev = synth.events(100000, 480, 640, 77)
    p = np.where(ev[:, 3] > 0, 1.0, -1.0)
    xytp = np.stack([ev[:, 1], ev[:, 2], ev[:, 0], p], axis=1)
    ref = ref_port.mvsec_events_to_voxel(xytp, 5, 480, 640, False)
    for mode in ("atomic", "deterministic"):
        got = cf.eventsToVoxel(xytp.copy(), 5, 480, 640, mode=mode)
        assert_voxel_close(got, ref)
    assert abs(float(got.astype(np.float64).sum()) - float(p.sum())) <= 1e-2


def test_zero_flow_gate_matches_the_reference_branch(cuda_device):
    """SURVEY 8f rank 1: `if not flow_final.any(): keep rec_img0 / states` (e2v_model.py:184-191) evaluated on the
    device.  All-zero flow (incl. -0.0) -> outputs are the inputs (NOT the zero-flow warp, which shifts every pixel,
    SURVEY F6); one non-zero or NaN element anywhere -> the ordinary warp; the whole step is capturable in a CUDA
    graph and re-evaluates the predicate on every replay."""
    img, codes, flow = (dev_t(a, cuda_device) for a in synth.warp_inputs(2, 64, 96, seed=3, code_channels=16, flow_kind="smooth"))
    zero = torch.zeros_like(flow)
    zero[1, 0, 5, 7] = -0.0
    assert cf.flow_any(zero).item() == 0 and cf.flow_any(flow).item() == 1
    odd = torch.zeros(1037, device=cuda_device)      # tail handling (n % 4 != 0)
    assert cf.flow_any(odd).item() == 0
    odd[-1] = 1e-30
    assert cf.flow_any(odd).item() == 1
    odd[-1] = float("nan")
    assert cf.flow_any(odd).item() == 1
    for mode in ("forward", "backward"):
        wi, wz = cf.warp_frame_and_codes(img, codes, zero, mode, skip_zero_flow=True)
        assert torch.equal(wi, img) and torch.equal(wz, codes)
        ref_i, ref_z = ref_port.warp_frame_and_codes(img.cpu(), codes.cpu(), zero.cpu(), mode)
        assert (ref_i - img.cpu()).abs().max() > 1e-3          # the un-gated zero-flow warp is not the identity ...
        ui, uz = cf.warp_frame_and_codes(img, codes, zero, mode)
        assert (ui.cpu() - ref_i).abs().max() <= 1e-4 and (uz.cpu() - ref_z).abs().max() <= 1e-4   # ... and we match it
        one = zero.clone()
        one[0, 1, 3, 3] = 2.5
        gi, gz = cf.warp_frame_and_codes(img, codes, one, mode, skip_zero_flow=True)
        ri, rz = ref_port.warp_frame_and_codes(img.cpu(), codes.cpu(), one.cpu(), mode)
        assert (gi.cpu() - ri).abs().max() <= 1e-4 and (gz.cpu() - rz).abs().max() <= 1e-4
    # graph capture: the predicate is re-evaluated on the device at every replay
    fbuf = flow.clone()
    s = torch.cuda.Stream(cuda_device)
    with torch.cuda.stream(s):
        cf.warp_frame_and_codes(img, codes, fbuf, "forward", skip_zero_flow=True)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            gi, gz = cf.warp_frame_and_codes(img, codes, fbuf, "forward", skip_zero_flow=True)
        g.replay()
        torch.cuda.synchronize()
        ri, _ = ref_port.warp_frame_and_codes(img.cpu(), codes.cpu(), flow.cpu(), "forward")
        assert (gi.cpu() - ri).abs().max() <= 1e-4
        fbuf.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(gi, img) and torch.equal(gz, codes)


# -------------------------------------------------------------------- fwl ---
def test_fwl_golden_and_config_shape(golden, cuda_device):
    """voxel_warping_flow_loss (FWL metric, SURVEY 8f rank 4): warped channels within the warp tolerance
    (1e-4 abs) of the reference's own output, variance within 1e-5 relative; then a 480x640 grid against
    the oracle port, and the FWL ratio itself (loss(flow) / loss(0))."""
    g = golden("fwl")
    voxel, disp = dev_t(g["voxel"], cuda_device), dev_t(g["disp"], cuda_device)
    for rev in (False, True):
        loss, extra = cf.voxel_warping_flow_loss(voxel, disp, output_images=True, reverse_time=rev)
        assert last_kernel() == "moments_finish_kernel"
        assert loss.device.type == "cuda" and loss.dim() == 0 and loss.dtype == torch.float32
        assert extra["voxel_grid"] is voxel
        np.testing.assert_allclose(extra["voxel_grid_warped"].cpu().numpy(), g[f"warped_{int(rev)}"], rtol=0, atol=1e-4)
        assert abs(loss.item() - float(g[f"loss_{int(rev)}"])) <= 1e-5 * abs(float(g[f"loss_{int(rev)}"]))
    zero = cf.voxel_warping_flow_loss(voxel, torch.zeros_like(disp))
    assert abs(zero.item() - float(g["loss_zero_flow"])) <= 1e-5 * float(g["loss_zero_flow"])
    # config-5 frame, batch 2
    ev = [synth.events(100000, 480, 640, 900 + b) for b in range(2)]
    vox = np.stack([ref_port.voxel_grid_numpy(e, 5, 640, 480) for e in ev]).astype(np.float32)
    _, _, flow = synth.warp_inputs(2, 480, 640, seed=17, code_channels=8, flow_kind="smooth")
    ref_var, ref_sum, ref_warped = ref_port.voxel_flow_warp(torch.from_numpy(vox), torch.from_numpy(flow))
    loss, extra = cf.voxel_warping_flow_loss(dev_t(vox, cuda_device), dev_t(flow, cuda_device), output_images=True)
    assert (extra["voxel_grid_warped"].cpu() - ref_warped).abs().max().item() <= 1e-4
    assert abs(loss.item() - ref_var.item()) <= 1e-5 * ref_var.item()
    fwl = loss / cf.voxel_warping_flow_loss(dev_t(vox, cuda_device), torch.zeros(2, 2, 480, 640, device=cuda_device))
    ref0, _, _ = ref_port.voxel_flow_warp(torch.from_numpy(vox), torch.zeros(2, 2, 480, 640))
    assert abs(fwl.item() - (ref_var / ref0).item()) <= 1e-5
    with pytest.raises(ValueError):   # the reference divides by C - 1
        cf.voxel_warping_flow_loss(torch.zeros(1, 1, 8, 8, device=cuda_device), torch.zeros(1, 2, 8, 8, device=cuda_device))


# ------------------------------------------------------------------- corr ---
def corr_err(got, ref):
    """Normwise error max|err| / max|ref|, after asserting the element-wise agreement north_star asks for:
    the fraction of elements with |err| <= 1e-3 * (|ref| + rms(ref)) (SURVEY.md H3) must be >= 95 %."""
    g, r = got.astype(np.float64), ref.astype(np.float64)
    err = np.abs(g - r)
    rms = float(np.sqrt(np.mean(r * r))) if r.size else 0.0
    frac = float((err <= 1e-3 * (np.abs(r) + rms)).mean()) if err.size else 1.0
    CORR_FRACTIONS.append(frac)
    assert frac >= 0.95, f"only {frac:.4f} of the elements within 1e-3*(|ref|+rms)"
    return float(err.max() / max(np.abs(r).max(), 1e-30))


CORR_FRACTIONS = []   # H3 agreement fraction of every correlation / lookup comparison of this session


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("tf32", 1e-3)])
def test_corr_golden(golden, cuda_device, precision, tol):
    g = golden("corr")
    blk = cf.CorrBlock(dev_t(g["fmap1"], cuda_device), dev_t(g["fmap2"], cuda_device), num_levels=4, radius=4,
                       precision=precision)
    assert len(blk.corr_pyramid) == 4
    for l in range(4):
        assert tuple(blk.corr_pyramid[l].shape) == g[f"pyr{l}"].shape
        assert corr_err(*g.pick(f"pyr{l}", blk.corr_pyramid[l].cpu().numpy())) <= tol, f"level {l}"
    out = blk(dev_t(g["coords"], cuda_device))
    assert tuple(out.shape) == g["lookup"].shape and out.is_contiguous()
    assert corr_err(*g.pick("lookup", out.cpu().numpy())) <= tol
    vol = cf.CorrBlock.corr(dev_t(g["fmap1"], cuda_device), dev_t(g["fmap2"], cuda_device), precision=precision)
    assert tuple(vol.shape) == (1, 16, 24, 1, 16, 24)


def test_corr_f16_operands_match_tf32(cuda_device):
    """CF_CORR_F16: fp16 copies of the operands, scaled per batch item by a power of two, through tcgen05 kind::f16.
    The operands carry the same 11-bit significands as TF32 operands, so the two paths differ only by the fp32
    summation order inside the MMAs (K = 16 against K = 8 per instruction): <= 1e-5 of max|ref| apart, also for inputs
    far outside the fp16 range; 3-D operand boxes (24x32), per-atom boxes (36x44) and an all-zero map."""
    for (H, W, B, scale) in ((192, 256, 2, 1.0), (288, 352, 1, 1.0), (192, 256, 1, 3.0e6), (192, 256, 1, 1.0e-9)):
        f1, f2, _ = synth.corr_inputs(B, H, W, 9)
        a, b = dev_t(f1, cuda_device) * scale, dev_t(f2, cuda_device)
        t32 = cf.build_pyramid(a, b, 4, precision="tf32")
        f16 = cf.build_pyramid(a, b, 4, precision="f16")
        assert last_kernel() in ("corr_tc_kernel<f16>", "avg_pool_two_levels_kernel")
        ref = cf.build_pyramid(a, b, 4, precision="fp32")
        for l in range(4):
            assert corr_err(f16[l].cpu().numpy(), t32[l].cpu().numpy()) <= 1e-5, (H, W, scale, l)
            assert corr_err(f16[l].cpu().numpy(), ref[l].cpu().numpy()) <= 1e-3
    z = torch.zeros(1, 256, 24, 32, device=cuda_device)
    for lvl in cf.build_pyramid(z, dev_t(synth.corr_inputs(1, 192, 256, 1)[1], cuda_device), 4, precision="f16"):
        assert not lvl.any()


def test_corr_pair_kernel_subprocess(cuda_device):
    """The cta_group::2 variant of the tensor-core correlation (CF_TC_FLAGS bit6, read once per process, hence the
    subprocess): 256-row UMMAs across a CTA pair.  Checked against the fp32 SIMT kernel at an even tile count
    (24x32, 3-D operand boxes), an odd one (36x44: 13 query tiles -> one dummy tile, per-atom boxes, N/2 not on
    a box boundary) and 60x80 (BN = 160: half tiles of 2.5 boxes)."""
    import os
    import subprocess
    import sys
    code = """
import numpy as np, torch
import cistaflow_b200 as cf
from cistaflow_b200 import synth, _lib
dev = torch.device('cuda', 0)
for (H, W, B) in ((192, 256, 2), (288, 352, 2), (480, 640, 1)):
    f1, f2, _ = synth.corr_inputs(B, H, W, 5)
    a, b = torch.from_numpy(f1).to(dev), torch.from_numpy(f2).to(dev)
    ref = cf.build_pyramid(a, b, 4, precision='fp32')
    cf.build_pyramid(a, b, 2, precision='tf32')   # two levels: the fused kernel is the only launch
    assert _lib.load().cf_last_kernel().decode() == 'corr_tc_kernel<pair>', _lib.load().cf_last_kernel()
    got = cf.build_pyramid(a, b, 4, precision='tf32')
    for l in range(4):
        r = ref[l].float(); g = got[l].float()
        err = (g - r).abs().max().item() / r.abs().max().item()
        assert err <= 1e-3, (H, W, l, err)
print('PAIR_OK')
"""
    env = dict(os.environ, CF_TC_FLAGS="64")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=env,
                         cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert res.returncode == 0 and "PAIR_OK" in res.stdout, res.stdout + res.stderr


def test_corr_golden_odd_sizes(golden, cuda_device):
    """15x20 maps, 3 levels, radius 3: avg_pool floors, runtime-radius lookup kernel."""
    g = golden("corr")
    blk = cf.CorrBlock(dev_t(g["odd/fmap1"], cuda_device), dev_t(g["odd/fmap2"], cuda_device), num_levels=3, radius=3,
                       precision="fp32")
    for l in range(3):
        assert tuple(blk.corr_pyramid[l].shape) == g[f"odd/pyr{l}"].shape
        assert corr_err(*g.pick(f"odd/pyr{l}", blk.corr_pyramid[l].cpu().numpy())) <= 1e-5
    assert corr_err(*g.pick("odd/lookup", blk(dev_t(g["odd/coords"], cuda_device)).cpu().numpy())) <= 1e-5
    blk_tc = cf.CorrBlock(dev_t(g["odd/fmap1"], cuda_device), dev_t(g["odd/fmap2"], cuda_device), num_levels=3, radius=3,
                          precision="tf32")  # 15x20: N % 4 == 0, odd h -> un-fused tensor-core path
    for l in range(3):
        assert corr_err(*g.pick(f"odd/pyr{l}", blk_tc.corr_pyramid[l].cpu().numpy())) <= 1e-3


@pytest.mark.parametrize("h,w,levels,radius", [(16, 24, 4, 4), (15, 20, 3, 3)])
def test_corr_block_backward_matches_autograd_of_the_reference_ops(cuda_device, h, w, levels, radius):
    """SURVEY 8f rank 2: gradients through CorrBlock (pyramid build + lookup) w.r.t. both feature maps and the
    lookup coordinates, against torch.autograd through the oracle port on CPU (fp32 correlation path)."""
    rng = np.random.default_rng(12)
    B, D = 2, 64
    f1 = rng.standard_normal((B, D, h, w)).astype(np.float32)
    f2 = rng.standard_normal((B, D, h, w)).astype(np.float32)
    ys, xs = np.meshgrid(np.arange(h, dtype=np.float32), np.arange(w, dtype=np.float32), indexing="ij")
    coords = (np.stack([xs, ys])[None] + 2.5 * rng.standard_normal((B, 2, h, w))).astype(np.float32)
    coords[0, :, 0, 0] = [-7.3, h + 5.2]     # window partly / wholly outside the map
    k = 2 * radius + 1
    gout = rng.standard_normal((B, levels * k * k, h, w)).astype(np.float32)
    rf1, rf2, rc = (torch.from_numpy(a).requires_grad_() for a in (f1, f2, coords))
    ref_port.corr_lookup(ref_port.corr_pyramid(rf1, rf2, levels), rc, radius).backward(torch.from_numpy(gout))
    df1, df2, dc = (dev_t(a, cuda_device).requires_grad_() for a in (f1, f2, coords))
    blk = cf.CorrBlock(df1, df2, num_levels=levels, radius=radius, precision="fp32")
    out = blk(dc)
    assert out.requires_grad
    out.backward(dev_t(gout, cuda_device))
    for got, ref, name in ((df1.grad, rf1.grad, "fmap1"), (df2.grad, rf2.grad, "fmap2")):
        assert corr_err(got.cpu().numpy(), ref.numpy()) <= 1e-4, name
    # the coordinate gradient jumps where a sample sits on a pixel boundary: compare away from those
    err = (dc.grad.cpu() - rc.grad).abs()
    scale = float(rc.grad.abs().max())
    assert err.max().item() <= 2e-3 * scale and (err > 1e-4 * scale).float().mean().item() < 1e-3


def test_lookup_on_reference_pyramid(golden, cuda_device):
    """Feed the REFERENCE's pyramid to our lookup: isolates the gather from the GEMM.  (The fixture stores the pyramid
    rows of a sample of the queries; a query's lookup reads only its own rows.)"""
    g = golden("corr")
    pyr = [dev_t(g[f"pyr{l}"], cuda_device) for l in range(4)]
    out = cf.corr_lookup(pyr, dev_t(g["coords"], cuda_device), 4)
    assert corr_err(*g.pick("lookup", out.cpu().numpy())) <= 1e-4
    assert np.abs(out.cpu().numpy()[0, :, 0, 0]).max() == 0.0  # query far outside: zero padding everywhere


@pytest.mark.parametrize("h,w,batch", [(180, 240, 8), (260, 346, 1), (480, 640, 1), (624, 970, 1), (128, 192, 2)])
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("tf32", 1e-3)])
def test_corr_vs_oracle_config_shapes(cuda_device, h, w, batch, precision, tol):
    f1, f2, coords = synth.corr_inputs(batch, h, w, seed=9)
    ref_pyr = ref_port.corr_pyramid(torch.from_numpy(f1), torch.from_numpy(f2), 4)
    blk = cf.CorrBlock(dev_t(f1, cuda_device), dev_t(f2, cuda_device), precision=precision)
    for l in range(4):
        assert tuple(blk.corr_pyramid[l].shape) == tuple(ref_pyr[l].shape)
        assert corr_err(blk.corr_pyramid[l].cpu().numpy(), ref_pyr[l].numpy()) <= tol, f"level {l}"
    ref_out = ref_port.corr_lookup(ref_pyr, torch.from_numpy(coords), 4)
    assert corr_err(blk(dev_t(coords, cuda_device)).cpu().numpy(), ref_out.numpy()) <= tol


def test_corr_full_size_properties(cuda_device):
    """624x970 (config 4: N = 9920, 394 MB level 0): symmetry corr(f1,f2)[i,j] ==
    corr(f2,f1)[j,i] on a sample, level-1 == 2x2 mean of level 0, lookup at integer
    coords with zero fraction returns the level-0 entries."""
    f1, f2, _ = synth.corr_inputs(1, 624, 970, seed=4)
    a, b = dev_t(f1, cuda_device), dev_t(f2, cuda_device)
    h, w = a.shape[-2:]
    N = h * w
    blk = cf.CorrBlock(a, b, precision="tf32")
    l0 = blk.corr_pyramid[0].view(N, h, w)
    idx = torch.randint(0, N, (64,), device=cuda_device)
    exact = (a[0].reshape(256, N)[:, idx].double().T @ b[0].reshape(256, N).double()) / 16.0
    got = l0.view(N, N)[idx].double()
    assert (got - exact).abs().max().item() <= 1e-3 * exact.abs().max().item()
    pooled = torch.nn.functional.avg_pool2d(l0[idx], 2, 2)
    assert (blk.corr_pyramid[1].view(N, h // 2, w // 2)[idx] - pooled).abs().max().item() <= 1e-5
    coords = cf.coords_grid(1, h, w, device=cuda_device)
    out = blk(coords)
    centre = out[0, 4 * 9 + 4].reshape(N)          # level 0, i = j = r
    assert torch.equal(centre, l0.view(N, N).diagonal())


# ------------------------------------------------------------ model traces ---
@pytest.mark.parametrize("trace", ["trace_eiflow", "trace_eraft"])
def test_model_trace_replay(golden, cuda_device, trace):
    """Every hot-path call the reference model made on its 3rd recurrent frame,
    replayed through the CUDA path (real feature / flow statistics, ImagePadder shapes)."""
    g = golden(trace)
    H, W, nev, n_lookup, n_warp = (int(v) for v in g["meta"])
    grid = cf.events_to_voxel_grid(synth.events(nev, H, W, int(g["voxel/seed"])), 5, W, H, mode="deterministic")
    got, ref = g.pick("voxel/grid", grid)
    assert np.array_equal(bits(got), bits(ref))
    np.testing.assert_allclose(*g.pick("voxel/normalised", cf.event_preprocess(grid, "std", True)), rtol=1e-5, atol=1e-5)
    blk = cf.CorrBlock(dev_t(g["corr/fmap1"], cuda_device), dev_t(g["corr/fmap2"], cuda_device), num_levels=4, radius=4)
    for l in range(4):
        assert corr_err(*g.pick(f"corr/pyr{l}", blk.corr_pyramid[l].cpu().numpy())) <= 1e-3
    for k in range(n_lookup):
        if f"lookup{k}/out" in g:
            out = blk(dev_t(g[f"lookup{k}/coords"], cuda_device))
            assert corr_err(*g.pick(f"lookup{k}/out", out.cpu().numpy())) <= 1e-3
    frame = cf.FrameWarp("forward")
    for k in range(n_warp):
        out = frame.warp_frame(dev_t(g[f"warp{k}/in"], cuda_device), dev_t(g[f"warp{k}/flow"], cuda_device))
        np.testing.assert_allclose(*g.pick(f"warp{k}/out", out.cpu().numpy()), rtol=0, atol=1e-4)
    wi, wz = cf.warp_frame_and_codes(dev_t(g["warp0/in"], cuda_device), dev_t(g["warp1/in"], cuda_device),
                                     dev_t(g["flow_final"], cuda_device), "forward")
    np.testing.assert_allclose(*g.pick("warp0/out", wi.cpu().numpy()), rtol=0, atol=1e-4)
    np.testing.assert_allclose(*g.pick("warp1/out", wz.cpu().numpy()), rtol=0, atol=1e-4)


# ------------------------------------------------- agreement summaries (run last) ---
def test_zz_voxel_atomic_agreement_summary(parity_report):
    """Runs last in this file's voxel block order-independently: reports min / mean of the literal-tolerance fractions."""
    if VOXEL_FRACTIONS:
        parity_report.add("voxel_atomic_literal_1e-5*(|ref|+1)", comparisons=len(VOXEL_FRACTIONS),
                          min_fraction=min(VOXEL_FRACTIONS), mean_fraction=float(np.mean(VOXEL_FRACTIONS)))
        print(f"voxel atomic mode: {len(VOXEL_FRACTIONS)} comparisons, min fraction within 1e-5*(|ref|+1) = {min(VOXEL_FRACTIONS):.6f}")


def test_zz_corr_agreement_summary(parity_report):
    if CORR_FRACTIONS:
        parity_report.add("corr_H3_1e-3*(|ref|+rms)", comparisons=len(CORR_FRACTIONS), min_fraction=min(CORR_FRACTIONS),
                          mean_fraction=float(np.mean(CORR_FRACTIONS)))
        print(f"correlation: {len(CORR_FRACTIONS)} comparisons, min fraction within 1e-3*(|ref|+rms) = {min(CORR_FRACTIONS):.6f}")
