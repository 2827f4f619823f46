"""torch.use_deterministic_algorithms(True) across the library: the deterministic warp adjoint
(include/cistaflow_det.h, csrc/warp_backward_det.cu), the fixed-order CorrBlock coordinate gradient, and the voxel
mode the flag selects.

Under the flag the warp gradients must agree with CPU autograd through the oracle port at the tolerances of the atomic
path's tests, and be bitwise equal from call to call, on a side stream and in a CUDA graph.  The flag is switched on
only inside ``deterministic_algorithms()``, which restores the previous state (warn_only included), so later tests in
the session run the default paths.
"""
import contextlib
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DET_KERNELS = ("warp_backward_det_gather_kernel", "warp_backward_det_flow_half_kernel")


@contextlib.contextmanager
def deterministic_algorithms(warn_only=False):
    """The flag on, with the cuBLAS workspace setting torch requires for matmul under it; restores both."""
    prev = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    prev_env = os.environ.get("CUBLAS_WORKSPACE_CONFIG")
    os.environ["CUBLAS_WORKSPACE_CONFIG"] = ":4096:8"
    torch.use_deterministic_algorithms(True, warn_only=warn_only)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])
        if prev_env is None:
            os.environ.pop("CUBLAS_WORKSPACE_CONFIG", None)
        else:
            os.environ["CUBLAS_WORKSPACE_CONFIG"] = prev_env


@pytest.fixture
def deterministic():
    with deterministic_algorithms():
        yield


def _header_symbols(name):
    text = open(os.path.join(ROOT, "include", name)).read()
    return sorted(re.findall(r"CF_API\s+[\w\s\*]+?\b(cf_\w+)\s*\(", text))


def last_kernel():
    from cistaflow_b200 import _lib
    return _lib.load().cf_last_kernel().decode()


def dev_t(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


# ----------------------------------------------------------------------------------------------------- CPU ---
def test_det_header_matches_ctypes_table_and_library():
    import cistaflow_b200 as cf
    from cistaflow_b200 import _lib
    syms = _header_symbols("cistaflow_det.h")
    assert syms == sorted(["cf_warp_backward_det_workspace_bytes", "cf_warp_backward_det"])
    assert syms == sorted(_lib.DET_SYMBOLS)
    assert len(_header_symbols("cistaflow.h")) == 26 and len(_header_symbols("cistaflow_altcorr.h")) == 3
    assert not set(syms) & set(_lib.SYMBOLS) and not set(syms) & set(_lib.ALTCORR_SYMBOLS)
    lib = cf.load_library()
    for name in syms:
        assert getattr(lib, name).restype == _lib.DET_SYMBOLS[name][0]


def _workspace_formula(B, C, H, W, fH, fW):
    """The bound cistaflow_det.h documents, written out."""
    if B == 0 or C == 0:
        return 0
    half = (fH, fW) != (H, W)
    up = lambda x: (x + 255) // 256 * 256   # noqa: E731
    plane = H * W
    chunk = min(B, 0xFFFFFFFF // (4 * plane))
    pix = chunk * plane
    n = 4 * pix
    return (5 * up(4 * n) + up(4 * (pix + 1)) + up(4 * 256 * -(-n // 4096)) + (up(8 * pix) if half else 0)) + 256


def test_det_workspace_formula():
    import cistaflow_b200 as cf
    lib = cf.load_library()
    for shape in [(8, 1, 180, 240, 180, 240), (8, 128, 90, 120, 180, 240), (64, 1, 480, 640, 480, 640),
                  (64, 128, 240, 320, 480, 640), (2, 5, 31, 45, 31, 45), (2, 16, 18, 24, 37, 49), (1, 1, 1, 1, 3, 3)]:
        n = lib.cf_warp_backward_det_workspace_bytes(*shape)
        assert n == _workspace_formula(*shape), shape
        B, C, H, W = shape[:4]
        assert 20 * 4 * B * H * W <= n <= 24 * 4 * B * H * W + 12 * 256, shape
    # 4*B*H*W >= 2^32: the batch runs in chunks, the workspace is sized for one chunk
    big = (65535, 1, 1024, 1024, 1024, 1024)
    assert lib.cf_warp_backward_det_workspace_bytes(*big) == _workspace_formula(*big) < 24 * 2 ** 32
    # the codes warp of 64 x 240x320 items
    assert abs(lib.cf_warp_backward_det_workspace_bytes(64, 128, 240, 320, 480, 640) / 1e9 - 0.46) < 0.01
    assert lib.cf_warp_backward_det_workspace_bytes(0, 3, 8, 8, 8, 8) == 0
    assert lib.cf_warp_backward_det_workspace_bytes(2, 0, 8, 8, 8, 8) == 0
    assert lib.cf_warp_backward_det_workspace_bytes(2, 3, 8, 8, 9, 9) == 0      # flow neither equal nor twice the size
    assert lib.cf_warp_backward_det_workspace_bytes(2, 3, 0, 8, 0, 8) == 0


def test_flag_resolves_the_voxel_mode():
    from cistaflow_b200 import event_process as ep
    assert ep.resolve_mode(None) == ep.DEFAULT_MODE
    assert ep.resolve_mode("atomic_l2") == "atomic_l2"
    with deterministic_algorithms():
        assert ep.resolve_mode(None) == "deterministic"
        assert ep.resolve_mode("atomic") == "atomic"          # an explicit mode wins
        with pytest.raises(RuntimeError, match="deterministic implementation"):
            ep.events_to_voxel_grid_packed(torch.zeros(4, dtype=torch.int64), torch.tensor([0, 4]), 5, 8, 8)
    with deterministic_algorithms(warn_only=True):
        assert torch.is_deterministic_algorithms_warn_only_enabled()
    assert ep.resolve_mode(None) == ep.DEFAULT_MODE
    assert not torch.is_deterministic_algorithms_warn_only_enabled()


# ----------------------------------------------------------------------------------------------------- GPU ---
def _warp_case(kind, shape, mode):
    """(image-or-codes, flow, grad_out, half) as float32 arrays; flow at twice the image size for the 'half' kinds."""
    from cistaflow_b200 import synth
    B, C, H, W = shape
    rng = np.random.default_rng(5)
    img = rng.standard_normal(shape).astype(np.float32)
    gout = rng.standard_normal(shape).astype(np.float32)
    if kind in ("half", "half_odd"):
        fH, fW = 2 * H + (kind == "half_odd"), 2 * W + (kind == "half_odd")
        _, _, flow = synth.warp_inputs(B, fH, fW, seed=9, code_channels=8, flow_kind="smooth")
        return img, flow, gout, True
    if kind == "converge":
        # every pixel samples the same point (7.3, 5.6): 4*H*W records in four buckets
        ys, xs = np.meshgrid(np.arange(H, dtype=np.float32), np.arange(W, dtype=np.float32), indexing="ij")
        s = -1.0 if mode == "forward" else 1.0
        flow = np.stack([(7.3 - xs) / s, (5.6 - ys) / s])[None].repeat(B, 0).astype(np.float32)
        return img, flow, gout, False
    _, _, flow = synth.warp_inputs(B, H, W, seed=8, code_channels=8, flow_kind=kind)
    flow[0, :, 0, 0] = [-3.0 * W, 2.5 * H]      # far outside: reflected several times
    return img, flow, gout, False


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["forward", "backward"])
@pytest.mark.parametrize("kind,shape", [
    ("noise", (2, 3, 18, 22)), ("smooth", (1, 128, 90, 120)), ("smooth", (2, 5, 31, 45)),
    ("noise", (2, 40, 24, 36)),                          # C not a multiple of the 32-channel groups
    ("half", (2, 16, 18, 24)), ("half_odd", (2, 16, 18, 24)),   # fused x0.5 down-sampling, even and odd flow
    ("converge", (2, 6, 20, 28)),
])
def test_det_warp_backward_matches_autograd_of_the_reference_ops(cuda_device, deterministic, mode, kind, shape):
    """Gradients of forwardWarp / backWarp under the flag against torch.autograd through the oracle port on CPU, at
    the tolerances of the atomic path's test."""
    import cistaflow_b200 as cf
    from oracle import ref_port
    img, flow, gout, half = _warp_case(kind, shape, mode)
    ri, rf = torch.from_numpy(img).requires_grad_(), torch.from_numpy(flow).requires_grad_()
    ref_port.warp(ri, ref_port.downsample_flow(rf) if half else rf, mode).backward(torch.from_numpy(gout))
    di, df = dev_t(img, cuda_device).requires_grad_(), dev_t(flow, cuda_device).requires_grad_()
    B, C, H, W = shape
    out = (cf.forwardWarp(W, H) if mode == "forward" else cf.backWarp(W, H))(di, df)
    out.backward(dev_t(gout, cuda_device))
    assert last_kernel() == DET_KERNELS[1 if half else 0]
    scale_i = max(1.0, float(ri.grad.abs().max()))
    scale_f = max(1.0, float(rf.grad.abs().max()))
    assert (di.grad.cpu() - ri.grad).abs().max().item() <= 1e-4 * scale_i
    err = (df.grad.cpu() - rf.grad).abs()
    assert err.max().item() <= 2e-3 * scale_f, err.max().item()
    assert (err > 1e-4 * scale_f).float().mean().item() < 1e-3


def _det_c_call(lib, gout, img, flow, gi, gf, sign, ws, stream):
    from cistaflow_b200 import _lib
    B, C, H, W = img.shape
    return lib.cf_warp_backward_det(gout.data_ptr(), img.data_ptr(), flow.data_ptr(), _lib.ptr(gi), _lib.ptr(gf), B, C,
                                    H, W, flow.shape[2], flow.shape[3], sign, ws.data_ptr(), ws.numel(), stream)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,half", [((3, 40, 64, 96), False), ((2, 48, 40, 56), True)])
def test_det_warp_backward_is_bitwise_reproducible(cuda_device, shape, half):
    """Three calls, a side stream and a graph-captured call of the C entry point give the same bits; outputs are
    pre-filled with NaN, so an element left unwritten fails."""
    import cistaflow_b200 as cf
    from cistaflow_b200 import _lib, synth
    B, C, H, W = shape
    rng = np.random.default_rng(11)
    img = dev_t(rng.standard_normal(shape).astype(np.float32), cuda_device)
    gout = dev_t(rng.standard_normal(shape).astype(np.float32), cuda_device)
    fH, fW = (2 * H, 2 * W) if half else (H, W)
    flow = dev_t(synth.warp_inputs(B, fH, fW, seed=12, code_channels=8, flow_kind="noise")[2], cuda_device)

    def grads():
        di, df = img.clone().requires_grad_(), flow.clone().requires_grad_()
        cf.warp(di, df, -1.0).backward(gout)
        return di.grad, df.grad

    with deterministic_algorithms():
        runs = [grads() for _ in range(3)]
        assert last_kernel() == DET_KERNELS[1 if half else 0]
        side = torch.cuda.Stream(cuda_device)
        side.wait_stream(torch.cuda.current_stream(cuda_device))
        with torch.cuda.stream(side):
            runs.append(grads())
        torch.cuda.current_stream(cuda_device).wait_stream(side)
    for gi, gf in runs[1:]:
        assert torch.equal(gi, runs[0][0]) and torch.equal(gf, runs[0][1])

    lib = _lib.load()
    ws = torch.empty(lib.cf_warp_backward_det_workspace_bytes(B, C, H, W, fH, fW), dtype=torch.uint8, device=cuda_device)
    gi = torch.full_like(img, float("nan"))
    gf = torch.full_like(flow, float("nan"))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        rc = _det_c_call(lib, gout, img, flow, gi, gf, -1.0, ws, torch.cuda.current_stream(cuda_device).cuda_stream)
    assert rc == 0, lib.cf_last_error()
    graph.replay()
    torch.cuda.synchronize(cuda_device)
    assert torch.equal(gi, runs[0][0]) and torch.equal(gf, runs[0][1])

    # the flag restored: the default (atomic) adjoint again, agreeing to summation order
    gi_a, gf_a = grads()
    assert last_kernel() == "warp_backward_kernel"
    assert (gi_a - gi).abs().max().item() <= 1e-5 * max(1.0, gi.abs().max().item())
    assert (gf_a - gf).abs().max().item() <= 1e-4 * max(1.0, gf.abs().max().item())


@pytest.mark.gpu
def test_det_warp_backward_c_errors(cuda_device):
    from cistaflow_b200 import _lib
    lib = _lib.load()
    img = torch.zeros(1, 2, 8, 8, device=cuda_device)
    flow = torch.zeros(1, 2, 8, 8, device=cuda_device)
    gi, gf = torch.empty_like(img), torch.empty_like(flow)
    nbytes = lib.cf_warp_backward_det_workspace_bytes(1, 2, 8, 8, 8, 8)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=cuda_device)
    s = torch.cuda.current_stream(cuda_device).cuda_stream
    assert _det_c_call(lib, img, img, flow, gi, gf, -1.0, ws, s) == 0
    assert lib.cf_warp_backward_det(img.data_ptr(), img.data_ptr(), flow.data_ptr(), gi.data_ptr(), gf.data_ptr(),
                                    1, 2, 8, 8, 8, 8, -1.0, ws.data_ptr(), nbytes - 1, s) == -5      # CF_ERR_WORKSPACE
    assert lib.cf_warp_backward_det(img.data_ptr(), img.data_ptr(), flow.data_ptr(), gi.data_ptr(), gf.data_ptr(),
                                    1, 2, 8, 8, 8, 8, -1.0, None, 0, s) == -5
    assert _det_c_call(lib, img, img, flow, None, None, -1.0, ws, s) == -2                     # CF_ERR_NULL
    assert lib.cf_warp_backward_det(img.data_ptr(), None, flow.data_ptr(), None, gf.data_ptr(),
                                    1, 2, 8, 8, 8, 8, -1.0, ws.data_ptr(), nbytes, s) == -2       # grad_flow needs img
    assert _det_c_call(lib, img, img, flow, gi, gf, 0.5, ws, s) == -1                          # CF_ERR_INVALID_ARG
    assert lib.cf_warp_backward_det(img.data_ptr(), img.data_ptr(), flow.data_ptr(), gi.data_ptr(), gf.data_ptr(),
                                    1, 2, 8, 8, 9, 9, -1.0, ws.data_ptr(), nbytes, s) == -1
    torch.cuda.synchronize(cuda_device)


def _lookup_qt(levels, radius):
    """The queries per CTA cf_corr_lookup_backward picks (its smem_bytes, 200 KB cap)."""
    K = 2 * radius + 1
    P = K + 1
    smem = lambda qt: (qt * (((levels * P * P) | 1) + ((levels * K * K) | 1)) + 2 * qt + 2 * 256) * 4   # noqa: E731
    return 16 if smem(16) <= 200 * 1024 else 8


@pytest.mark.gpu
@pytest.mark.parametrize("B,h,w,levels,radius,qt", [(2, 24, 32, 4, 4, 16), (1, 32, 32, 6, 8, 8)])
def test_corr_coordinate_gradient_is_bitwise_reproducible(cuda_device, B, h, w, levels, radius, qt):
    import cistaflow_b200 as cf
    assert _lookup_qt(levels, radius) == qt
    gen = torch.Generator(device="cpu").manual_seed(21)
    f1, f2 = (torch.randn(B, 64, h, w, generator=gen).to(cuda_device) for _ in range(2))
    coords = (cf.coords_grid(B, h, w) + 3.0 * torch.randn(B, 2, h, w, generator=gen)).to(cuda_device)
    blk = cf.CorrBlock(f1, f2, num_levels=levels, radius=radius)
    gout = torch.randn(B, levels * (2 * radius + 1) ** 2, h, w, generator=gen).to(cuda_device)
    grads = []
    for _ in range(3):
        c = coords.clone().requires_grad_()
        blk(c).backward(gout)
        assert last_kernel() == "corr_lookup_backward_kernel"
        grads.append(c.grad)
    assert torch.isfinite(grads[0]).all() and grads[0].abs().max().item() > 0
    for g in grads[1:]:
        assert torch.equal(g, grads[0])


@pytest.mark.gpu
def test_flag_selects_the_deterministic_voxel_mode(cuda_device):
    import cistaflow_b200 as cf
    from cistaflow_b200 import synth
    H, W = 48, 64
    ev, off = synth.event_windows(3, 3000, H, W, seed=31)
    ev_d, off_d = dev_t(ev, cuda_device), dev_t(off, cuda_device)
    det = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, W, H, flavour="numpy", mode="deterministic")
    packed = cf.pack_events(ev_d, off_d)
    ref_packed = cf.events_to_voxel_grid_packed(packed, off_d, 5, W, H)
    win = ev[:off[1]]
    mv = dict(xs=win[:, 1], ys=win[:, 2], ts=win[:, 0], ps=(win[:, 3] > 0).astype(np.float64), B=5, sensor_size=(H, W))
    mv_det = cf.events_to_voxel_torch(**mv, mode="deterministic")
    with deterministic_algorithms():
        got = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, W, H, flavour="numpy")
        assert last_kernel() == "det_accumulate_kernel"
        assert torch.equal(got.view(torch.int32), det.view(torch.int32))
        assert torch.equal(cf.events_to_voxel_torch(**mv).view(torch.int32), mv_det.view(torch.int32))   # mvsec_utils
        atom = cf.events_to_voxel_grid_batched(ev_d, off_d, 5, W, H, flavour="numpy", mode="atomic")
        assert last_kernel() == "voxel_scatter_atomic_kernel"                # an explicit mode is honoured
        assert (atom - det).abs().max().item() <= 1e-5 * (det.abs().max().item() + 1)
        with pytest.raises(RuntimeError, match="deterministic implementation"):
            cf.events_to_voxel_grid_packed(packed, off_d, 5, W, H)
    with deterministic_algorithms(warn_only=True):
        with pytest.warns(UserWarning, match="deterministic implementation"):
            out = cf.events_to_voxel_grid_packed(packed, off_d, 5, W, H)
    assert (out - ref_packed).abs().max().item() <= 1e-5 * (ref_packed.abs().max().item() + 1)


def _training_step(dev, inputs):
    """CorrBlock build + 6 lookups + the frame and codes warps + a scalar loss + backward(); returns every gradient."""
    import cistaflow_b200 as cf
    f1, f2, frame, codes, flow, target, wl = (t.clone().requires_grad_(t.is_floating_point() and k < 5)
                                              for k, t in enumerate(inputs))
    B, _, h, w = f1.shape
    blk = cf.CorrBlock(f1, f2, num_levels=4, radius=4)
    coords0 = cf.coords_grid(B, h, w, device=dev) + 0.5 * flow[:, :, ::2, ::2]
    loss = 0.0
    for k in range(6):
        corr = blk(coords0 + (k + 1) / 6.0 * flow[:, :, ::2, ::2])
        loss = loss + (corr * wl[k]).mean()
    warped = cf.forwardWarp(frame.shape[3], frame.shape[2])(frame, flow)
    warped_codes = cf.warp(codes, flow, -1.0)                  # codes at half resolution: the fused x0.5 flow
    loss = loss + ((warped - target) ** 2).mean() + 1e-3 * (warped_codes ** 2).sum()
    loss.backward()
    return [t.grad for t in (f1, f2, frame, codes, flow)]


@pytest.mark.gpu
def test_training_step_replay_is_bitwise_reproducible(cuda_device):
    gen = torch.Generator(device="cpu").manual_seed(41)
    B, D, h, w = 2, 64, 24, 32
    H, W = 2 * h, 2 * w
    inputs = [torch.randn(B, D, h, w, generator=gen), torch.randn(B, D, h, w, generator=gen),
              torch.rand(B, 1, H, W, generator=gen), torch.randn(B, 16, h, w, generator=gen),
              3.0 * torch.randn(B, 2, H, W, generator=gen), torch.rand(B, 1, H, W, generator=gen),
              torch.randn(6, 1, 4 * 81, h, w, generator=gen)]
    inputs = [t.to(cuda_device) for t in inputs]
    with deterministic_algorithms():
        first = _training_step(cuda_device, inputs)
        second = _training_step(cuda_device, inputs)
    for a, b in zip(first, second):
        assert a is not None and torch.isfinite(a).all()
        assert torch.equal(a, b)
