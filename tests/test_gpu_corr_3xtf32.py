"""CF_CORR_3XTF32: the correlation pyramid on the tensor cores with split operands (x = hi + lo, both exact TF32 values,
three kind::tf32 MMAs per K step), held to the 1e-5 normwise bound of the fp32 SIMT kernel.

Also the only fp32-accurate check of the default ``auto`` path at the headline launch (64 x 256 x 60x80), where it runs
on fp16 operand copies."""
import numpy as np
import pytest
import torch

import cistaflow_b200 as cf
from cistaflow_b200 import _lib, synth
from oracle import ref_port

TOL = 1e-5   # what the fp32 SIMT path is held to


def dev_t(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def last_kernel():
    return _lib.load().cf_last_kernel().decode()


def corr_err(got, ref):
    """Normwise error max|err| / max|ref|, after asserting that >= 95 % of the elements satisfy
    |err| <= 1e-3 * (|ref| + rms(ref)) (SURVEY.md H3)."""
    g, r = np.asarray(got).astype(np.float64), np.asarray(ref).astype(np.float64)
    err = np.abs(g - r)
    rms = float(np.sqrt(np.mean(r * r))) if r.size else 0.0
    frac = float((err <= 1e-3 * (np.abs(r) + rms)).mean()) if err.size else 1.0
    assert frac >= 0.95, f"only {frac:.4f} of the elements within 1e-3*(|ref|+rms)"
    return float(err.max() / max(np.abs(r).max(), 1e-30))


def corr_err_dev(got, ref, rows=4096):
    """corr_err on the device, in float64 chunks of rows (the headline's level 0 is 5.9 GB)."""
    g2, r2 = got.reshape(got.shape[0], -1), ref.reshape(ref.shape[0], -1)
    sq, rmax = 0.0, 0.0
    for i in range(0, r2.shape[0], rows):
        r = r2[i:i + rows].double()
        sq += float((r * r).sum())
        rmax = max(rmax, float(r.abs().max()))
    rms = (sq / r2.numel()) ** 0.5
    emax, inside = 0.0, 0
    for i in range(0, r2.shape[0], rows):
        r, g = r2[i:i + rows].double(), g2[i:i + rows].double()
        e = (g - r).abs()
        emax = max(emax, float(e.max()))
        inside += int((e <= 1e-3 * (r.abs() + rms)).sum())
    frac = inside / r2.numel()
    assert frac >= 0.95, f"only {frac:.4f} of the elements within 1e-3*(|ref|+rms)"
    return emax / max(rmax, 1e-30)


def exact_pyramid(f1, f2, levels):
    """The pyramid in float64 on the device: the contraction the fp32 reference approximates."""
    B, D, h, w = f1.shape
    N = h * w
    vol = torch.matmul(f1.double().reshape(B, D, N).transpose(1, 2), f2.double().reshape(B, D, N)) / float(D) ** 0.5
    pyr = [vol.reshape(B * N, 1, h, w)]
    for _ in range(levels - 1):
        pyr.append(torch.nn.functional.avg_pool2d(pyr[-1], 2, stride=2))
    return pyr


def normwise(got, ref):
    return float((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


# ------------------------------------------------------------------------------------------------------ CPU ---
def test_workspace_bytes_and_precision_name():
    import __graft_entry__ as entry
    entry.build()
    lib = _lib.load()
    for (B, D, h, w) in ((1, 32, 1, 1), (2, 256, 60, 80), (64, 256, 60, 80), (1, 48, 5, 3), (3, 64, 15, 20)):
        per_map = -(-(B * D * h * w * 4) // 256) * 256
        assert lib.cf_corr_workspace_bytes(B, D, h, w, 4, _lib.CORR_3XTF32) == 4 * per_map
        assert lib.cf_corr_workspace_bytes(B, D, h, w, 4, _lib.CORR_TF32) == 0
        assert lib.cf_corr_workspace_bytes(B, D, h, w, 4, _lib.CORR_FP32) == 0
    assert lib.cf_corr_workspace_bytes(0, 256, 60, 80, 4, _lib.CORR_3XTF32) == 0
    assert cf.corr._PREC["3xtf32"] == _lib.CORR_3XTF32


# ------------------------------------------------------------------------------------------------------ GPU ---
@pytest.mark.gpu
def test_golden(golden, cuda_device):
    g = golden("corr")
    f1, f2 = dev_t(g["fmap1"], cuda_device), dev_t(g["fmap2"], cuda_device)
    cf.build_pyramid(f1, f2, 2, precision="3xtf32")   # two levels: the fused kernel is the last launch
    assert last_kernel() == "corr_tc_kernel<3xtf32>"
    blk = cf.CorrBlock(f1, f2, num_levels=4, radius=4, precision="3xtf32")
    for l in range(4):
        assert tuple(blk.corr_pyramid[l].shape) == g[f"pyr{l}"].shape
        assert corr_err(*g.pick(f"pyr{l}", blk.corr_pyramid[l].cpu().numpy())) <= TOL, f"level {l}"
    out = blk(dev_t(g["coords"], cuda_device))
    assert corr_err(*g.pick("lookup", out.cpu().numpy())) <= TOL
    vol = cf.CorrBlock.corr(f1, f2, precision="3xtf32")
    assert tuple(vol.shape) == (1, 16, 24, 1, 16, 24)
    assert corr_err(*g.pick("pyr0", vol.reshape(g["pyr0"].shape).cpu().numpy())) <= TOL


@pytest.mark.gpu
def test_golden_odd_sizes(golden, cuda_device):
    """15x20 maps (odd h: the un-fused tensor-core path), 3 levels, radius 3."""
    g = golden("corr")
    f1, f2 = dev_t(g["odd/fmap1"], cuda_device), dev_t(g["odd/fmap2"], cuda_device)
    cf.build_pyramid(f1, f2, 1, precision="3xtf32")
    assert last_kernel() == "corr_tc_kernel<3xtf32>"
    blk = cf.CorrBlock(f1, f2, num_levels=3, radius=3, precision="3xtf32")
    for l in range(3):
        assert corr_err(*g.pick(f"odd/pyr{l}", blk.corr_pyramid[l].cpu().numpy())) <= TOL, f"level {l}"
    assert corr_err(*g.pick("odd/lookup", blk(dev_t(g["odd/coords"], cuda_device)).cpu().numpy())) <= TOL
    exact = exact_pyramid(f1, f2, 3)
    t32 = cf.build_pyramid(f1, f2, 3, precision="tf32")
    for l in range(3):
        assert 10 * normwise(blk.corr_pyramid[l], exact[l]) <= normwise(t32[l], exact[l]), f"level {l}"


# 24x32 deep fusion (levels 0-3 in the epilogue), 36x44 per-atom boxes (N % 32 != 0, level 1 fused), 60x80 pair2 (BN = 160),
# 80x124 BN = 248 (not a multiple of 32: per-atom fmap2 boxes), 16x24 deep fusion with two items
@pytest.mark.gpu
@pytest.mark.parametrize("h,w,batch", [(180, 240, 8), (260, 346, 1), (480, 640, 1), (624, 970, 1), (128, 192, 2)])
def test_config_shapes_vs_oracle(cuda_device, h, w, batch):
    f1, f2, coords = synth.corr_inputs(batch, h, w, seed=9)
    a, b = dev_t(f1, cuda_device), dev_t(f2, cuda_device)
    cf.build_pyramid(a, b, 2, precision="3xtf32")
    assert last_kernel() == "corr_tc_kernel<3xtf32>"
    ref_pyr = ref_port.corr_pyramid(torch.from_numpy(f1), torch.from_numpy(f2), 4)
    blk = cf.CorrBlock(a, b, precision="3xtf32")
    for l in range(4):
        assert tuple(blk.corr_pyramid[l].shape) == tuple(ref_pyr[l].shape)
        assert corr_err(blk.corr_pyramid[l].cpu().numpy(), ref_pyr[l].numpy()) <= TOL, f"level {l}"
    ref_out = ref_port.corr_lookup(ref_pyr, torch.from_numpy(coords), 4)
    assert corr_err(blk(dev_t(coords, cuda_device)).cpu().numpy(), ref_out.numpy()) <= TOL


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,B,scale", [(192, 256, 2, 1.0), (288, 352, 1, 1.0), (192, 256, 1, 3.0e6), (192, 256, 1, 1.0e-9)])
def test_split_error_ten_times_below_tf32(cuda_device, H, W, B, scale):
    """Against a float64 contraction the split operands are >= 10x closer than TF32 operands, also for inputs far outside
    the unit range (3-D operand boxes at 24x32, per-atom boxes at 36x44)."""
    f1, f2, _ = synth.corr_inputs(B, H, W, 9)
    a, b = dev_t(f1, cuda_device) * scale, dev_t(f2, cuda_device)
    exact = exact_pyramid(a, b, 4)
    x3 = cf.build_pyramid(a, b, 4, precision="3xtf32")
    t32 = cf.build_pyramid(a, b, 4, precision="tf32")
    for l in range(4):
        e3, et = normwise(x3[l], exact[l]), normwise(t32[l], exact[l])
        assert e3 <= TOL and 10 * e3 <= et, (l, e3, et)


@pytest.mark.gpu
def test_zero_map_gives_zero_pyramid(cuda_device):
    z = torch.zeros(1, 256, 24, 32, device=cuda_device)
    for lvl in cf.build_pyramid(z, dev_t(synth.corr_inputs(1, 192, 256, 1)[1], cuda_device), 4, precision="3xtf32"):
        assert not lvl.any()


@pytest.mark.gpu
def test_headline_launch(cuda_device):
    """64 x 256 x 60x80: 3xTF32 against float64 on a fixed sample of query rows, and the default path (fp16 operand
    copies at this launch) against 3xTF32 on every level."""
    B, D, h, w = 64, 256, 60, 80
    N = h * w
    gen = torch.Generator(device=cuda_device).manual_seed(64)
    a = torch.randn(B, D, h, w, device=cuda_device, generator=gen)
    b = torch.randn(B, D, h, w, device=cuda_device, generator=gen)
    x3 = cf.build_pyramid(a, b, 4, precision="3xtf32")
    l0 = x3[0].view(B, N, N)
    rows = torch.randint(0, N, (256,), device=cuda_device, generator=gen)
    for item in (0, 17, 40, 63):
        exact = (a[item].reshape(D, N)[:, rows].double().T @ b[item].reshape(D, N).double()) / float(D) ** 0.5
        assert normwise(l0[item, rows], exact) <= TOL, item
        pooled = torch.nn.functional.avg_pool2d(exact.view(-1, 1, h, w), 2, stride=2)
        assert normwise(x3[1].view(B, N, -1)[item, rows], pooled.view(len(rows), -1)) <= TOL, item
    auto = cf.build_pyramid(a, b, 4, precision="auto")
    for l in range(4):
        assert corr_err_dev(auto[l], x3[l]) <= 1e-3, f"level {l}"


@pytest.mark.gpu
def test_deterministic_and_graph_capture(cuda_device):
    f1, f2, _ = synth.corr_inputs(4, 480, 640, seed=5)
    a, b = dev_t(f1, cuda_device), dev_t(f2, cuda_device)
    first = cf.build_pyramid(a, b, 4, precision="3xtf32")
    second = cf.build_pyramid(a, b, 4, precision="3xtf32")
    for x, y in zip(first, second):
        assert torch.equal(x, y)
    out = [torch.empty_like(t) for t in first]
    s = torch.cuda.Stream(cuda_device)
    with torch.cuda.stream(s):
        cf.build_pyramid(a, b, 4, precision="3xtf32", out=out)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            cf.build_pyramid(a, b, 4, precision="3xtf32", out=out)
        for t in out:
            t.fill_(float("nan"))
        g.replay()
        torch.cuda.synchronize()
    for x, y in zip(out, first):
        assert torch.equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,levels,radius", [(16, 24, 4, 4), (15, 20, 3, 3)])
def test_corr_block_backward_matches_autograd_of_the_reference_ops(cuda_device, h, w, levels, radius):
    rng = np.random.default_rng(12)
    B, D = 2, 64
    f1 = rng.standard_normal((B, D, h, w)).astype(np.float32)
    f2 = rng.standard_normal((B, D, h, w)).astype(np.float32)
    ys, xs = np.meshgrid(np.arange(h, dtype=np.float32), np.arange(w, dtype=np.float32), indexing="ij")
    coords = (np.stack([xs, ys])[None] + 2.5 * rng.standard_normal((B, 2, h, w))).astype(np.float32)
    coords[0, :, 0, 0] = [-7.3, h + 5.2]     # window partly / wholly outside the map
    k = 2 * radius + 1
    gout = rng.standard_normal((B, levels * k * k, h, w)).astype(np.float32)
    rf1, rf2, rc = (torch.from_numpy(x).requires_grad_() for x in (f1, f2, coords))
    ref_port.corr_lookup(ref_port.corr_pyramid(rf1, rf2, levels), rc, radius).backward(torch.from_numpy(gout))
    df1, df2, dc = (dev_t(x, cuda_device).requires_grad_() for x in (f1, f2, coords))
    blk = cf.CorrBlock(df1, df2, num_levels=levels, radius=radius, precision="3xtf32")
    out = blk(dc)
    assert out.requires_grad
    out.backward(dev_t(gout, cuda_device))
    for got, ref, name in ((df1.grad, rf1.grad, "fmap1"), (df2.grad, rf2.grad, "fmap2")):
        assert corr_err(got.cpu().numpy(), ref.numpy()) <= 1e-4, name
    err = (dc.grad.cpu() - rc.grad).abs()     # the coordinate gradient jumps on pixel boundaries: compare away from them
    scale = float(rc.grad.abs().max())
    assert err.max().item() <= 2e-3 * scale and (err > 1e-4 * scale).float().mean().item() < 1e-3


@pytest.mark.gpu
def test_errors_through_the_c_abi(cuda_device):
    lib = _lib.load()
    stream = _lib.stream_ptr(cuda_device)

    def build(a, b, ws_ptr, ws_bytes):
        B, D, h, w = a.shape
        pyr = [torch.empty((B * h * w, 1, h >> l, w >> l), device=cuda_device) for l in range(4)]
        rc = lib.cf_corr_build(a.data_ptr(), b.data_ptr(), B, D, h, w, 4, _lib.pointer_array(pyr), _lib.CORR_3XTF32,
                               ws_ptr, ws_bytes, stream)
        return rc, pyr

    f1, f2, _ = synth.corr_inputs(1, 192, 256, 3)
    a, b = dev_t(f1, cuda_device), dev_t(f2, cuda_device)
    need = lib.cf_corr_workspace_bytes(1, 256, 24, 32, 4, _lib.CORR_3XTF32)
    ws = torch.empty(need + 256, dtype=torch.uint8, device=cuda_device)
    rc, _ = build(a, b, None, 0)
    assert rc == -5 and "3XTF32" in lib.cf_last_error().decode()
    rc, _ = build(a, b, ws.data_ptr(), need - 16)
    assert rc == -5 and "3XTF32" in lib.cf_last_error().decode()
    rc, _ = build(a, b, ws.data_ptr() + 4, need)
    assert rc == -3
    rc, pyr = build(a, b, ws.data_ptr(), need)
    assert rc == 0
    ref = cf.build_pyramid(a, b, 4, precision="fp32")
    for l in range(4):
        assert corr_err(pyr[l].cpu().numpy(), ref[l].cpu().numpy()) <= TOL

    # D = 48: no tensor-core tiling -- CF_ERR_UNSUPPORTED from C, the fp32 kernel from Python
    g = torch.Generator(device=cuda_device).manual_seed(48)
    a48 = torch.randn(2, 48, 24, 32, device=cuda_device, generator=g)
    b48 = torch.randn(2, 48, 24, 32, device=cuda_device, generator=g)
    need48 = lib.cf_corr_workspace_bytes(2, 48, 24, 32, 4, _lib.CORR_3XTF32)
    ws48 = torch.empty(need48, dtype=torch.uint8, device=cuda_device)
    rc, _ = build(a48, b48, ws48.data_ptr(), need48)
    assert rc == -7
    got = cf.build_pyramid(a48, b48, 4, precision="3xtf32")
    ref = cf.build_pyramid(a48, b48, 4, precision="fp32")
    for x, y in zip(got, ref):
        assert torch.equal(x, y)
