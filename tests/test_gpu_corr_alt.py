"""AlternateCorrBlock: the on-demand correlation lookup (include/cistaflow_altcorr.h, csrc/corr_alt.cu).

The lookup must equal CorrBlock's (the pyramid of the all-pairs volume, sampled by cf_corr_lookup) up to fp32
summation order and operand rounding, since avg_pool2d is linear.  It is held to the golden fixtures of the
reference, to replays of the running models' coordinates, and to a float64 evaluation of the same definition on the
device, at 1e-5 (fp32) and 1e-3 (tf32) normwise.
"""
import ctypes
import inspect
import os
import re
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONFIG_SHAPES = [(8, 24, 32), (64, 36, 44), (64, 60, 80), (1, 80, 124), (2, 92, 160)]   # (B, h, w) at D = 256


def _header_symbols(name):
    text = open(os.path.join(ROOT, "include", name)).read()
    return sorted(re.findall(r"CF_API\s+[\w\s\*]+?\b(cf_\w+)\s*\(", text))


# ----------------------------------------------------------------------------------------------------- CPU ---
def test_altcorr_header_matches_ctypes_table_and_library():
    import cistaflow_b200 as cf
    from cistaflow_b200 import _lib
    syms = _header_symbols("cistaflow_altcorr.h")
    assert syms == sorted(["cf_corr_alt_workspace_bytes", "cf_corr_alt_prepare", "cf_corr_alt_lookup"])
    assert syms == sorted(_lib.ALTCORR_SYMBOLS)
    assert len(_header_symbols("cistaflow.h")) == 26 and sorted(_lib.SYMBOLS) == _header_symbols("cistaflow.h")
    lib = cf.load_library()
    for name in syms:
        assert getattr(lib, name).restype == _lib.ALTCORR_SYMBOLS[name][0]


def test_altcorr_workspace_formula():
    import cistaflow_b200 as cf
    from cistaflow_b200 import _lib
    lib = cf.load_library()
    for B, h, w in CONFIG_SHAPES:
        for D in (256, 48):
            for prec in (_lib.CORR_AUTO, _lib.CORR_TF32, _lib.CORR_FP32):
                n = lib.cf_corr_alt_workspace_bytes(B, D, h, w, 4, prec)
                assert 2 * B * D * h * w * 4 <= n <= 3 * B * D * h * w * 4 + 256 * 5
    assert lib.cf_corr_alt_workspace_bytes(0, 256, 60, 80, 4, _lib.CORR_AUTO) == 0
    assert lib.cf_corr_alt_workspace_bytes(64, 256, 60, 80, 4, _lib.CORR_F16) == 0      # unsupported precision
    # headline: about 0.73 GB, against 7.8 GB for the 4-level pyramid
    assert abs(lib.cf_corr_alt_workspace_bytes(64, 256, 60, 80, 4, _lib.CORR_AUTO) / 1e9 - 0.73) < 0.01


def test_install_rebinds_alternate_corr_block(monkeypatch):
    import importlib
    import cistaflow_b200 as cf
    inst = importlib.import_module("cistaflow_b200.install")
    sentinel = object()
    raft_corr = types.ModuleType("DCEIFlow.core.corr.raft_corr")
    raft_corr.CorrBlock = raft_corr.AlternateCorrBlock = sentinel
    eraft_corr = types.ModuleType("ERAFT.corr")
    eraft_corr.CorrBlock = sentinel          # has no AlternateCorrBlock: none is added
    for m in (raft_corr, eraft_corr):
        monkeypatch.setitem(sys.modules, m.__name__, m)
    done = inst.install(import_missing=False, parts=("corr",))
    assert raft_corr.AlternateCorrBlock is cf.AlternateCorrBlock and raft_corr.CorrBlock is cf.CorrBlock
    assert "DCEIFlow.core.corr.raft_corr.AlternateCorrBlock" in done
    assert not hasattr(eraft_corr, "AlternateCorrBlock")
    inst.uninstall()
    assert raft_corr.AlternateCorrBlock is sentinel


def test_alternate_corr_block_rejects_unknown_precision():
    import cistaflow_b200 as cf
    with pytest.raises(ValueError, match="precision 'bf16'"):
        cf.AlternateCorrBlock(None, None, precision="bf16")


def test_alternate_corr_block_signature_mirrors_corr_block():
    import cistaflow_b200 as cf
    p = list(inspect.signature(cf.CorrBlock.__init__).parameters.values())[1:5]
    q = list(inspect.signature(cf.AlternateCorrBlock.__init__).parameters.values())[1:5]
    assert [(x.name, x.default) for x in q] == [(x.name, x.default) for x in p]
    assert [x.name for x in q] == ["fmap1", "fmap2", "num_levels", "radius"]


# ----------------------------------------------------------------------------------------------------- GPU ---
def _torch():
    import torch
    return torch


def dev_t(a, device):
    torch = _torch()
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def corr_err(got, ref):
    from test_gpu_parity import corr_err as ce
    return ce(got, ref)


def normwise(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    return float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30))


def last_kernel():
    from cistaflow_b200 import _lib
    return _lib.load().cf_last_kernel().decode()


def feature_maps(B, D, h, w, device, seed):
    torch = _torch()
    g = torch.Generator(device=device).manual_seed(seed)
    return (torch.randn(B, D, h, w, device=device, generator=g), torch.randn(B, D, h, w, device=device, generator=g))


def smooth_coords(B, h, w, device, seed, sigma=0.5):
    """coords_grid + an affine flow field + N(0, sigma^2)."""
    import cistaflow_b200 as cf
    torch = _torch()
    g = torch.Generator(device=device).manual_seed(seed)
    grid = cf.coords_grid(B, h, w, device=device)
    xs, ys = grid[:, 0] - w / 2, grid[:, 1] - h / 2
    flow = torch.stack([0.04 * xs - 0.03 * ys + 2.7, 0.02 * xs + 0.05 * ys - 1.6], 1)
    return grid + flow + sigma * torch.randn(B, 2, h, w, device=device, generator=g)


def noise_coords(B, h, w, device, seed, sigma=5.0):
    import cistaflow_b200 as cf
    torch = _torch()
    g = torch.Generator(device=device).manual_seed(seed)
    return cf.coords_grid(B, h, w, device=device) + sigma * torch.randn(B, 2, h, w, device=device, generator=g)


def reference_f64(f1, f2, coords, levels, radius, n_samples=2048, seed=0):
    """The on-demand definition in float64 on the device for sampled queries: level l at target (y, x) is
    <fmap1[:, q], avg_pool2d^l(fmap2)[:, y, x]> / sqrt(D), zero outside the map, sampled bilinearly around
    coords / 2^l with the transposed window.  Returns (sample index tuple, [S, levels*(2r+1)^2])."""
    torch = _torch()
    F = torch.nn.functional
    B, D, h, w = f1.shape
    g = torch.Generator(device=f1.device).manual_seed(seed)
    S = min(n_samples, B * h * w)
    flat = torch.randperm(B * h * w, device=f1.device, generator=g)[:S]
    bs, ys, xs = flat // (h * w), (flat // w) % h, flat % w
    q1 = f1.double()[bs, :, ys, xs]                              # [S, D]
    c = coords.double()[bs, :, ys, xs].clamp(-1e6, 1e6)          # [S, 2]
    K, P = 2 * radius + 1, 2 * radius + 2
    lvl = f2.double()
    outs = []
    for l in range(levels):
        if l:
            lvl = F.avg_pool2d(lvl, 2, 2)
        hl, wl = lvl.shape[2:]
        s = c / 2 ** l
        fl = torch.floor(s)
        frac = s - fl
        base = fl.long() - radius
        off = torch.arange(P, device=f1.device)
        X, Y = base[:, 0:1] + off, base[:, 1:2] + off               # [S, P]
        ok = ((X >= 0) & (X < wl))[:, None, :] & ((Y >= 0) & (Y < hl))[:, :, None]   # [S, Py, Px]
        cl = lvl.permute(0, 2, 3, 1)                                # [B, hl, wl, D]
        t = cl[bs[:, None, None], Y.clamp(0, hl - 1)[:, :, None], X.clamp(0, wl - 1)[:, None, :]]   # [S, Py, Px, D]
        v = torch.einsum("spxd,sd->spx", t, q1) / D ** 0.5 * ok
        fx, fy = frac[:, 0, None, None], frac[:, 1, None, None]
        top = v[:, :-1, :-1] * (1 - fx) + v[:, :-1, 1:] * fx         # [S, j, i]
        bot = v[:, 1:, :-1] * (1 - fx) + v[:, 1:, 1:] * fx
        win = top * (1 - fy) + bot * fy                              # [S, j (y), i (x)]
        outs.append(win.transpose(1, 2).reshape(S, K * K))           # channel i*K + j
    return (bs, ys, xs), torch.cat(outs, 1)


def pick(out, idx):
    bs, ys, xs = idx
    return out[bs, :, ys, xs]


def tiles_on_tensor_cores(tc, f32):
    """Fraction of the 16x8 query tiles (per batch item) whose tf32 output differs from the fp32 one anywhere: the
    tiles the tensor cores served (TF32 operand rounding), where the fp32 kernel would give identical bits."""
    torch = _torch()
    B, C, h, w = tc.shape
    diff = (tc != f32).any(1)                                        # [B, h, w]
    th, tw = -(-h // 8), -(-w // 16)
    pad = torch.zeros(B, th * 8, tw * 16, dtype=torch.bool, device=tc.device)
    pad[:, :h, :w] = diff
    return pad.view(B, th, 8, tw, 16).any(4).any(2).float().mean().item()


def check_f64(blk_out, f1, f2, coords, levels, radius, tol):
    idx, ref = reference_f64(f1, f2, coords, levels, radius)
    e = normwise(pick(blk_out, idx).cpu().numpy(), ref.cpu().numpy())
    assert e <= tol, e
    return e


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("tf32", 1e-3)])
def test_alt_corr_golden(golden, cuda_device, precision, tol):
    import cistaflow_b200 as cf
    g = golden("corr")
    blk = cf.AlternateCorrBlock(dev_t(g["fmap1"], cuda_device), dev_t(g["fmap2"], cuda_device), 4, 4, precision=precision)
    out = blk(dev_t(g["coords"], cuda_device))
    assert tuple(out.shape) == g["lookup"].shape and out.is_contiguous()
    assert corr_err(*g.pick("lookup", out.cpu().numpy())) <= tol
    blk = cf.AlternateCorrBlock(dev_t(g["odd/fmap1"], cuda_device), dev_t(g["odd/fmap2"], cuda_device), num_levels=3,
                                radius=3, precision=precision)
    assert corr_err(*g.pick("odd/lookup", blk(dev_t(g["odd/coords"], cuda_device)).cpu().numpy())) <= tol


@pytest.mark.gpu
@pytest.mark.parametrize("trace", ["trace3_eiflow", "trace3_eraft"])
def test_alt_corr_model_trace_replay(golden, cuda_device, trace):
    """Coordinates of the running reference models (last refinement iteration of three consecutive frames)."""
    import cistaflow_b200 as cf
    g = golden(trace)
    frames = int(g["meta"][3])
    for f in range(frames):
        n_lookup = int(g[f"f{f}/counts"][0])
        f1, f2 = dev_t(g[f"f{f}/fmap1"], cuda_device), dev_t(g[f"f{f}/fmap2"], cuda_device)
        coords = dev_t(g[f"f{f}/coords{n_lookup - 1}"], cuda_device)
        out = cf.AlternateCorrBlock(f1, f2, 4, 4)(coords)
        assert corr_err(*g.pick(f"f{f}/lookup_last", out[:, ::4].cpu().numpy())) <= 1e-3
        # the models' coordinates stay on the tensor cores: every tile carries TF32 operand rounding
        assert tiles_on_tensor_cores(out, cf.AlternateCorrBlock(f1, f2, 4, 4, precision="fp32")(coords)) == 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("B,h,w", CONFIG_SHAPES)
def test_alt_corr_against_float64(cuda_device, B, h, w):
    import cistaflow_b200 as cf
    torch = _torch()
    f1, f2 = feature_maps(B, 256, h, w, cuda_device, seed=h * w)
    coords = smooth_coords(B, h, w, cuda_device, seed=B)
    with torch.no_grad():
        got32 = cf.AlternateCorrBlock(f1, f2, precision="fp32")(coords)
        assert last_kernel() == "corr_alt_simt_kernel"
        gottc = cf.AlternateCorrBlock(f1, f2, precision="tf32")(coords)
        assert last_kernel() == "corr_alt_tc_kernel"
    check_f64(got32, f1, f2, coords, 4, 4, 1e-5)
    check_f64(gottc, f1, f2, coords, 4, 4, 1e-3)
    # the tensor cores served these smooth coordinates: TF32 operand rounding is visible, and bounded
    d = normwise(gottc.cpu().numpy(), got32.cpu().numpy())
    assert 1e-6 < d <= 1e-3, d
    if (B, h, w) == (64, 60, 80):   # the headline: the whole output against the materialized pyramid
        ref = cf.CorrBlock(f1, f2, precision="fp32")(coords).cpu().numpy()
        assert normwise(got32.cpu().numpy(), ref) <= 1e-5
        assert normwise(gottc.cpu().numpy(), ref) <= 1e-3


@pytest.mark.gpu
def test_alt_corr_coordinate_stress(cuda_device):
    import cistaflow_b200 as cf
    torch = _torch()
    B, h, w = 4, 36, 44
    f1, f2 = feature_maps(B, 256, h, w, cuda_device, seed=5)
    noise = noise_coords(B, h, w, cuda_device, seed=6)
    mixed = smooth_coords(B, h, w, cuda_device, seed=7)
    mixed[:, :, :, w // 2:] = noise[:, :, :, w // 2:]          # tiles on both paths in one launch
    for coords in (noise, mixed):
        for prec, tol in (("fp32", 1e-5), ("auto", 1e-3)):
            check_f64(cf.AlternateCorrBlock(f1, f2, precision=prec)(coords), f1, f2, coords, 4, 4, tol)
    served = tiles_on_tensor_cores(cf.AlternateCorrBlock(f1, f2)(mixed), cf.AlternateCorrBlock(f1, f2, precision="fp32")(mixed))
    assert 0.0 < served < 1.0, served                          # both kernels served tiles of this launch
    blk = cf.AlternateCorrBlock(f1, f2)
    far = cf.coords_grid(B, h, w, device=cuda_device) + 1000.0
    assert not blk(far).any()
    assert not blk(-far).any()
    bad = smooth_coords(B, h, w, cuda_device, seed=8)
    bad[0, 0, 3, 5], bad[1, 1, 10, 20], bad[2, 0, 30, 40] = float("inf"), float("-inf"), float("nan")
    bad[3, :, :8, :16] = float("nan")                          # a whole tile
    ref = cf.CorrBlock(f1, f2)(bad)
    for prec in ("auto", "fp32"):
        got = cf.AlternateCorrBlock(f1, f2, precision=prec)(bad)
        for (b, y, x) in ((0, 3, 5), (1, 10, 20), (2, 30, 40), (3, 2, 7)):
            assert torch.equal(got[b, :, y, x], ref[b, :, y, x])


@pytest.mark.gpu
@pytest.mark.parametrize("D,levels,radius", [(32, 4, 4), (64, 3, 3), (256, 2, 2), (256, 5, 4), (64, 4, 7), (256, 4, 8),
                                             (128, 1, 0), (48, 4, 4)])
def test_alt_corr_other_shapes(cuda_device, D, levels, radius):
    """Every radius 0..8 on the tensor cores for smooth coordinates: each 16x8 tile of the tf32 output carries TF32
    operand rounding (differs from the fp32 kernel's bits).  D = 48 has no tensor-core tiling: fp32 kernel, same bits."""
    import cistaflow_b200 as cf
    torch = _torch()
    B, h, w = 2, 40, 52
    f1, f2 = feature_maps(B, D, h, w, cuda_device, seed=D + radius)
    coords = smooth_coords(B, h, w, cuda_device, seed=levels)
    got32 = cf.AlternateCorrBlock(f1, f2, levels, radius, precision="fp32")(coords)
    assert tuple(got32.shape) == (B, levels * (2 * radius + 1) ** 2, h, w)
    check_f64(got32, f1, f2, coords, levels, radius, 1e-5)
    gottc = cf.AlternateCorrBlock(f1, f2, levels, radius, precision="tf32")(coords)
    if D % 32:
        assert torch.equal(gottc, got32)
        return
    assert tiles_on_tensor_cores(gottc, got32) == 1.0
    assert 1e-6 < normwise(gottc.cpu().numpy(), got32.cpu().numpy()) <= 1e-3
    check_f64(gottc, f1, f2, coords, levels, radius, 1e-3)


@pytest.mark.gpu
def test_alt_corr_determinism_graph_and_streams(cuda_device):
    import cistaflow_b200 as cf
    torch = _torch()
    B, h, w = 8, 24, 32
    f1, f2 = feature_maps(B, 256, h, w, cuda_device, seed=11)
    coords = [smooth_coords(B, h, w, cuda_device, seed=s) for s in range(5)] + [noise_coords(B, h, w, cuda_device, seed=9)]
    eager = [cf.AlternateCorrBlock(f1, f2)(c) for c in coords]
    again = [cf.AlternateCorrBlock(f1, f2)(c) for c in coords]
    assert all(torch.equal(a, b) for a, b in zip(eager, again))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        blk = cf.AlternateCorrBlock(f1, f2)
        captured = [blk(c) for c in coords]
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(eager, captured))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        side = cf.AlternateCorrBlock(f1, f2)(coords[0])
    s.synchronize()
    assert torch.equal(side, eager[0])


@pytest.mark.gpu
def test_alt_corr_is_inference_only(cuda_device):
    import cistaflow_b200 as cf
    torch = _torch()
    f1, f2 = feature_maps(1, 64, 16, 16, cuda_device, seed=1)
    with pytest.raises(RuntimeError, match="inference-only"):
        cf.AlternateCorrBlock(f1.requires_grad_(), f2)
    blk = cf.AlternateCorrBlock(f1.detach(), f2)
    with pytest.raises(RuntimeError, match="inference-only"):
        blk(cf.coords_grid(1, 16, 16, device=cuda_device).requires_grad_())
    with torch.no_grad():
        blk(cf.coords_grid(1, 16, 16, device=cuda_device).requires_grad_())


@pytest.mark.gpu
def test_alt_corr_c_error_codes(cuda_device):
    import cistaflow_b200 as cf
    from cistaflow_b200 import _lib
    torch = _torch()
    lib = cf.load_library()
    B, D, h, w = 1, 64, 16, 16
    f1, f2 = feature_maps(B, D, h, w, cuda_device, seed=2)
    coords = cf.coords_grid(B, h, w, device=cuda_device)
    out = torch.empty(B, 4 * 81, h, w, device=cuda_device)
    n = lib.cf_corr_alt_workspace_bytes(B, D, h, w, 4, _lib.CORR_AUTO)
    st = torch.empty(n + 64, dtype=torch.uint8, device=cuda_device)
    s = _lib.stream_ptr(cuda_device)
    prep = lambda state, nbytes, prec=_lib.CORR_AUTO, levels=4, hh=h: lib.cf_corr_alt_prepare(  # noqa: E731
        f1.data_ptr(), f2.data_ptr(), B, D, hh, w, levels, prec, state, nbytes, s)
    assert prep(None, n) == -5 and prep(st.data_ptr(), n - 1) == -5
    assert prep(st.data_ptr() + 4, n) == -3
    assert prep(st.data_ptr(), n, levels=7) == -1 and prep(st.data_ptr(), n, levels=0) == -1
    assert prep(st.data_ptr(), n, hh=4) == -1                       # 4x16 has no level 3
    assert prep(st.data_ptr(), n, prec=_lib.CORR_F16) == -7 and prep(st.data_ptr(), n, prec=_lib.CORR_3XTF32) == -7
    assert prep(st.data_ptr(), n, prec=9) == -1
    assert prep(st.data_ptr(), n) == 0
    look = lambda state, radius=4, prec=_lib.CORR_AUTO: lib.cf_corr_alt_lookup(  # noqa: E731
        state, coords.data_ptr(), B, D, h, w, 4, radius, prec, out.data_ptr(), s)
    assert look(None) == -5 and look(st.data_ptr() + 4) == -3
    assert look(st.data_ptr(), radius=9) == -1 and look(st.data_ptr(), radius=-1) == -1
    assert look(st.data_ptr(), prec=_lib.CORR_F16) == -7
    assert look(st.data_ptr()) == 0
    torch.cuda.synchronize()
    with pytest.raises(ValueError):
        cf.AlternateCorrBlock(f1, f2, num_levels=7)


@pytest.mark.gpu
def test_alt_corr_memory_at_the_headline(cuda_device):
    import cistaflow_b200 as cf
    torch = _torch()
    B, D, h, w = 64, 256, 60, 80
    f1, f2 = feature_maps(B, D, h, w, cuda_device, seed=3)
    coords = smooth_coords(B, h, w, cuda_device, seed=3)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(cuda_device)
    base = torch.cuda.memory_allocated(cuda_device)
    blk = cf.AlternateCorrBlock(f1, f2)
    out = blk(coords)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated(cuda_device) - base
    state = blk.state.numel()
    assert grown <= state + out.numel() * 4 + (64 << 20), (grown, state)
    assert grown < 1.2e9
