"""The opt-in fp16 correlation pyramid (include/cistaflow_half.h): cf_corr_build_half and cf_corr_lookup_half.

The build is held to its contract branch by branch: level 0 is RN_f16 of what cf_corr_build stores for the same
precision (bit for bit, and within the fp32 path's float64 bound plus half an fp16 ulp), and every pooled level is
RN_f16 of ((a + b) + c) + d, x 0.25, summed in float32 over the stored level above (bit for bit against a numpy
restatement).  The lookup on an fp16 pyramid equals cf_corr_lookup on the widened pyramid bit for bit.  Outputs are
written into NaN-filled buffers with guard regions, as in test_gpu_corr_branches.py."""
import os
import re
import subprocess
import sys
from collections import namedtuple

import numpy as np
import pytest

from guarded_buffers import GUARD

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HALF_NAN = 0x7E00
U11 = 2.0 ** -11


def _header_symbols(name):
    text = open(os.path.join(ROOT, "include", name)).read()
    return sorted(re.findall(r"CF_API\s+[\w\s\*]+?\b(cf_\w+)\s*\(", text))


# ----------------------------------------------------------------------------------------------------- CPU ---
def test_half_header_matches_ctypes_table_and_library():
    import cistaflow_b200 as cf
    from cistaflow_b200 import _lib
    syms = _header_symbols("cistaflow_half.h")
    assert syms == sorted(["cf_corr_build_half", "cf_corr_lookup_half"]) == sorted(_lib.HALF_SYMBOLS)
    assert len(_header_symbols("cistaflow.h")) == 26 and sorted(_lib.SYMBOLS) == _header_symbols("cistaflow.h")
    assert not set(syms) & (set(_lib.SYMBOLS) | set(_lib.ALTCORR_SYMBOLS) | set(_lib.DET_SYMBOLS))
    lib = cf.load_library()
    for name in syms:
        assert getattr(lib, name).restype == _lib.HALF_SYMBOLS[name][0]


def test_storage_is_validated_without_a_gpu():
    import torch
    import cistaflow_b200 as cf
    f = torch.zeros(1, 32, 4, 8)
    for bad in ("fp16", "F16", "bf16", "f64", ""):
        with pytest.raises(ValueError, match="storage"):
            cf.build_pyramid(f, f, 2, storage=bad or "x")
        with pytest.raises(ValueError, match="storage"):
            cf.CorrBlock(f, f, 2, 1, storage=bad or "x")
    for prec in ("fp32", "3xtf32"):
        with pytest.raises(ValueError, match="fp32 accuracy"):
            cf.build_pyramid(f, f, 2, precision=prec, storage="f16")
    with pytest.raises(ValueError, match="D % 32"):
        cf.build_pyramid(torch.zeros(1, 48, 4, 8), torch.zeros(1, 48, 4, 8), 2, storage="f16")
    with pytest.raises(ValueError, match="h\\*w % 8"):
        cf.build_pyramid(torch.zeros(1, 32, 6, 6), torch.zeros(1, 32, 6, 6), 2, storage="f16")


def test_f16_storage_is_inference_only():
    import torch
    import cistaflow_b200 as cf
    f = torch.zeros(1, 32, 4, 8, requires_grad=True)
    with pytest.raises(RuntimeError, match="inference-only"):
        cf.CorrBlock(f, f.detach(), 2, 1, storage="f16")


_DEFAULT_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
from cistaflow_b200 import corr
print(corr.DEFAULT_STORAGE)
"""


@pytest.mark.parametrize("env,expect", [(None, "f32"), ("f16", "f16"), ("f32", "f32")])
def test_storage_default_from_environment(env, expect):
    e = dict(os.environ)
    e.pop("CISTAFLOW_CORR_STORAGE", None)
    if env is not None:
        e["CISTAFLOW_CORR_STORAGE"] = env
    flags = ["-s"] if sys.flags.no_user_site else []
    res = subprocess.run([sys.executable, *flags, "-c", _DEFAULT_SCRIPT, ROOT], env=e, cwd=ROOT, capture_output=True,
                         text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    assert res.stdout.strip() == expect


# ------------------------------------------------------------------------------------------------- helpers ---
def half_guarded(shapes, device):
    """fp16 views of the given shapes inside one buffer of fp16 NaN, GUARD halves of NaN around each, views on 16-byte
    boundaries."""
    import torch
    offs, pos = [], GUARD
    for s in shapes:
        offs.append(pos)
        pos = -(-(pos + int(np.prod(s))) // 8) * 8 + GUARD
    buf = torch.full((pos,), HALF_NAN, dtype=torch.int16, device=device).view(torch.float16)
    return buf, [buf[o:o + int(np.prod(s))].view(s) for o, s in zip(offs, shapes)]


def assert_half_written_and_guarded(buf, views, what):
    import torch
    inside = torch.zeros(buf.numel(), dtype=torch.bool, device=buf.device)
    for v in views:
        o = (v.data_ptr() - buf.data_ptr()) // 2
        inside[o:o + v.numel()] = True
    bits = buf.view(torch.int16)
    assert bool((bits[inside] != HALF_NAN).all()), f"{what}: unwritten elements (the kernels never store NaN here)"
    assert bool((bits[~inside] == HALF_NAN).all()), f"{what}: guard halves overwritten"


def same_half(a, b):
    """bit-identical, NaN matching any NaN"""
    a, b = np.asarray(a, np.float16), np.asarray(b, np.float16)
    nan = np.isnan(a)
    return bool((nan == np.isnan(b)).all() and (a.view(np.uint16)[~nan] == b.view(np.uint16)[~nan]).all())


def pool_f32_restated(level):
    """RN_f16((((a + b) + c) + d) * 0.25) in float32 over the 2x2 windows of a stored fp16 level [M, 1, H, W] (floor)."""
    a = np.asarray(level, np.float32)
    H, W = a.shape[-2] // 2, a.shape[-1] // 2
    a = a[..., :2 * H, :2 * W]
    with np.errstate(invalid="ignore"):   # inf + -inf -> NaN, as on the device
        s = a[..., 0::2, 0::2] + a[..., 0::2, 1::2]
        s = s + a[..., 1::2, 0::2]
        s = s + a[..., 1::2, 1::2]
    return (s * np.float32(0.25)).astype(np.float16)


# ------------------------------------------------------------------------------------------------ build table ---
Row = namedtuple("Row", "branch B D h w levels R deep pair2")
BUILD_ROWS = [
    Row("R == 0 (w > 128)", 2, 256, 16, 136, 4, 0, 0, 0),
    Row("R == 0, odd w, B = 1", 1, 256, 16, 29, 4, 0, 0, 0),
    Row("plain R = 6, BN = 216", 2, 256, 30, 36, 4, 6, 0, 0),
    Row("deep = 1, partial last tile, B = 3", 3, 256, 12, 24, 4, 8, 1, 0),
    Row("deep = 1, levels = 3", 2, 256, 32, 32, 3, 8, 1, 0),
    *[Row(f"deep = 2, D = {D}", 2, D, 24, 32, 4, 8, 2, 0) for D in (32, 64, 96, 160, 512)],
    Row("pair2", 2, 256, 12, 96, 4, 2, 0, 1),
    Row("pair2, b_sw64 with fp16 operands", 4, 256, 20, 80, 4, 2, 0, 1),
    Row("fp16-misaligned level 1 (396 halves per query), B = 5", 5, 256, 36, 44, 4, 4, 0, 0),
    Row("stream_l0 (fp16 volume > 64 MB), misaligned level 1", 16, 256, 36, 44, 4, 4, 0, 0),
    Row("AUTO picks fp16 operands", 10, 256, 32, 64, 4, 4, 0, 0),
    Row("tile narrower than one {64 x 32} box", 3, 64, 4, 8, 2, 4, 0, 0),
    *[Row(f"levels = {L}", 2, 256, 32, 32, L, 8 if L > 1 else 0, {1: 0, 2: 0, 3: 1}.get(L, 2), 0) for L in (1, 2, 5, 6)],
]
BUILD_CASES = [pytest.param(row, prec, id=f"{row.B}x{row.D}x{row.h}x{row.w}-L{row.levels}-{prec}")
               for row in BUILD_ROWS for prec in ("tf32", "auto", "f16") if prec != "f16" or row.D % 128 == 0]


def half_kernel_name(prec, B, D, h, w):
    from test_gpu_corr_branches import auto_is_f16
    f16 = prec == "f16" or (prec == "auto" and auto_is_f16(B, D, h, w))
    return "corr_tc_half_kernel<f16>" if f16 else "corr_tc_half_kernel"


def build_half(f1, f2, levels, prec):
    """(views, launches the build made, name of its last kernel)"""
    import torch
    import cistaflow_b200 as cf
    from cistaflow_b200 import _lib
    lib = _lib.load()
    B, D, h, w = f1.shape
    shapes = [(B * h * w, 1, h >> l, w >> l) for l in range(levels)]
    buf, views = half_guarded(shapes, f1.device)
    n0 = lib.cf_launch_count()
    cf.build_pyramid(f1, f2, levels, precision=prec, out=views, storage="f16")
    torch.cuda.synchronize()
    last = lib.cf_last_kernel().decode()
    assert_half_written_and_guarded(buf, views, f"levels={levels} fp16 build")
    return views, lib.cf_launch_count() - n0, last


@pytest.mark.gpu
@pytest.mark.parametrize("row,prec", BUILD_CASES)
def test_half_build_branch(cuda_device, parity_report, row, prec):
    import torch
    import cistaflow_b200 as cf
    from cistaflow_b200 import _lib
    from test_gpu_corr_branches import build_coefficient, check_levels, exact_and_magnitude, f16_floor, plan
    B, D, h, w, L = row.B, row.D, row.h, row.w, row.levels
    R, deep, pair2, fused = plan(h, w, L)
    assert (R, deep, pair2) == (row.R, row.deep, row.pair2), f"the row's stated branch is not the planner's: {plan(h, w, L)}"
    g = torch.Generator(device=cuda_device).manual_seed(1000 * h + w + D + L)
    f1 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    f2 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    lib = _lib.load()
    # the contraction alone (levels = 1), then the whole pyramid: the launches beyond the first build's are pooling kernels
    one, n_one, last_one = build_half(f1, f2, 1, prec)
    assert last_one == half_kernel_name(prec, B, D, h, w)
    views, n_all, last = build_half(f1, f2, L, prec)
    pools = n_all - n_one
    pooled = 0 if pools == 0 else 2 * pools - (1 if last == "avg_pool2x2_half_kernel" else 0)
    assert pools == 0 or last in ("avg_pool2x2_half_kernel", "avg_pool_two_levels_half_kernel"), last
    assert L - 1 - pooled == fused, f"{row.branch}: {pools} pooling launches, last {last}"
    # level 0 = RN_f16 of the fp32 build's level 0, bit for bit ...
    with torch.no_grad():
        ref32 = cf.build_pyramid(f1, f2, L, precision=prec, storage="f32")
    for got in (one[0], views[0]):
        assert torch.equal(got.view(torch.int16), ref32[0].half().view(torch.int16)), f"{row.branch}: level 0 != RN_f16(fp32)"
    # ... and within the fp32 path's float64 bound plus half an fp16 ulp and the subnormal spacing
    ref, mag = exact_and_magnitude(f1, f2, 1)
    floor = f16_floor(f1, f2) if half_kernel_name(prec, B, D, h, w).endswith("<f16>") else None
    worst = check_levels([views[0].float()], ref, mag, build_coefficient(prec, D), B, floor, row.branch,
                         extra=[U11 * views[0].double().abs() + 2.0 ** -25])
    # every pooled level: the float32 restatement of the stated order on the stored level above, bit for bit
    for l in range(1, L):
        assert same_half(views[l].cpu().numpy(), pool_f32_restated(views[l - 1].cpu().numpy())), f"{row.branch}: level {l}"
    parity_report.add("corr_half/build", branch=row.branch, shape=f"{B}x{D}x{h}x{w}", levels=L, precision=prec,
                      fused=fused, pool_launches=pools, worst_err_over_bound=worst)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["overflow", "nan"])
@pytest.mark.parametrize("prec", ["tf32", "f16"])
def test_half_build_overflow_and_nan(cuda_device, case, prec):
    """|v| >= 65520 is stored as +-inf and NaN stays NaN (no clamping), level 0 and every pooled level."""
    import torch
    import cistaflow_b200 as cf
    B, D, h, w, L = 2, 256, 24, 32, 5
    g = torch.Generator(device=cuda_device).manual_seed(3)
    f1 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    f2 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    if case == "overflow":
        f1 *= 1000.0
        f2 *= 200.0
    else:
        f1[0, :, 3, 5] = float("nan")
        f2[1, 7, 10, :] = float("nan")
    views, _, _ = build_half(f1, f2, L, prec) if case == "overflow" else (None, 0, None)
    if case == "nan":   # NaN levels: the guard check cannot tell NaN from unwritten, so build into plain tensors
        views = cf.build_pyramid(f1, f2, L, precision=prec, storage="f16")
    with torch.no_grad():
        ref32 = cf.build_pyramid(f1, f2, L, precision=prec, storage="f32")
    l0 = views[0].cpu().numpy()
    assert same_half(l0, ref32[0].half().cpu().numpy())
    if case == "overflow":
        assert np.isinf(l0).mean() > 0.1 and (np.abs(ref32[0].cpu().numpy()) >= 65520).sum() == np.isinf(l0).sum()
    else:
        assert np.isnan(l0).any() and not np.isnan(l0).all()
    for l in range(1, L):
        assert same_half(views[l].cpu().numpy(), pool_f32_restated(views[l - 1].cpu().numpy())), f"{case}: level {l}"


# -------------------------------------------------------------------------------------------------- lookups ---
LOOKUP_CASES = [(L, r) for L in range(1, 7) for r in range(9)]


@pytest.fixture(scope="module")
def half_lookup_problem(cuda_device):
    import torch
    from test_gpu_corr_branches import LB, LH, LW
    g = torch.Generator(device=cuda_device).manual_seed(78)
    N = LH * LW
    pyr = [(torch.randn(LB * N, 1, LH >> l, LW >> l, device=cuda_device, generator=g) * 30).half() for l in range(6)]
    pyr[0].view(-1)[::997] = float("inf")      # a few non-finite taps: they flow through the same arithmetic
    pyr[1].view(-1)[::1499] = float("nan")
    return pyr


@pytest.mark.gpu
@pytest.mark.parametrize("levels,radius", LOOKUP_CASES)
def test_half_lookup_equals_widened(cuda_device, half_lookup_problem, levels, radius):
    """cf_corr_lookup_half == cf_corr_lookup on the widened pyramid, bit for bit, for the whole batch (32 queries per
    CTA, or the radius-4 kernel's balanced count) and for item 0 alone (16 queries per CTA); the coordinates are
    integers, half-integers, out-of-map, far-out, +-inf and NaN (lookup_coords)."""
    import torch
    import cistaflow_b200 as cf
    from cistaflow_b200 import _lib
    from test_gpu_corr_branches import LB, LH, LW, lookup_coords
    pyr = half_lookup_problem[:levels]
    N = LH * LW
    coords = lookup_coords(LB, LH, LW, radius, cuda_device, seed=10 * levels + radius + 5)
    name = "corr_lookup_r4l4_half_kernel" if (levels, radius) == (4, 4) else "corr_lookup_half_kernel"
    for p, c in ((pyr, coords), ([q[:N] for q in pyr], coords[:1].contiguous())):
        got = cf.corr_lookup(p, c, radius)
        assert _lib.load().cf_last_kernel().decode() == name
        ref = cf.corr_lookup([q.float() for q in p], c, radius)
        assert torch.equal(got.view(torch.int32), ref.view(torch.int32)), f"levels={levels} radius={radius}"


_FORCED_QT_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
import torch
import cistaflow_b200 as cf
from cistaflow_b200 import _lib
B, h, w = 4, 37, 24
N = h * w
dev = torch.device("cuda", 0)
g = torch.Generator(device=dev).manual_seed(5)
pyr = [(10 * torch.randn(B * N, 1, h >> l, w >> l, device=dev, generator=g)).half() for l in range(4)]
ys, xs = torch.meshgrid(torch.arange(h, device=dev), torch.arange(w, device=dev), indexing="ij")
coords = torch.stack([xs, ys]).float()[None] + 6 * torch.randn(B, 2, h, w, device=dev, generator=g)
out = cf.corr_lookup(pyr, coords, 4)
assert _lib.load().cf_last_kernel().decode() == "corr_lookup_r4l4_half_kernel"
ref = cf.corr_lookup([p.float() for p in pyr], coords, 4)
assert torch.equal(out.view(torch.int32), ref.view(torch.int32))
torch.save(out.cpu(), sys.argv[2])
"""


@pytest.mark.gpu
def test_half_lookup_forced_query_counts(cuda_device, tmp_path):
    """Every CF_LOOKUP_QT (even counts 16..32, read once per process): the fp16 radius-4 kernel equals the fp32 one on
    the widened pyramid, and every count gives the same bits."""
    import torch
    outs = {}
    flags = ["-s"] if sys.flags.no_user_site else []
    for qt in [None, *range(16, 33, 2)]:
        env = dict(os.environ)
        env.pop("CF_LOOKUP_QT", None)
        if qt is not None:
            env["CF_LOOKUP_QT"] = str(qt)
        path = str(tmp_path / f"out_{qt}.pt")
        res = subprocess.run([sys.executable, *flags, "-c", _FORCED_QT_SCRIPT, ROOT, path], env=env, cwd=ROOT,
                             capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, f"CF_LOOKUP_QT={qt}:\n{res.stdout}\n{res.stderr}"
        outs[qt] = torch.load(path)
    base = outs.pop(None)
    for qt, o in outs.items():
        assert torch.equal(o.view(torch.int32), base.view(torch.int32)), f"CF_LOOKUP_QT={qt}"


# --------------------------------------------------------------------------------------------- model traces ---
@pytest.mark.gpu
@pytest.mark.parametrize("trace", ["trace3_eiflow", "trace3_eraft"])
def test_half_model_trace_replay(golden, cuda_device, trace):
    """Coordinates of the running reference models through CorrBlock(storage="f16"): within the golden lookups' bound
    (1e-3 of the largest value, as for the fp32 pyramid) plus the fp16 storage term 2^-11."""
    import torch
    import cistaflow_b200 as cf
    from test_gpu_parity import corr_err
    g = golden(trace)
    for f in range(int(g["meta"][3])):
        n_lookup = int(g[f"f{f}/counts"][0])
        f1 = torch.from_numpy(np.ascontiguousarray(g[f"f{f}/fmap1"])).to(cuda_device)
        f2 = torch.from_numpy(np.ascontiguousarray(g[f"f{f}/fmap2"])).to(cuda_device)
        coords = torch.from_numpy(np.ascontiguousarray(g[f"f{f}/coords{n_lookup - 1}"])).to(cuda_device)
        blk = cf.CorrBlock(f1, f2, 4, 4, storage="f16")
        assert all(p.dtype == torch.float16 for p in blk.corr_pyramid)
        out = blk(coords)
        assert out.dtype == torch.float32
        assert corr_err(*g.pick(f"f{f}/lookup_last", out[:, ::4].cpu().numpy())) <= 1e-3 + U11


# ------------------------------------------------------------------------------------------------ behaviour ---
@pytest.mark.gpu
def test_half_repeatable_side_stream_and_graph(cuda_device):
    import torch
    import cistaflow_b200 as cf
    B, D, h, w = 4, 256, 36, 44
    g = torch.Generator(device=cuda_device).manual_seed(11)
    f1 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    f2 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    coords = cf.coords_grid(B, h, w, device=cuda_device) + 3 * torch.randn(B, 2, h, w, device=cuda_device, generator=g)

    def run():
        blk = cf.CorrBlock(f1, f2, 4, 4, storage="f16")
        return blk.corr_pyramid, blk(coords)

    pyr_a, out_a = run()
    pyr_b, out_b = run()
    s = torch.cuda.Stream(device=cuda_device)
    s.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(s):
        pyr_c, out_c = run()
    torch.cuda.current_stream(cuda_device).wait_stream(s)
    for pyr, out in ((pyr_b, out_b), (pyr_c, out_c)):
        assert all(torch.equal(x.view(torch.int16), y.view(torch.int16)) for x, y in zip(pyr_a, pyr))
        assert torch.equal(out_a.view(torch.int32), out.view(torch.int32))
    # capture the build and a lookup into a CUDA graph and replay it
    pyr = [torch.empty_like(p) for p in pyr_a]
    out = torch.empty_like(out_a)
    s.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(s):     # warm-up outside the capture (workspace allocation)
        cf.build_pyramid(f1, f2, 4, out=pyr, storage="f16")
        cf.corr_lookup(pyr, coords, 4, out=out)
    torch.cuda.current_stream(cuda_device).wait_stream(s)
    for p in pyr:
        p.fill_(0)
    out.fill_(0)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cf.build_pyramid(f1, f2, 4, out=pyr, storage="f16")
        cf.corr_lookup(pyr, coords, 4, out=out)
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(x.view(torch.int16), y.view(torch.int16)) for x, y in zip(pyr_a, pyr))
    assert torch.equal(out_a.view(torch.int32), out.view(torch.int32))


@pytest.mark.gpu
def test_half_c_error_codes(cuda_device):
    import torch
    from cistaflow_b200 import _lib
    lib = _lib.load()
    dev = cuda_device
    B, D, h, w, L = 2, 64, 8, 16, 2
    f = torch.randn(B, D, h, w, device=dev)
    pyr = [torch.empty(B * h * w, 1, h >> l, w >> l, dtype=torch.float16, device=dev) for l in range(L)]
    coords = torch.zeros(B, 2, h, w, device=dev)
    out = torch.empty(B, L * 9, h, w, device=dev)
    arr = _lib.pointer_array(pyr)
    stream = _lib.stream_ptr(dev)

    def build(*, D_=D, h_=h, w_=w, L_=L, prec=_lib.CORR_TF32, p=arr, f1=f.data_ptr()):
        return lib.cf_corr_build_half(f1, f.data_ptr(), B, D_, h_, w_, L_, p, prec, None, 0, stream)

    assert build() == 0
    assert build(prec=_lib.CORR_FP32) == -7 and build(prec=_lib.CORR_3XTF32) == -7
    assert build(prec=9) == -1
    assert build(D_=48) == -7 and build(h_=6, w_=6) == -7
    assert build(L_=0) == -1 and build(L_=7) == -1 and build(h_=1, L_=2) == -1
    assert build(f1=None) == -2 and build(p=None) == -2
    assert build(prec=_lib.CORR_F16) == 0   # D % 128 != 0: TF32 operands, no workspace needed
    assert build(prec=_lib.CORR_AUTO) == 0
    look = lambda **k: lib.cf_corr_lookup_half(k.get("p", arr), coords.data_ptr(), B, h, w, k.get("L", L), k.get("r", 1),
                                               out.data_ptr(), stream)
    assert look() == 0
    assert look(r=9) == -1 and look(r=-1) == -1 and look(L=0) == -1 and look(L=7) == -1
    assert look(p=None) == -2
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_half_peak_memory_at_headline(cuda_device):
    """The fp16 pyramid's peak memory growth at 64 x 60x80 is about half the fp32 pyramid's (operand copies included)."""
    import torch
    import cistaflow_b200 as cf
    B, D, h, w = 64, 256, 60, 80
    g = torch.Generator(device=cuda_device).manual_seed(1)
    f1 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    f2 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    growth = {}
    for st in ("f32", "f16"):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        base = torch.cuda.memory_allocated(cuda_device)
        torch.cuda.reset_peak_memory_stats(cuda_device)
        with torch.no_grad():
            blk = cf.CorrBlock(f1, f2, 4, 4, storage=st)
        torch.cuda.synchronize()
        growth[st] = torch.cuda.max_memory_allocated(cuda_device) - base
        del blk
    ratio = growth["f16"] / growth["f32"]
    assert 0.45 <= ratio <= 0.55, (growth, ratio)
