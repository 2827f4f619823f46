"""The correlation build, lookup and lookup backward on every branch of their dispatch, element by element against float64.

Each comparison bounds every element by the error model of the arithmetic the kernel does. The model uses the
magnitudes the element is made of: |f1|^T |f2| / sqrt(D) for the volume, sum |w * p| for a bilinear sample. The bound
is not fitted to what a kernel happens to return. It is asserted separately per (batch item, level), so a wrong small
item or level cannot hide behind a large one. Outputs are written into NaN-filled buffers with guard regions. An
element the kernel skipped stays NaN, and a write outside the output changes a guard.

Which branch a build took is read from the launches: cf_last_kernel() names the contraction, and the number and kind of
pooling launches after it give the levels its epilogue produced. ``plan`` restates the planner's rules
(corr_volume_tensor_core in csrc/corr_build_tc.cu) so that every row of the build table names its branch and the
launches confirm it."""
import math
import os
import subprocess
import sys
from collections import namedtuple

import numpy as np
import pytest
import torch

import cistaflow_b200 as cf
from cistaflow_b200 import _lib
from guarded_buffers import assert_written_and_guarded, guarded

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U11 = 2.0 ** -11     # unit roundoff of a TF32 / fp16 significand
U24 = 2.0 ** -24     # unit roundoff of fp32


def dev_t(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def last_kernel():
    return _lib.load().cf_last_kernel().decode()


def launch_count():
    return _lib.load().cf_launch_count()


# ----------------------------------------------------------------------------------------- planner restatement ---
MAX_BN = 256


def _align(x, a):
    return -(-x // a) * a


def plan(h, w, levels, level2_aligned=True):
    """(R, deep, pair2, fused) as corr_volume_tensor_core picks them (no experiment flags): R whole target rows per tile,
    deep = levels 2 (1) or 2 and 3 (2) pooled in the epilogue, pair2 = level 2 from tile pairs, fused = levels beyond
    level 0 that the contraction's launch writes."""
    R = 0
    if levels > 1 and w % 4 == 0 and h % 2 == 0 and 2 * w <= MAX_BN:
        R = min(2 * (MAX_BN // (2 * w)), h)
        while R > 0 and (R - 1) * w + _align(w, 32) > MAX_BN:
            R -= 2
        if w <= 32 and w % 8 == 0:
            if R >= 8 and h % 8 == 0:
                R &= ~7
            elif R >= 4 and h % 4 == 0:
                R &= ~3
    l2 = levels > 2 and level2_aligned
    deep = 0
    if R > 0 and w <= 32 and l2 and R % 4 == 0 and w % 8 == 0 and h % 4 == 0:
        deep = 2 if (levels > 3 and R % 8 == 0 and h % 8 == 0) else 1
    pair2 = int(R == 2 and deep == 0 and l2 and h % 4 == 0 and w % 16 == 0 and _align(R * w, 16) + w // 2 <= MAX_BN)
    fused = 1 + (pair2 or deep) if R else 0
    return R, deep, pair2, fused


def auto_is_f16(B, D, h, w):
    N = h * w
    return N % 64 == 0 and N >= 2048 and B * N >= 19200 and D % 128 == 0


def tc_kernel_name(prec, B, D, h, w):
    if prec == "auto":
        prec = "f16" if auto_is_f16(B, D, h, w) else "tf32"
    return {"tf32": "corr_tc_kernel", "3xtf32": "corr_tc_kernel<3xtf32>", "f16": "corr_tc_kernel<f16>"}[prec]


def fused_from_launches(levels, pool_launches, last):
    """Pooling after the contraction: two levels per avg_pool_two_levels_kernel, the last odd level by
    avg_pool2x2_kernel (cf_corr_build), so the launch count and the last kernel give the pooled level count."""
    pooled = 0 if pool_launches == 0 else 2 * pool_launches - (1 if last == "avg_pool2x2_kernel" else 0)
    return levels - 1 - pooled


# ------------------------------------------------------------------------------------------ float64 references ---
def pool_levels(vol, levels):
    pyr = [vol]
    for _ in range(levels - 1):
        pyr.append(torch.nn.functional.avg_pool2d(pyr[-1], 2, stride=2))
    return pyr


def exact_and_magnitude(f1, f2, levels):
    """The pyramid in float64 (f1^T f2 / sqrt(D), then avg_pool2d with floor) and the same of |f1|^T |f2| / sqrt(D)."""
    B, D, h, w = f1.shape
    N = h * w
    a, b = f1.double().reshape(B, D, N), f2.double().reshape(B, D, N)
    s = float(D) ** 0.5
    vol = (a.transpose(1, 2) @ b / s).reshape(B * N, 1, h, w)
    mag = (a.abs().transpose(1, 2) @ b.abs() / s).reshape(B * N, 1, h, w)
    return pool_levels(vol, levels), pool_levels(mag, levels)


def build_coefficient(prec, D):
    """|err| <= coef * magnitude.  TF32 / fp16 operands round to an 11-bit significand (each product off by < 2u), the
    3xTF32 split leaves < 2^-21 of each product, and D fp32 accumulations add gamma_D = D * 2^-24; a factor 2 covers the
    epilogue's scale and pooling roundings."""
    gamma = D * U24
    if prec == "3xtf32":
        return 2 * (2.0 ** -21 + gamma)
    if prec == "fp32":
        return 2 * gamma
    return 2 * (2 * U11 + gamma)


def f16_floor(f1, f2):
    """Absolute floor per batch item for fp16 operands.  fmap_to_half* scales item b of a map by up = 2^(13 - ilogb(max))
    so the largest magnitude lands in [2^13, 2^14).  A scaled value below the fp16 normal range then rounds to a
    subnormal step of 2^-24, an absolute error of <= 2^-25 / up <= 2^-38 * max in the input's units.  Summed over D
    products, and divided by sqrt(D), that adds (d1 * max2 + d2 * max1) * sqrt(D) <= 2 * 2^-38 * max1 * max2 * sqrt(D)
    to any element. The floor below is twice that."""
    B, D = f1.shape[:2]
    m1 = f1.double().reshape(B, -1).abs().amax(1)
    m2 = f2.double().reshape(B, -1).abs().amax(1)
    return 4 * 2.0 ** -38 * m1 * m2 * float(D) ** 0.5


def check_levels(got, ref, mag, coef, B, floor=None, what="", extra=None):
    """max(|got - ref| / (coef * mag + floor + extra)) <= 1 for every (batch item, level); returns the largest ratio.
    floor is per batch item, extra (a list of per-level tensors) per element.  A zero bound demands an exact zero."""
    worst = 0.0
    for l, (g, r, a) in enumerate(zip(got, ref, mag)):
        hl, wl = g.shape[-2:]
        g, r, a = g.reshape(B, -1, hl * wl), r.reshape(B, -1, hl * wl), a.reshape(B, -1, hl * wl)
        e = extra[l].reshape(B, -1, hl * wl) if extra is not None else None
        for b in range(B):
            bound = coef * a[b] + (float(floor[b]) if floor is not None else 0.0)
            if e is not None:
                bound = bound + e[b]
            err = (g[b].double() - r[b]).abs()
            ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300),
                                torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))
            m = float(ratio.max())
            if not m <= 1.0:
                q, yx = divmod(int(ratio.argmax()), hl * wl)
                raise AssertionError(f"{what}: level {l} item {b}: err/bound = {m:.3g} at (b={b}, q={q}, y={yx // wl}, "
                                     f"x={yx % wl}): got {float(g[b, q, yx]):.9g}, exact {float(r[b, q, yx]):.9g}")
            worst = max(worst, m)
    return worst


# ------------------------------------------------------------------------------------------------- build sweep ---
Row = namedtuple("Row", "branch B D h w levels R deep pair2")
BUILD_ROWS = [
    Row("partial last tile (4 of 8 rows), deep=1", 2, 256, 20, 32, 4, 8, 1, 0),
    Row("partial last tile (4 of 8 rows), deep=1, B=3", 3, 256, 12, 24, 4, 8, 1, 0),
    Row("partial last tile (2 of 4 rows), LSU stores", 2, 256, 18, 40, 4, 4, 0, 0),
    Row("R=6, BN=216", 2, 256, 30, 36, 4, 6, 0, 0),
    Row("R=2 without pair2, LSU stores", 2, 256, 10, 100, 4, 2, 0, 0),
    Row("R=2 with pair2, small", 2, 256, 12, 96, 4, 2, 0, 1),
    Row("R=4, BN=256", 2, 256, 32, 64, 4, 4, 0, 0),
    Row("unfused, w > 128", 2, 256, 16, 136, 4, 0, 0, 0),
    Row("unfused, w % 4 != 0", 2, 256, 16, 30, 4, 0, 0, 0),
    Row("unfused, odd w", 1, 256, 16, 29, 4, 0, 0, 0),
    Row("levels=1", 2, 256, 32, 32, 1, 0, 0, 0),
    Row("levels=2", 2, 256, 32, 32, 2, 8, 0, 0),
    Row("levels=3, deep=1", 2, 256, 32, 32, 3, 8, 1, 0),
    Row("levels=5, deep=2 + one pooled level", 2, 256, 32, 32, 5, 8, 2, 0),
    Row("levels=6, deep=2 + two pooled levels", 2, 256, 32, 32, 6, 8, 2, 0),
    *[Row(f"D={D}, deep=2", 2, D, 24, 32, 4, 8, 2, 0) for D in (32, 64, 96, 160, 512)],
    *[Row(f"D={D}, per-atom boxes", 2, D, 36, 44, 4, 4, 0, 0) for D in (32, 64, 96, 160, 512)],
    Row("AUTO picks f16 (N=2048, B*N >= 19200)", 10, 256, 32, 64, 4, 4, 0, 0),
    Row("f16 b_sw64 + pair2", 4, 256, 20, 80, 4, 2, 0, 1),
    Row("stream_l0 (volume > 64 MB)", 8, 256, 36, 44, 4, 4, 0, 0),
    Row("levels=1, rows below the volume in each item's last query tile", 8, 128, 20, 80, 1, 0, 0, 0),
]
BUILD_CASES = [pytest.param(row, prec, id=f"{row.B}x{row.D}x{row.h}x{row.w}-L{row.levels}-{prec}")
               for row in BUILD_ROWS for prec in ("tf32", "3xtf32", "auto", "f16") if prec != "f16" or row.D % 128 == 0]
def run_build(f1, f2, levels, prec, misalign=None):
    """Build into guarded views; returns (level 0 of a levels=1 build, views, pooling launches after the contraction,
    last kernel).  The launches before the contraction (operand conversion) are counted by the levels=1 build of the
    same maps, which never pools."""
    B, D, h, w = f1.shape
    dev = f1.device
    shapes = [(B * h * w, 1, h >> l, w >> l) for l in range(levels)]
    n0 = launch_count()
    buf1, one = guarded(shapes[:1], dev)
    cf.build_pyramid(f1, f2, 1, precision=prec, out=one)
    n1 = launch_count()
    assert last_kernel() == tc_kernel_name(prec, B, D, h, w)
    buf, views = guarded(shapes, dev, misalign)
    cf.build_pyramid(f1, f2, levels, precision=prec, out=views)
    n2 = launch_count()
    torch.cuda.synchronize()
    assert_written_and_guarded(buf1, one, "levels=1 build")
    assert_written_and_guarded(buf, views, f"levels={levels} build")
    return one, views, (n2 - n1) - (n1 - n0), last_kernel()


@pytest.mark.parametrize("row,prec", BUILD_CASES)
def test_build_branch(cuda_device, parity_report, row, prec):
    B, D, h, w, L = row.B, row.D, row.h, row.w, row.levels
    R, deep, pair2, fused = plan(h, w, L)
    assert (R, deep, pair2) == (row.R, row.deep, row.pair2), f"the row's stated branch is not what the planner picks: {plan(h, w, L)}"
    g = torch.Generator(device=cuda_device).manual_seed(1000 * h + w + D + L)
    f1 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    f2 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    one, views, pools, last = run_build(f1, f2, L, prec)
    assert fused_from_launches(L, pools, last) == fused, f"{row.branch}: {pools} pooling launches, last {last}"
    ref, mag = exact_and_magnitude(f1, f2, L)
    coef = build_coefficient(prec, D)
    floor = f16_floor(f1, f2) if tc_kernel_name(prec, B, D, h, w) == "corr_tc_kernel<f16>" else None
    worst = check_levels(views, ref, mag, coef, B, floor, row.branch)
    worst = max(worst, check_levels(one, ref, mag, coef, B, floor, f"{row.branch}, levels=1"))
    parity_report.add("corr_branches/build", branch=row.branch, shape=f"{B}x{D}x{h}x{w}", levels=L, precision=prec,
                      fused=fused, pool_launches=pools, worst_err_over_bound=worst)
    if L == 1:   # CorrBlock.corr is the levels=1 build, viewed [B, h, w, 1, h, w]
        vol = cf.CorrBlock.corr(f1, f2, precision=prec)
        assert tuple(vol.shape) == (B, h, w, 1, h, w)
        check_levels([vol.reshape(B * h * w, 1, h, w)], ref, mag, coef, B, floor, "CorrBlock.corr")


@pytest.mark.parametrize("prec", ["tf32", "3xtf32", "auto", "f16"])
def test_build_per_item_scale(cuda_device, parity_report, prec):
    """Items scaled by 2^20, 1, 2^-20 and 0 (both maps), checked item by item: fp16 operands are scaled per item
    (inv_scale[b] in the epilogue), and a normwise check would see only the largest item."""
    B, D, h, w, L = 4, 256, 24, 32, 4
    g = torch.Generator(device=cuda_device).manual_seed(20)
    s = torch.tensor([2.0 ** 20, 1.0, 2.0 ** -20, 0.0], device=cuda_device).view(B, 1, 1, 1)
    f1 = torch.randn(B, D, h, w, device=cuda_device, generator=g) * s
    f2 = torch.randn(B, D, h, w, device=cuda_device, generator=g) * s
    one, views, pools, last = run_build(f1, f2, L, prec)
    assert fused_from_launches(L, pools, last) == plan(h, w, L)[3]
    ref, mag = exact_and_magnitude(f1, f2, L)
    floor = f16_floor(f1, f2) if tc_kernel_name(prec, B, D, h, w) == "corr_tc_kernel<f16>" else None
    worst = check_levels(views, ref, mag, build_coefficient(prec, D), B, floor, f"per-item scale, {prec}")
    worst = max(worst, check_levels(one, ref, mag, build_coefficient(prec, D), B, floor, f"per-item scale, {prec}, levels=1"))
    for l in range(L):
        assert not views[l].view(B, -1)[3].any(), f"the zero item is not zero at level {l}"
    parity_report.add("corr_branches/build", branch="per-item scale 2^20, 1, 2^-20, 0", shape=f"{B}x{D}x{h}x{w}",
                      levels=L, precision=prec, worst_err_over_bound=worst)


@pytest.mark.parametrize("prec", ["tf32", "3xtf32", "auto"])
@pytest.mark.parametrize("h,w", [(60, 80), (24, 32)])
def test_build_misaligned_level2(cuda_device, parity_report, prec, h, w):
    """level2 one float off a 16-byte boundary turns the epilogue's level-2 pooling (pair2 at 60x80, deep at 24x32) off:
    the pooling kernels then produce more levels, and both builds meet the same element-wise bound."""
    B, D, L = 2, 256, 4
    g = torch.Generator(device=cuda_device).manual_seed(h + w)
    f1 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    f2 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    ref, mag = exact_and_magnitude(f1, f2, L)
    fused = {}
    for mis in (None, 2):
        _, views, pools, last = run_build(f1, f2, L, prec, misalign=mis)
        fused[mis] = fused_from_launches(L, pools, last)
        assert fused[mis] == plan(h, w, L, level2_aligned=mis is None)[3]
        worst = check_levels(views, ref, mag, build_coefficient(prec, D), B, None, f"level2 misaligned={mis is not None}")
        parity_report.add("corr_branches/build", branch=f"level2 misaligned={mis is not None}", shape=f"{B}x{D}x{h}x{w}",
                          levels=L, precision=prec, fused=fused[mis], pool_launches=pools, worst_err_over_bound=worst)
    assert fused[2] < fused[None], fused


# ------------------------------------------------------------------------------------------------ lookup sweep ---
def clamp_coords(c):
    """The kernels' clamp: fminf(fmaxf(c, -1e6), 1e6), which sends NaN to -1e6."""
    return torch.where(torch.isnan(c), torch.full_like(c, -1.0e6), c).clamp(-1.0e6, 1.0e6)


def ref_lookup(pyr, coords, r, with_magnitude=True, unit_weights=False):
    """Bilinear samples of the (2r+1)^2 window around coords / 2^l in float64, zero outside the map, channel
    l*(2r+1)^2 + i*(2r+1) + j at (x + i - r, y + j - r) (the transposed window).  Differentiable in pyr and coords.
    Also returns sum |w * p| and sum |p| over the four taps of each output element.  unit_weights: every tap weighs 1
    (its adjoint counts, per pyramid element, the output gradients that reach it)."""
    B, _, h, w = coords.shape
    N, K = h * w, 2 * r + 1
    P = K + 1
    dev = coords.device
    c = clamp_coords(coords.double())
    cx, cy = c[:, 0].reshape(B * N), c[:, 1].reshape(B * N)
    off = torch.arange(P, device=dev)
    rows = torch.arange(B * N, device=dev)[:, None, None]
    outs, mags = [], []
    for l, p in enumerate(pyr):
        Hl, Wl = p.shape[-2:]
        sx, sy = cx / 2 ** l, cy / 2 ** l
        x0, y0 = torch.floor(sx), torch.floor(sy)
        fx, fy = (sx - x0)[:, None, None], (sy - y0)[:, None, None]
        X = x0.long()[:, None] - r + off
        Y = y0.long()[:, None] - r + off
        ok = ((Y >= 0) & (Y < Hl))[:, :, None] & ((X >= 0) & (X < Wl))[:, None, :]
        idx = (rows * Hl + Y.clamp(0, Hl - 1)[:, :, None]) * Wl + X.clamp(0, Wl - 1)[:, None, :]
        patch = torch.where(ok, p.reshape(-1)[idx].double(), torch.zeros((), dtype=torch.float64, device=dev))  # [BN, y, x]
        ws = ((1 - fx) * (1 - fy), fx * (1 - fy), (1 - fx) * fy, fx * fy) if not unit_weights else (1.0,) * 4
        taps = (patch[:, :K, :K], patch[:, :K, 1:], patch[:, 1:, :K], patch[:, 1:, 1:])   # sample (i, j) -> [., j, i]
        o = sum(wk * t for wk, t in zip(ws, taps))
        outs.append(o.transpose(1, 2).reshape(B, N, K * K))
        if with_magnitude:
            m = sum(wk * t.abs() for wk, t in zip(ws, taps))
            a = sum(t.abs() for t in taps)
            mags.append(torch.stack([m, a]).detach().transpose(2, 3).reshape(2, B, N, K * K))
    out = torch.cat(outs, 2).permute(0, 2, 1).reshape(B, -1, h, w)
    if not with_magnitude:
        return out, None
    mag, tap = torch.cat(mags, 3).permute(0, 1, 3, 2).reshape(2, B, -1, h, w)
    return out, (mag, tap)


# A bilinear sample is <= 4 products w * p summed in fp32: under 8 units of 2^-24 of sum |w * p| (both the generic
# kernel's 4-FMA form and the radius-4 kernel's two lerps).  The fraction f = s - floor(s) is exact in fp32 except for
# -1 < s < 0, where s + 1 rounds by <= 2^-25, and 1 - f rounds by <= 2^-25 more: a weight can be off by 2^-23 in
# absolute terms (WEIGHT_ABS), however small it is, which adds 2^-23 * sum |p| over the four taps.
LOOKUP_COEF = 8 * U24
WEIGHT_ABS = 2.0 ** -23


def check_lookup(got, ref, mags, what):
    mag, tap = mags
    err = (got.double() - ref).abs()
    bound = LOOKUP_COEF * mag + WEIGHT_ABS * tap + 2.0 ** -149
    ratio = err / bound
    m = float(ratio.max())
    if not m <= 1.0:
        b, c, y, x = np.unravel_index(int(ratio.argmax()), tuple(got.shape))
        raise AssertionError(f"{what}: err/bound = {m:.3g} at (b={b}, channel={c}, y={y}, x={x}): "
                             f"got {float(got[b, c, y, x]):.9g}, exact {float(ref[b, c, y, x]):.9g}")
    return m


def lookup_coords(B, h, w, r, device, seed):
    """Per query, x and y each of one kind (x kind = q % 10, y kind = (q // 10) % 10): smooth flow, noise, exact
    integers, half-integers, windows partly outside, wholly outside, +-inf, NaN, far beyond the clamp, and
    within 1e-6 of an integer."""
    g = torch.Generator(device=device).manual_seed(seed)
    ys, xs = torch.meshgrid(torch.arange(h, device=device), torch.arange(w, device=device), indexing="ij")
    out = []
    for base, ext, kind in ((xs, w, torch.arange(h * w, device=device) % 10),
                            (ys, h, (torch.arange(h * w, device=device) // 10) % 10)):
        base = base.reshape(-1).float()[None].expand(B, -1)
        kind = kind[None].expand(B, -1)
        u = torch.rand(B, h * w, device=device, generator=g)
        n = torch.randn(B, h * w, device=device, generator=g)
        i = torch.randint(-3, ext + 3, (B, h * w), device=device, generator=g).float()
        side = torch.where(u < 0.5, -1.0, 1.0)
        choices = [
            base + 1.5 * torch.sin(base * 0.37) + 0.25 * n,               # smooth
            (ext + 2 * r + 6) * u - (r + 3),                               # noise
            i,                                                             # integers
            i + 0.5,                                                       # half-integers
            torch.where(u < 0.5, -r + 2 * r * u, ext - 1 + r * (2 * u - 1)) + 0.3,   # partly outside
            torch.where(u < 0.5, -40.0 * (r + 2) - 7.25 * u, ext + 40.0 * (r + 2) + 7.25 * u),  # wholly outside
            side * math.inf,
            torch.full_like(u, math.nan),
            side * (1.0e7 + 3.0e9 * u),                                    # far beyond the +-1e6 clamp
            i + torch.where(u < 0.5, 1.0e-6, -1.0e-6),                     # a hair off an integer
        ]
        val = torch.zeros_like(u)
        for k, ch in enumerate(choices):
            val = torch.where(kind == k, ch, val)
        out.append(val)
    return torch.stack(out, 1).reshape(B, 2, h, w).contiguous()


LB, LH, LW = 8, 48, 64     # B * ceil(N / 32) = 768 CTAs: the 32-query kernels; one item alone: the 16-query kernels


@pytest.fixture(scope="module")
def lookup_problem(cuda_device):
    sms = torch.cuda.get_device_properties(cuda_device).multi_processor_count
    N = LH * LW
    assert LB * -(-N // 32) >= 4 * sms and -(-N // 32) < 4 * sms, "the sizes no longer select both query counts"
    g = torch.Generator(device=cuda_device).manual_seed(77)
    pyr = [torch.randn(LB * N, 1, LH >> l, LW >> l, device=cuda_device, generator=g) for l in range(6)]
    return pyr


LOOKUP_CASES = [(L, r) for L in range(1, 7) for r in (0, 1, 2, 3, 4, 5, 7, 8)]


@pytest.mark.parametrize("levels,radius", LOOKUP_CASES)
def test_lookup_sweep(cuda_device, parity_report, lookup_problem, levels, radius):
    """The whole batch (32 queries per CTA, or the radius-4 kernel's balanced count) against float64, and item 0 alone
    (16 queries per CTA) bit-identical to it: the per-element arithmetic does not depend on the query count."""
    pyr = lookup_problem[:levels]
    N, K = LH * LW, 2 * radius + 1
    coords = lookup_coords(LB, LH, LW, radius, cuda_device, seed=10 * levels + radius)
    name = "corr_lookup_r4l4_kernel" if (levels, radius) == (4, 4) else "corr_lookup_kernel"
    buf, (out,) = guarded([(LB, levels * K * K, LH, LW)], cuda_device)
    cf.corr_lookup(pyr, coords, radius, out=out)
    assert last_kernel() == name
    buf1, (one,) = guarded([(1, levels * K * K, LH, LW)], cuda_device)
    cf.corr_lookup([p[:N] for p in pyr], coords[:1].contiguous(), radius, out=one)
    assert last_kernel() == name
    torch.cuda.synchronize()
    assert_written_and_guarded(buf, [out], "lookup, whole batch")
    assert_written_and_guarded(buf1, [one], "lookup, one item")
    ref, mag = ref_lookup(pyr, coords, radius)
    worst = check_lookup(out, ref, mag, f"levels={levels} radius={radius}")
    assert torch.equal(one.view(torch.int32), out[:1].view(torch.int32)), "16- and 32-query kernels differ"
    parity_report.add("corr_branches/lookup", levels=levels, radius=radius, worst_err_over_bound=worst)


_FORCED_QT_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
import torch
import cistaflow_b200 as cf
from cistaflow_b200 import _lib
B, h, w = 4, 37, 23
N = h * w
dev = torch.device("cuda", 0)
g = torch.Generator(device=dev).manual_seed(5)
pyr = [torch.randn(B * N, 1, h >> l, w >> l, device=dev, generator=g) for l in range(4)]
ys, xs = torch.meshgrid(torch.arange(h, device=dev), torch.arange(w, device=dev), indexing="ij")
coords = torch.stack([xs, ys]).float()[None] + 6 * torch.randn(B, 2, h, w, device=dev, generator=g)
out = cf.corr_lookup(pyr, coords, 4)
assert _lib.load().cf_last_kernel().decode() == "corr_lookup_r4l4_kernel"
torch.save(out.cpu(), sys.argv[2])
"""


def test_lookup_forced_query_counts(cuda_device, tmp_path):
    """CF_LOOKUP_QT (read once per process) at every even count 16..32 on N = 851 queries (a multiple of none of them):
    every count gives the same bits."""
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
    assert not torch.isnan(base).any()
    for qt, o in outs.items():
        assert torch.equal(o.view(torch.int32), base.view(torch.int32)), f"CF_LOOKUP_QT={qt}"


# ---------------------------------------------------------------------------------------------- backward sweep ---
BWD_CASES = [(23, 37, L, r) for L in (1, 3, 5) for r in (0, 1, 4, 8)] + [(23, 37, 4, 4), (33, 45, 6, 7), (33, 45, 6, 8)]


def backward_coords(B, h, w, device, seed):
    g = torch.Generator(device=device).manual_seed(seed)
    ys, xs = torch.meshgrid(torch.arange(h, device=device), torch.arange(w, device=device), indexing="ij")
    c = torch.stack([xs, ys]).float()[None] + 2.5 * torch.randn(B, 2, h, w, device=device, generator=g)
    c[0, :, 0, 0] = torch.tensor([-7.3, h + 5.2])         # window partly / wholly outside the map
    c[0, :, 0, 1] = torch.tensor([-60.5, 3.25])
    c[-1, :, 1, :5] = torch.tensor([3.0, 4.5, 7.0, 1.5, 9.0], device=device)   # integers and half-integers
    return c


def coord_grad_magnitude(pyr, coords, r, gabs):
    """Per query and axis: sum over channels of |g| * 2^-l * ((|p01| + |p00|)(1 - fy) + (|p11| + |p10|) fy) (x), the
    same with the roles of x and y swapped (y): what the kernel's coordinate-gradient sum is made of.  Also the sum over
    channels of |g| * 2^-l * (|p00| + |p01| + |p10| + |p11|), which scales the weights' absolute error."""
    B, _, h, w = coords.shape
    N, K = h * w, 2 * r + 1
    P = K + 1
    dev = coords.device
    c = coords.double()
    cx, cy = c[:, 0].reshape(B * N), c[:, 1].reshape(B * N)
    off = torch.arange(P, device=dev)
    rows = torch.arange(B * N, device=dev)[:, None, None]
    g = gabs.double().reshape(B, len(pyr), K, K, N).permute(0, 4, 1, 3, 2).reshape(B * N, len(pyr), K, K)  # [., l, j, i]
    mx = torch.zeros(B * N, dtype=torch.float64, device=dev)
    my, mt = torch.zeros_like(mx), torch.zeros_like(mx)
    for l, p in enumerate(pyr):
        Hl, Wl = p.shape[-2:]
        sx, sy = cx / 2 ** l, cy / 2 ** l
        x0, y0 = torch.floor(sx), torch.floor(sy)
        fx, fy = (sx - x0)[:, None, None], (sy - y0)[:, None, None]
        X = x0.long()[:, None] - r + off
        Y = y0.long()[:, None] - r + off
        ok = ((Y >= 0) & (Y < Hl))[:, :, None] & ((X >= 0) & (X < Wl))[:, None, :]
        idx = (rows * Hl + Y.clamp(0, Hl - 1)[:, :, None]) * Wl + X.clamp(0, Wl - 1)[:, None, :]
        a = torch.where(ok, p.reshape(-1)[idx].double().abs(), torch.zeros((), dtype=torch.float64, device=dev))
        a00, a01, a10, a11 = a[:, :K, :K], a[:, :K, 1:], a[:, 1:, :K], a[:, 1:, 1:]
        gl = g[:, l] / 2 ** l
        mx += (gl * ((a01 + a00) * (1 - fy) + (a11 + a10) * fy)).sum((1, 2))
        my += (gl * ((a10 + a00) * (1 - fx) + (a11 + a01) * fx)).sum((1, 2))
        mt += (gl * (a00 + a01 + a10 + a11)).sum((1, 2))
    return torch.stack([mx.view(B, h, w), my.view(B, h, w)], 1), mt.view(B, 1, h, w)


def near_integer(coords, levels, tol=1e-4):
    """Queries whose x or y fraction at some level is within tol of an integer: the sampled patch, and with it the
    coordinate gradient, jumps there."""
    m = torch.zeros(coords.shape[0], coords.shape[2], coords.shape[3], dtype=torch.bool, device=coords.device)
    for l in range(levels):
        s = coords.double() / 2 ** l
        f = s - torch.floor(s)
        m |= ((f < tol) | (f > 1 - tol)).any(1)
    return m


@pytest.mark.parametrize("mode", ["both", "coords", "pyramid"])
@pytest.mark.parametrize("h,w,levels,radius,B", [(*c, 2) for c in BWD_CASES] + [(36, 44, 4, 4, 4)])
def test_lookup_backward_sweep(cuda_device, parity_report, mode, h, w, levels, radius, B):
    """cf_corr_lookup_backward through CorrBlock against float64 autograd of the same gather, for both gradients, the
    coordinate gradient alone (pyramid built without grad) and the pyramid gradient alone (coordinates without grad)."""
    D, N, K = 32, h * w, 2 * radius + 1
    g = torch.Generator(device=cuda_device).manual_seed(h * 100 + levels * 10 + radius)
    f1 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    f2 = torch.randn(B, D, h, w, device=cuda_device, generator=g)
    coords = backward_coords(B, h, w, cuda_device, seed=radius + 7 * levels)
    gout = torch.randn(B, levels * K * K, h, w, device=cuda_device, generator=g)
    want_pyr, want_coords = mode in ("both", "pyramid"), mode in ("both", "coords")
    if want_pyr:
        f1.requires_grad_()
        f2.requires_grad_()
        blk = cf.CorrBlock(f1, f2, num_levels=levels, radius=radius)
        for p in blk.corr_pyramid:
            p.retain_grad()
    else:
        with torch.no_grad():
            blk = cf.CorrBlock(f1, f2, num_levels=levels, radius=radius)
    if want_coords:
        coords.requires_grad_()
    out = blk(coords)
    out.backward(gout)
    assert last_kernel() == "corr_lookup_backward_kernel"
    assert (coords.grad is not None) == want_coords

    pyr_d = [p.detach().double().requires_grad_() for p in blk.corr_pyramid]
    cd = coords.detach().double().requires_grad_()
    ref, _ = ref_lookup(pyr_d, cd, radius, with_magnitude=False)
    ref_gp = torch.autograd.grad(ref, [*pyr_d, cd], gout.double())
    report = {}
    if want_pyr:
        ga = gout.double().abs()
        mags = torch.autograd.grad(ref_lookup(pyr_d, cd.detach(), radius, with_magnitude=False)[0], pyr_d, ga)
        taps = torch.autograd.grad(ref_lookup(pyr_d, cd.detach(), radius, False, unit_weights=True)[0], pyr_d, ga)
        # each patch element is <= 4 products g * w summed: 8 units of 2^-24 of sum |g * w|, plus WEIGHT_ABS * sum |g|
        # for the weights' absolute error.  An element outside every query's patch has a zero bound and must be exactly 0.
        report["pyramid"] = check_levels([p.grad for p in blk.corr_pyramid], ref_gp[:levels], mags, 8 * U24, B, None,
                                         "pyramid gradient", extra=[WEIGHT_ABS * t for t in taps])
    if want_coords:
        mag, tap = coord_grad_magnitude([p.detach() for p in blk.corr_pyramid], coords.detach(), radius, gout.abs())
        # per thread ceil(L K^2 / 16) or fewer sums, <= 32 threads per query into shared memory, ~8 roundings per term
        coef = (levels * -(-K * K // 16) + 32 + 8) * U24
        keep = ~near_integer(coords.detach(), levels)[:, None].expand(-1, 2, -1, -1)
        err = (coords.grad.double() - ref_gp[levels]).abs()
        ratio = (err / (coef * mag + WEIGHT_ABS * tap + 2.0 ** -149))[keep]
        masked = int((~keep).sum()) // 2
        assert masked < B * N // 4, f"{masked} of {B * N} queries masked"
        worst = float(ratio.max())
        assert worst <= 1.0, f"coordinate gradient: err/bound = {worst:.3g} ({masked} queries masked)"
        report["coords"] = worst
        report["coords_masked"] = masked
    parity_report.add("corr_branches/lookup_backward", mode=mode, shape=f"{B}x{h}x{w}", levels=levels, radius=radius,
                      **report)


@pytest.mark.parametrize("h,w,levels", [(16, 29, 5), (33, 61, 6)])
def test_pyramid_backward_levels(cuda_device, h, w, levels):
    """_PyramidFunction.backward (the avg-pool adjoint into level 0, then two GEMMs) against float64 autograd of the
    exact pyramid at 5 and 6 levels, with odd sizes whose floored rows and columns get no gradient."""
    B, D = 2, 32
    N = h * w
    g = torch.Generator(device=cuda_device).manual_seed(h * w + levels)
    f1 = torch.randn(B, D, h, w, device=cuda_device, generator=g).requires_grad_()
    f2 = torch.randn(B, D, h, w, device=cuda_device, generator=g).requires_grad_()
    grads = [torch.randn(B * N, 1, h >> l, w >> l, device=cuda_device, generator=g) for l in range(levels)]
    blk = cf.CorrBlock(f1, f2, num_levels=levels, radius=1, precision="3xtf32")
    sum((gl * p).sum() for gl, p in zip(grads, blk.corr_pyramid)).backward()

    d1, d2 = f1.detach().double().requires_grad_(), f2.detach().double().requires_grad_()
    exact, _ = exact_and_magnitude(d1, d2, levels)
    sum((gl.double() * p).sum() for gl, p in zip(grads, exact)).backward()
    # magnitude: |f2| . |G|^T / sqrt(D) (and |f1| . |G|) with |G| the adjoint of the |grads|, through autograd
    vol = torch.zeros(B * N, 1, h, w, dtype=torch.float64, device=cuda_device, requires_grad=True)
    (G,) = torch.autograd.grad(sum((gl.double().abs() * p).sum() for gl, p in zip(grads, pool_levels(vol, levels))), vol)
    G = G.reshape(B, N, N)
    a1, a2 = d1.detach().abs().reshape(B, D, N), d2.detach().abs().reshape(B, D, N)
    s = float(D) ** 0.5
    m1 = (a2 @ G.transpose(1, 2) / s).reshape(B, D, h, w)
    m2 = (a1 @ G / s).reshape(B, D, h, w)
    # fp32: the adjoint adds <= levels roundings per element, each GEMM sums N products (gamma_N); factor 2
    coef = 2 * (N + 2 * levels) * U24
    for got, ref, m, name in ((f1.grad, d1.grad, m1, "fmap1"), (f2.grad, d2.grad, m2, "fmap2")):
        ratio = (got.double() - ref).abs() / (coef * m + 2.0 ** -149)
        assert float(ratio.max()) <= 1.0, f"grad {name}: err/bound = {float(ratio.max()):.3g}"
