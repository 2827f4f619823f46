"""The warp forward and both warp adjoints on every branch of their dispatch, element by element against float64.

The kernels compute the sample position in fp32 with ATen CUDA's operation sequence (warp_common.cuh: make_taps,
grad_pos): (x + sign*u) / W, - 0.5, * 2, then ((g + 1) / 2) * (W - 1), reflect (fmod, floor(a / span)) and clip with
fmaxf / fminf, so NaN goes to 0.  ``positions32`` restates that sequence in numpy float32, so for a flow at the
image's resolution the reference has the kernel's taps and lambdas bit for bit.  The lambdas ix - x0 and (x0 + 1) - ix
are exact in fp32; everything after them (weights, products, sums) is float64.

Bounds (u = 2^-24).  Each is derived from the arithmetic, asserted per (batch item, channel group), and a zero bound
demands an exact zero:
  * forward:      |got - ref| <= 8u * sum_k |w_k v_k|: one rounding per weight product and a four-term FMA chain.
  * fused flows:  the x0.5 down-sampled and the upflow8 flow are rounded bilinear sums the compiler may contract, so
                  they are not emulated.  Their lambdas are (fp32, exactly); the flow is summed in float64 and its error
                  is at most e = 4u * sum |lambda p| (x8 for upflow8, which scales by 8; through both stages for the
                  codes of the upflow8 step).  The position then is within
                      delta = e + 8u * (|x + sign*u| + W)
                  of the float64 position (the flow error times (W-1)/W < 1, plus at most 7 roundings of the position
                  chain, each < u * (|x + sign*u| + W)); reflect and clip are 1-Lipschitz.  The forward bound gains
                  delta_x * L_x + delta_y * L_y, with L the largest difference of neighbouring pixels around the taps
                  (the Lipschitz constant of the bilinear interpolant there).
  * flow_out:     upflow8 + unpad against float64 with the kernel's fp32 lambdas: 4u * 8 * sum |lambda p|.
  * grad_img:     a float64 scatter of g_p * w_k; a cell that receives n terms is within gamma_(n+1) sum |g w|, with
                  gamma_k = k u / (1 - k u) (the weight product, g * w and n - 1 additions round) -- any summation
                  order, so it holds for the atomic and the fixed-order sum.  A one-term cell reaches ~0.98 of it.  Half-resolution flow: every cell
                  a tap of a position within delta can reach counts towards n and receives |g| (delta_x + delta_y).
  * grad_flow:    gu = sign * 2 * mx * gix / W with gix = sum_c g_c (-v00 ay1 + v01 ay1 - v10 ay0 + v11 ay0) and mx
                  source_index_set_grad's multiplier, +-(W-1)/2, 0 on and beyond the clip border;
                  |err| <= (C + 8) u |2 mx / W| sum_c |g_c| (|v00| ay1 + |v01| ay1 + |v10| ay0 + |v11| ay0), likewise
                  for y.  Half-resolution flow: gu is continuous in iy with slope <= |2 mx / W| sum_c |g_c (v00 - v01 -
                  v10 + v11)|, which adds delta_y times that; the x0.5 adjoint adds (n + 3) u sum |lambda gu| for an
                  element that receives n terms.  gu jumps in ix (a tap boundary, a reflection, a clip border): where
                  the float64 position lies within delta_x of one, the reference is evaluated on both sides
                  (pre-reflection position -+ delta_x) and the kernel must lie within the bound of the interval they
                  span.  Nothing else is excused.

Outputs go into NaN-filled views with guard regions (guarded_buffers.py): an element left unwritten stays NaN, a stray
write changes a guard.  Each forward row names its branch and proves it: cf_last_kernel() names the kernel, ``route``
restates the host predicates of launch_warp_tma, and ``tile_mix`` restates the per-tile box test where a row is meant
to mix ring and fallback tiles."""
import math
import os
import subprocess
import sys
from collections import namedtuple

import numpy as np
import pytest
import torch

from guarded_buffers import assert_written_and_guarded, guarded

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
U24 = 2.0 ** -24
INT_MAX = 2 ** 31 - 1
TW, TH, BW, BH, CH_PER_CTA = 32, 16, 48, 24, 64     # warp_tma.cu: output tile, source box, channels per CTA


# ------------------------------------------------------------------------------------ fp32 position emulation ---
def reflect_clip32(v, size):
    """reflect_clip of warp_common.cuh on float32: fast path a < span, else fmod and floor(a / span) (converted with
    saturation, NaN -> 0, as (int) does on the device), then fminf(span, fmaxf(r, 0)): NaN and +-inf end at 0."""
    v = np.asarray(v, F32)
    if size == 1:
        return np.zeros_like(v)
    span = F32(size - 1)
    a = np.abs(v)
    with np.errstate(invalid="ignore", over="ignore"):
        extra = np.fmod(a, span).astype(F32)
        q = np.floor((a / span).astype(F32)).astype(np.float64)
    flips = np.where(np.isnan(q), 0.0, np.minimum(q, INT_MAX)).astype(np.int64)
    r = np.where(a < span, a, np.where(flips & 1, span - extra, extra)).astype(F32)
    return np.fmin(span, np.fmax(r, F32(0))).astype(F32)


def pre_position32(coord, flow, size, sign):
    """((g + 1) / 2) * (size - 1), g = 2 * ((coord + sign * flow) / size - 0.5), in the kernel's fp32 order."""
    with np.errstate(invalid="ignore", over="ignore"):
        t = (F32(coord) + F32(sign) * np.asarray(flow, F32)).astype(F32)
        g = (F32(2) * ((t / F32(size)).astype(F32) - F32(0.5))).astype(F32)
        return (((g + F32(1)) / F32(2)).astype(F32) * F32(size - 1)).astype(F32)


def grad_mult32(pre, size):
    """source_index_set_grad's multiplier: -1 for a negative position, flipped by an odd reflection, times
    (size - 1) / 2; 0 on and beyond the clip borders and for a one-pixel axis."""
    pre = np.asarray(pre, F32)
    if size == 1:
        return np.zeros_like(pre)
    span = F32(size - 1)
    m = np.where(pre < 0, F32(-1), F32(1))
    a = np.abs(pre)
    with np.errstate(invalid="ignore", over="ignore"):
        extra = np.fmod(a, span).astype(F32)
        q = np.floor((a / span).astype(F32)).astype(np.float64)
    flips = np.where(np.isnan(q), 0.0, np.minimum(q, INT_MAX)).astype(np.int64)
    m = np.where(flips & 1, -m, m)
    r = np.where(flips & 1, span - extra, extra)
    m = np.where((r <= 0) | (r >= span), F32(0), m)
    return (m * F32(span / 2)).astype(F32)


def grid32(B, H, W):
    return (np.broadcast_to(np.arange(W, dtype=F32)[None, None, :], (B, H, W)),
            np.broadcast_to(np.arange(H, dtype=F32)[None, :, None], (B, H, W)))


def positions32(u, v, sign):
    """The kernel's (ix, iy, mx, my) for a flow (u, v) [B, H, W] at the output's resolution, float32."""
    B, H, W = u.shape
    xs, ys = grid32(B, H, W)
    px, py = pre_position32(xs, u, W, sign), pre_position32(ys, v, H, sign)
    return reflect_clip32(px, W), reflect_clip32(py, H), grad_mult32(px, W), grad_mult32(py, H)


# ------------------------------------------------------------------------------------- float64 positions ---
def reflect_clip64(pre, size):
    """reflect + clip in float64 (non-finite -> 0, as the kernels do), and the multiplier of source_index_set_grad."""
    pre = np.asarray(pre, np.float64)
    if size == 1:
        return np.zeros_like(pre), np.zeros_like(pre)
    span = float(size - 1)
    fin = np.isfinite(pre)
    p = np.where(fin, pre, 0.0)
    a = np.abs(p)
    flips = np.floor(a / span)
    extra = a - flips * span
    odd = np.mod(flips, 2) == 1
    r = np.where(odd, span - extra, extra)
    m = np.where(p < 0, -1.0, 1.0) * np.where(odd, -1.0, 1.0)
    m = np.where((r <= 0) | (r >= span) | ~fin, 0.0, m) * span / 2
    return np.clip(np.where(fin, r, 0.0), 0.0, span), m


def pre_position64(coord, flow, size, sign):
    with np.errstate(invalid="ignore", over="ignore"):
        return (coord + sign * np.asarray(flow, np.float64)) / size * (size - 1)


def position_delta(coord, flow, size, sign, ferr):
    """delta of the module docstring: the flow error plus the roundings of the fp32 position chain."""
    with np.errstate(invalid="ignore", over="ignore"):
        d = ferr + 8 * U24 * (np.abs(coord + sign * np.asarray(flow, np.float64)) + size)
    return np.where(np.isfinite(d), d, 0.0)


# ---------------------------------------------------------------------------------------- fused flow fields ---
def half_lambdas(n, fn):
    """half_taps along one axis: i0, i1 and the fp32 lambdas l0, l1 of the x0.5 down-sampling of fn to n samples."""
    s = F32(fn - 1) / F32(n - 1) if n > 1 else F32(0)
    f = (F32(s) * np.arange(n, dtype=F32)).astype(F32)
    i0 = np.minimum(f.astype(np.int64), fn - 1)
    i1 = i0 + (i0 < fn - 1)
    l1 = np.clip(f - i0.astype(F32), F32(0), F32(1)).astype(F32)
    return i0, i1, (F32(1) - l1).astype(F32), l1


def up8_lambdas(n, ln, pad):
    """upflow8_at along one axis: taps and fp32 lambdas at destinations pad .. pad + n - 1 of the x8 grid."""
    s = F32(ln - 1) / F32(8 * ln - 1) if 8 * ln > 1 else F32(0)
    f = (F32(s) * (np.arange(n) + pad).astype(F32)).astype(F32)
    i0 = np.minimum(f.astype(np.int64), ln - 1)
    i1 = i0 + (i0 < ln - 1)
    l1 = np.clip(f - i0.astype(F32), F32(0), F32(1)).astype(F32)
    return i0, i1, (F32(1) - l1).astype(F32), l1


def resample64(field, ly, lx, scale=1.0, ferr=None):
    """sum lambda * p in float64 over [B, 2, n, m] fields, with the rounding bound 4u * sum |lambda p| (times scale)
    and, when ``ferr`` is given, the propagated error sum lambda * ferr of the input field."""
    y0, y1, ly0, ly1 = ly
    x0, x1, lx0, lx1 = lx
    f = np.asarray(field, np.float64)
    out = np.zeros(f.shape[:2] + (len(y0), len(x0)))
    mag = np.zeros_like(out)
    err = np.zeros_like(out)
    for yi, wy in ((y0, ly0), (y1, ly1)):
        for xi, wx in ((x0, lx0), (x1, lx1)):
            w = wy.astype(np.float64)[:, None] * wx.astype(np.float64)[None, :]
            p = f[:, :, yi][:, :, :, xi]
            with np.errstate(invalid="ignore"):
                out += w * p
                mag += np.abs(w * p)
            if ferr is not None:
                err += w * ferr[:, :, yi][:, :, :, xi]
    with np.errstate(invalid="ignore"):
        return scale * out, scale * 4 * U24 * mag + err


def half_flow64(flow, H, W):
    """The x0.5 down-sampled flow at [H, W] from [B, 2, fH, fW] (fp32 lambdas, float64 sums) and its error bound."""
    fH, fW = flow.shape[2:]
    return resample64(flow, half_lambdas(H, fH), half_lambdas(W, fW))


def upflow8_64(lr, H, W, pad_h, pad_w):
    lh, lw = lr.shape[2:]
    return resample64(lr, up8_lambdas(H, lh, pad_h), up8_lambdas(W, lw, pad_w), scale=8.0)


# ---------------------------------------------------------------------------------------------- references ---
Pos = namedtuple("Pos", "ix iy mx my dx dy")   # float32 or float64 positions [B,H,W], multipliers, position bounds


def exact_pos(u, v, sign):
    B, H, W = u.shape
    ix, iy, mx, my = positions32(u, v, sign)
    z = np.zeros((B, H, W))
    return Pos(ix, iy, mx, my, z, z)


def approx_pos(u, v, eu, ev, sign):
    """Positions from a float64 flow with error bounds (eu, ev)."""
    B, H, W = u.shape
    xs, ys = np.arange(W)[None, None, :], np.arange(H)[None, :, None]
    ix, mx = reflect_clip64(pre_position64(xs, u, W, sign), W)
    iy, my = reflect_clip64(pre_position64(ys, v, H, sign), H)
    return Pos(ix, iy, mx, my, position_delta(xs, u, W, sign, eu), position_delta(ys, v, H, sign, ev))


def _t(a, dev):
    return torch.as_tensor(np.ascontiguousarray(a), device=dev)


def taps64(ix, iy, H, W, dev):
    """x0, y0, and the float64 lambdas of positions ix, iy (any float dtype; the differences are exact)."""
    ix, iy = _t(ix, dev).double(), _t(iy, dev).double()
    fx, fy = torch.floor(ix), torch.floor(iy)
    return fx.long(), fy.long(), ix - fx, (fx + 1) - ix, iy - fy, (fy + 1) - iy


def _gather(img, yy, xx):
    """img [B, C, H, W] float64 at per-pixel (yy, xx) [B, h, w] -> [B, C, h, w]."""
    B, C, H, W = img.shape
    idx = (yy * W + xx).reshape(B, 1, -1).expand(B, C, -1)
    return img.reshape(B, C, H * W).gather(2, idx).reshape(B, C, *yy.shape[1:])


def _window_max(d, x0, y0, kx, ky):
    """max of d [B, C, h', w'] over rows y0 - 1 .. y0 + ky - 2 and columns x0 - 1 .. x0 + kx - 2 at every pixel."""
    B, C = d.shape[:2]
    p = torch.nn.functional.pad(d, (1, kx, 1, ky))
    m = torch.nn.functional.max_pool2d(p, (ky, kx), stride=1)
    return _gather(m, y0.clamp(0, m.shape[2] - 1), x0.clamp(0, m.shape[3] - 1))


def forward_ref(img, pos):
    """(out, bound) in float64 for img [B, C, H, W] (torch, any device) at the positions ``pos``."""
    B, C, H, W = img.shape
    dev = img.device
    x0, y0, ax0, ax1, ay0, ay1 = taps64(pos.ix, pos.iy, H, W, dev)
    x1, y1 = (x0 + 1).clamp(max=W - 1), (y0 + 1).clamp(max=H - 1)
    im = img.double()
    out = torch.zeros(B, C, *x0.shape[1:], dtype=torch.float64, device=dev)
    mag = torch.zeros_like(out)
    for yy, xx, w in ((y0, x0, ax1 * ay1), (y0, x1, ax0 * ay1), (y1, x0, ax1 * ay0), (y1, x1, ax0 * ay0)):
        t = _gather(im, yy, xx) * w[:, None]
        out += t
        mag += t.abs()
    bound = 8 * U24 * mag
    if np.any(pos.dx) or np.any(pos.dy):
        dx, dy = _t(pos.dx, dev)[:, None], _t(pos.dy, dev)[:, None]
        Lx = _window_max((im[..., 1:] - im[..., :-1]).abs(), x0, y0, 3, 4) if W > 1 else 0
        Ly = _window_max((im[..., 1:, :] - im[..., :-1, :]).abs(), x0, y0, 4, 3) if H > 1 else 0
        bound = bound + dx * Lx + dy * Ly
    return out, bound


def check(got, ref, bound, what, group=None):
    """max |got - ref| / bound <= 1 per (batch item, channel group of ``group`` channels); returns the worst ratio."""
    got = got.double().to(ref.device)
    B, C = ref.shape[:2]
    group = group or C
    worst = 0.0
    for b in range(B):
        for c0 in range(0, C, group):
            e = (got[b, c0:c0 + group] - ref[b, c0:c0 + group]).abs()
            bd = bound[b, c0:c0 + group] if bound.dim() == ref.dim() else bound[b]
            r = torch.where(bd > 0, e / bd.clamp_min(1e-300),
                            torch.where(e > 0, torch.full_like(e, math.inf), torch.zeros_like(e)))
            r = torch.where(torch.isnan(e), torch.full_like(e, math.inf), r)
            m = float(r.max()) if r.numel() else 0.0
            if not m <= 1.0:
                idx = np.unravel_index(int(r.reshape(-1).argmax()), tuple(r.shape))
                raise AssertionError(f"{what}: item {b} channels {c0}..: err/bound = {m:.3g} at {idx}: got "
                                     f"{float(got[b, c0:c0 + group][idx]):.9g}, exact {float(ref[b, c0:c0 + group][idx]):.9g}, "
                                     f"bound {float(bd[idx] if bd.dim() == r.dim() else 0):.3g}")
            worst = max(worst, m)
    return worst


# ------------------------------------------------------------------------------------- adjoint references ---
def _scatter(vals, cells, n):
    """sum of vals [B, C, P] into cells [B, P] (flat indices < n) per (b, c), float64."""
    B, C, P = vals.shape
    out = torch.zeros(B, C, n, dtype=torch.float64, device=vals.device)
    return out.scatter_add_(2, cells[:, None].expand(B, C, P), vals)


def _sides(pre, size, d):
    """(taps, multiplier) changes within d of the float64 pre-reflection position: returns the positions and
    multipliers at pre - d and pre + d, and where either side differs from the centre in floor(ix) or multiplier."""
    c, mc = reflect_clip64(pre, size)
    lo, ml = reflect_clip64(pre - d, size)
    hi, mh = reflect_clip64(pre + d, size)
    amb = (np.floor(lo) != np.floor(c)) | (np.floor(hi) != np.floor(c)) | (ml != mc) | (mh != mc)
    return (lo, ml), (hi, mh), amb & (d > 0)


def grad_flow_pixel(img, gout, ix, iy, mx, my, sign):
    """Per output pixel: (gu, gv) in float64 and their bounds without the delta terms, and the cross-derivative
    magnitudes for the delta terms."""
    B, C, H, W = img.shape
    dev = img.device
    x0, y0, ax0, ax1, ay0, ay1 = taps64(ix, iy, H, W, dev)
    xin, yin = (x0 + 1 < W)[:, None], (y0 + 1 < H)[:, None]
    im, g = img.double(), gout.double()
    x1, y1 = (x0 + 1).clamp(max=W - 1), (y0 + 1).clamp(max=H - 1)
    v00 = _gather(im, y0, x0)
    v01 = torch.where(xin, _gather(im, y0, x1), 0.0)
    v10 = torch.where(yin, _gather(im, y1, x0), 0.0)
    v11 = torch.where(xin & yin, _gather(im, y1, x1), 0.0)
    ax0, ax1, ay0, ay1 = (a[:, None] for a in (ax0, ax1, ay0, ay1))
    gix = (g * (-v00 * ay1 + v01 * ay1 - v10 * ay0 + v11 * ay0)).sum(1)
    giy = (g * (-v00 * ax1 - v01 * ax0 + v10 * ax1 + v11 * ax0)).sum(1)
    ga = g.abs()
    mgx = (ga * (v00.abs() * ay1 + v01.abs() * ay1 + v10.abs() * ay0 + v11.abs() * ay0)).sum(1)
    mgy = (ga * (v00.abs() * ax1 + v01.abs() * ax0 + v10.abs() * ax1 + v11.abs() * ax0)).sum(1)
    cross = (g * (v00 - v01 - v10 + v11)).abs().sum(1)
    kx, ky = 2 * _t(mx, dev).double() / W, 2 * _t(my, dev).double() / H
    coef = (C + 8) * U24
    return sign * kx * gix, sign * ky * giy, coef * kx.abs() * mgx, coef * ky.abs() * mgy, kx.abs() * cross, ky.abs() * cross


def backward_ref(img, gout, pos, sign, flow_shape=None):
    """float64 references and bounds of both gradients.  ``flow_shape`` (fH, fW) != (H, W): the flow gradient goes
    through the adjoint of the x0.5 down-sampling, with the either-side rule.  Returns (grad_img, bound_img,
    grad_flow_lo, grad_flow_hi, bound_flow, either_side_elements)."""
    B, C, H, W = img.shape
    dev = img.device
    g = gout.double()
    # grad_img: the centre taps, plus every cell a tap of a position within delta can reach
    x0, y0, ax0, ax1, ay0, ay1 = taps64(pos.ix, pos.iy, H, W, dev)
    xin, yin = x0 + 1 < W, y0 + 1 < H
    flat = lambda yy, xx: (yy.clamp(0, H - 1) * W + xx.clamp(0, W - 1)).reshape(B, -1)   # noqa: E731
    gf = g.reshape(B, C, -1)
    ref = torch.zeros(B, C, H * W, dtype=torch.float64, device=dev)
    mag = torch.zeros_like(ref)
    for yy, xx, w, ok in ((y0, x0, ax1 * ay1, None), (y0, x0 + 1, ax0 * ay1, xin), (y0 + 1, x0, ax1 * ay0, yin),
                          (y0 + 1, x0 + 1, ax0 * ay0, xin & yin)):
        w = w if ok is None else torch.where(ok, w, 0.0)
        t = gf * w.reshape(B, 1, -1)
        ref += _scatter(t, flat(yy, xx), H * W)
        mag += _scatter(t.abs(), flat(yy, xx), H * W)
    dx, dy = _t(pos.dx, dev).double(), _t(pos.dy, dev).double()
    ixd, iyd = _t(pos.ix, dev).double(), _t(pos.iy, dev).double()
    xlo, xhi = torch.floor(ixd - dx).clamp(min=0).long(), (torch.floor(ixd + dx) + 1).clamp(max=W - 1).long()
    ylo, yhi = torch.floor(iyd - dy).clamp(min=0).long(), (torch.floor(iyd + dy) + 1).clamp(max=H - 1).long()
    count = torch.zeros(B, H * W, dtype=torch.float64, device=dev)
    extra = torch.zeros_like(ref)
    spread = gf.abs() * (dx + dy).reshape(B, 1, -1)
    one = torch.ones(B, x0.numel() // B, dtype=torch.float64, device=dev)
    for oy in range(3):
        for ox in range(3):
            ok = ((ylo + oy <= yhi) & (xlo + ox <= xhi)).reshape(B, -1)
            cells = flat(ylo + oy, xlo + ox)
            count.scatter_add_(1, cells, torch.where(ok, one, 0.0))
            if bool(dx.any() or dy.any()):
                extra += _scatter(torch.where(ok[:, None], spread, 0.0), cells, H * W)
    k = (count[:, None] + 1) * U24
    bound_img = (k / (1 - k) * (mag + extra) + extra).reshape(B, C, H, W)

    # grad_flow per output pixel, with the either-side rule along each axis where delta > 0
    gu, gv, bu, bv, cu, cv = grad_flow_pixel(img, gout, pos.ix, pos.iy, pos.mx, pos.my, sign)
    bu, bv = bu + cu * dy, bv + cv * dx
    lo, hi = [gu, gv], [gu.clone(), gv.clone()]
    amb_any = torch.zeros_like(gu, dtype=torch.bool)
    if pos.dx.any() or pos.dy.any():
        xs, ys = np.arange(W)[None, None, :], np.arange(H)[None, :, None]
        for axis, (coord, size, d) in enumerate(((xs, W, pos.dx), (ys, H, pos.dy))):
            # recover the pre-reflection position from the flow through the stored sides of approx_pos
            pre = pos.pre[axis]
            side_lo, side_hi, amb = _sides(pre, size, d)
            amb_t = _t(amb, dev)
            amb_any |= amb_t
            for (p, m) in (side_lo, side_hi):
                args = [pos.ix, pos.iy, pos.mx, pos.my]
                args[axis], args[2 + axis] = p, m
                val = grad_flow_pixel(img, gout, *args, sign)[axis]
                lo[axis] = torch.where(amb_t, torch.minimum(lo[axis], val), lo[axis])
                hi[axis] = torch.where(amb_t, torch.maximum(hi[axis], val), hi[axis])
    if flow_shape is None or tuple(flow_shape) == (H, W):
        return (ref.reshape(B, C, H, W), bound_img, torch.stack(lo, 1), torch.stack(hi, 1), torch.stack([bu, bv], 1), 0)
    fH, fW = flow_shape
    y0h, y1h, ly0, ly1 = half_lambdas(H, fH)
    x0h, x1h, lx0, lx1 = half_lambdas(W, fW)
    flo = torch.zeros(B, 2, fH * fW, dtype=torch.float64, device=dev)
    fhi, fmag, fb, fcount = torch.zeros_like(flo), torch.zeros_like(flo), torch.zeros_like(flo), torch.zeros_like(flo)
    famb = torch.zeros_like(flo)
    pl, ph, pb = torch.stack(lo, 1).reshape(B, 2, -1), torch.stack(hi, 1).reshape(B, 2, -1), torch.stack([bu, bv], 1).reshape(B, 2, -1)
    pa = amb_any.reshape(B, 1, -1).double().expand(B, 2, -1)
    for yi, wy in ((y0h, ly0), (y1h, ly1)):
        for xi, wx in ((x0h, lx0), (x1h, lx1)):
            lam = _t((wy.astype(np.float64)[:, None] * wx.astype(np.float64)[None, :]).reshape(1, 1, -1), dev)
            cells = _t((yi[:, None] * fW + xi[None, :]).reshape(1, -1), dev).expand(B, -1)
            flo += _scatter(lam * pl, cells, fH * fW)
            fhi += _scatter(lam * ph, cells, fH * fW)
            fmag += _scatter(lam * torch.maximum(pl.abs(), ph.abs()), cells, fH * fW)
            fb += _scatter(lam * pb, cells, fH * fW)
            fcount += _scatter(torch.ones_like(pl), cells, fH * fW)
            famb += _scatter(pa, cells, fH * fW)
    bound = fb + (fcount + 3) * U24 * fmag
    sh = (B, 2, fH, fW)
    return (ref.reshape(B, C, H, W), bound_img, flo.reshape(sh), fhi.reshape(sh), bound.reshape(sh),
            int((famb[:, :1] > 0).sum()) * 2)


def approx_pos_with_pre(u, v, eu, ev, sign):
    p = approx_pos(u, v, eu, ev, sign)
    B, H, W = u.shape
    p = PosPre(*p, pre=(pre_position64(np.arange(W)[None, None, :], u, W, sign),
                        pre_position64(np.arange(H)[None, :, None], v, H, sign)))
    return p


PosPre = namedtuple("PosPre", Pos._fields + ("pre",))


def check_interval(got, lo, hi, bound, what):
    """got within bound of the interval [lo, hi], per batch item and flow channel; returns the worst ratio."""
    got = got.double().to(lo.device)
    e = torch.clamp(torch.maximum(lo - got, got - hi), min=0)
    zero = torch.zeros_like(e)
    worst = 0.0
    for b in range(got.shape[0]):
        for k in range(2):
            r = torch.where(bound[b, k] > 0, e[b, k] / bound[b, k].clamp_min(1e-300),
                            torch.where(e[b, k] > 0, torch.full_like(e[b, k], math.inf), zero[b, k]))
            r = torch.where(torch.isnan(got[b, k]), torch.full_like(r, math.inf), r)
            m = float(r.max())
            if not m <= 1.0:
                idx = np.unravel_index(int(r.reshape(-1).argmax()), tuple(r.shape))
                raise AssertionError(f"{what}: item {b} flow channel {k}: err/bound = {m:.3g} at {idx}: got "
                                     f"{float(got[b, k][idx]):.9g}, exact [{float(lo[b, k][idx]):.9g}, "
                                     f"{float(hi[b, k][idx]):.9g}], bound {float(bound[b, k][idx]):.3g}")
            worst = max(worst, m)
    return worst


# ------------------------------------------------------------------------------ host predicate restatement ---
def cdiv(a, b):
    return -(-a // b)


def route(B, C, H, W, aligned, sms, quad_env=None, path_direct=False):
    """launch_warp_tma's choice for a codes job [B, C, H, W]: None (the direct kernels) or the channel stride P of
    the staged kernel (P > 1 only for the quad-row tensor map, which serves W % 4 != 0)."""
    if path_direct or C < 8 or not aligned:
        return None
    quad = W % 4 != 0
    if quad:
        ctas = cdiv(W, TW) * cdiv(H, TH) * cdiv(C, CH_PER_CTA) * B
        if (C % 32 or W < 16 or H < BH or (ctas < 3 * sms and quad_env != "1") or B * C * H > INT_MAX
                or quad_env == "0"):
            return None
        return 1 if H % 4 == 0 else (4 if H % 2 else 2)
    return 1


def in_tiles(Hi, Wi, B, C, H, W, sms, image_ctas_env=False):
    """The image of the frame step rides in the first channel group's CTA of each codes tile."""
    ctas = cdiv(W, TW) * cdiv(H, TH) * cdiv(C, CH_PER_CTA) * B
    return Hi == 2 * H and Wi == 2 * W and ctas > 6 * sms and not image_ctas_env


def tile_mix(ix, iy, quad):
    """(ring tiles, fallback tiles) of the per-tile box test on taps from positions ix, iy [B, H, W]."""
    B, H, W = ix.shape
    x0 = np.floor(np.asarray(ix, np.float64)).astype(np.int64)
    y0 = np.floor(np.asarray(iy, np.float64)).astype(np.int64)
    x1, y1 = np.minimum(x0 + 1, W - 1), np.minimum(y0 + 1, H - 1)
    th, tw = cdiv(H, TH) * TH, cdiv(W, TW) * TW
    big, small = np.iinfo(np.int64).max, -1

    def tiles(a, fill):
        p = np.full((B, th, tw), fill, np.int64)
        p[:, :H, :W] = a
        return p.reshape(B, th // TH, TH, tw // TW, TW)
    mnx, mny = tiles(x0, big).min((2, 4)), tiles(y0, big).min((2, 4))
    mxx, mxy = tiles(x1, small).max((2, 4)), tiles(y1, small).max((2, 4))
    bx = mnx if quad else mnx & ~3
    fits = (mxx >= 0) & (mxx - bx < (BW - 3 if quad else BW)) & (mxy - mny < BH)
    return int(fits.sum()), int((~fits).sum())


def sm_count(dev):
    return torch.cuda.get_device_properties(dev).multi_processor_count


# ------------------------------------------------------------------------------------------- input builders ---
def smooth_flow(rng, B, H, W, amp=3.0):
    """Network-like flow: per item a random affine field plus a few sines (smooth, so taps of a tile fit the box)."""
    ys, xs = np.meshgrid(np.linspace(-1, 1, H), np.linspace(-1, 1, W), indexing="ij")
    out = np.empty((B, 2, H, W), F32)
    for b in range(B):
        a = rng.standard_normal(8)
        out[b, 0] = amp * (a[0] + a[1] * xs + a[2] * ys + 0.5 * np.sin(3 * xs + a[3]))
        out[b, 1] = amp * (a[4] + a[5] * xs + a[6] * ys + 0.5 * np.cos(2 * ys + a[7]))
    return out


def make_flow(kind, rng, B, H, W):
    if kind == "noise":
        return (5.0 * rng.standard_normal((B, 2, H, W))).astype(F32)
    f = smooth_flow(rng, B, H, W)
    if kind == "jump":     # a moving object: tiles on its border see taps more than a box apart
        f[:, :, H // 4: 3 * H // 4, W // 4: 3 * W // 4] += F32(37.0) * np.array([1, -1], F32)[:, None, None]
    elif kind == "converge":   # every pixel samples the same point: many terms per grad_img cell
        ys, xs = np.meshgrid(np.arange(H, dtype=F32), np.arange(W, dtype=F32), indexing="ij")
        f = np.stack([xs - F32(0.37 * (W - 1)), ys - F32(0.61 * (H - 1))])[None].repeat(B, 0).astype(F32)
    return f.astype(F32)


EDGE_KINDS = ("integer", "last", "zero", "span", "reflected", "far", "nan", "+inf", "-inf", "random")


def edge_targets(kind, rng, n, size):
    """Pre-reflection positions of one kind (float64), see ``edge_flow``."""
    span = max(size - 1, 1)
    if kind == "integer":
        return rng.integers(0, size, n).astype(np.float64)
    if kind == "last":
        return np.full(n, float(size - 1))
    if kind == "zero":
        return np.zeros(n)
    if kind == "span":   # after one reflection: -span (reflects onto span) and 2 * span (reflects onto 0)
        return np.where(rng.random(n) < 0.5, -float(span), 2.0 * span)
    if kind == "reflected":   # 2 to 10 spans out, both signs, on a tap or between taps
        k = rng.integers(2, 11, n)
        off = np.where(rng.random(n) < 0.5, rng.integers(0, size, n), rng.random(n) * span)
        return np.where(rng.random(n) < 0.5, -1.0, 1.0) * (k * span + off)
    return rng.random(n) * span


def search_flow(coord, target, size, sign):
    """float32 flow values whose emulated pre-reflection position equals ``target`` where some float32 within 256
    ulps of the float64 solution reaches it exactly; elsewhere the nearest one found."""
    u0 = (sign * (target * size / max(size - 1, 1) - coord)).astype(F32)
    tgt = target.astype(F32)
    best = u0.copy()
    hit = pre_position32(coord, u0, size, sign) == tgt
    up, dn = u0.copy(), u0.copy()
    for _ in range(256):
        up, dn = np.nextafter(up, F32(np.inf)), np.nextafter(dn, F32(-np.inf))
        for cand in (up, dn):
            h = (pre_position32(coord, cand, size, sign) == tgt) & ~hit
            best = np.where(h, cand, best)
            hit |= h
        if hit.all():
            break
    return best, hit


def edge_flow(rng, B, H, W, sign, finite=True):
    """A flow whose emulated positions land, per pixel and axis, on one kind of EDGE_KINDS: a tap (integer), the last
    pixel (the clamped x1 tap with weight 0), 0, the span after one reflection, 2-10 spans out, |x + u| = 1e6, NaN,
    +-inf.  Returns the flow and the fraction of targeted positions reached exactly."""
    kinds = [k for k in EDGE_KINDS if not finite or k not in ("nan", "+inf", "-inf")]
    n = B * H * W
    xs, ys = (a.reshape(-1).astype(np.float64) for a in grid32(B, H, W))
    flow = np.empty((2, n), F32)
    hits, total = 0, 0
    for axis, (coord, size, kind_idx) in enumerate(((xs, W, np.arange(n) % len(kinds)),
                                                    (ys, H, (np.arange(n) // len(kinds) + 1) % len(kinds)))):
        for k, kind in enumerate(kinds):
            sel = kind_idx == k
            m = int(sel.sum())
            if kind == "nan":
                flow[axis, sel] = np.nan
            elif kind in ("+inf", "-inf"):
                flow[axis, sel] = np.inf if kind == "+inf" else -np.inf
            elif kind == "far":
                s = np.where(rng.random(m) < 0.5, -1.0, 1.0)
                flow[axis, sel] = (sign * (s * 1.0e6 - coord[sel])).astype(F32)
            else:
                f, hit = search_flow(coord[sel], edge_targets(kind, rng, m, size), size, sign)
                flow[axis, sel] = f
                if kind != "random":
                    hits += int(hit.sum())
                    total += m
    flow = flow.reshape(2, B, H, W).transpose(1, 0, 2, 3)
    return np.ascontiguousarray(flow), hits / max(total, 1)


# ===================================================================================================== CPU ===
def test_position_emulation_reproduces_the_explicit_oracle_and_the_golden_warp(golden):
    """The float32 position emulation + float64 bilinear sums reproduces oracle.explicit.warp (the restatement of the
    reference) and the reference-generated golden outputs within the forward bound."""
    from oracle import explicit
    g = golden("warp")
    img, flow = g["img"], g["flow"]
    for sign, key in ((-1.0, "forward"), (1.0, "backward")):
        pos = exact_pos(flow[:, 0], flow[:, 1], sign)
        ref, bound = forward_ref(torch.from_numpy(img), pos)
        check(torch.from_numpy(explicit.warp(img, flow, sign)), ref, bound, f"explicit.warp sign={sign}")
        check(torch.from_numpy(g[key]), ref, bound, f"golden {key}")
    pos = exact_pos(np.zeros_like(flow[:, 0]), np.zeros_like(flow[:, 1]), -1.0)
    ref, bound = forward_ref(torch.from_numpy(img), pos)
    check(torch.from_numpy(g["zero_flow_forward"]), ref, bound, "golden zero flow")
    # the x0.5 down-sampled flow of the step fixture: float64 sums with fp32 lambdas within 4u sum |lambda p|
    step_flow = g["step/flow"]
    half, err = half_flow64(step_flow, *g["step/flow_half"].shape[2:])
    assert (np.abs(g["step/flow_half"] - half) <= err).all()
    up, uerr = upflow8_64(g["up8/flow_lr"], *g["up8/flow_final"].shape[2:], *(int(p) for p in g["up8/pad"]))
    assert (np.abs(g["up8/flow_final"] - up) <= uerr).all()


def test_fmax_clip_rule_on_non_finite_positions():
    """fmaxf(NaN, 0) == 0: NaN and +-inf positions land on 0 after reflect + clip (np.maximum would keep the NaN)."""
    v = np.array([np.nan, np.inf, -np.inf, 1e30, -0.0, 5.0], F32)
    assert reflect_clip32(v, 7).tolist() == [0.0, 0.0, 0.0, reflect_clip32(np.array([1e30], F32), 7)[0], 0.0, 5.0]
    # 1e30 / 6 floors to a value beyond INT_MAX: (int) saturates to INT_MAX, an odd flip count
    a = F32(1e30)
    assert reflect_clip32(np.array([a]), 7)[0] == F32(6) - np.fmod(a, F32(6))


@pytest.mark.parametrize("sign", [-1.0, 1.0])
@pytest.mark.parametrize("shape,kind", [((2, 3, 18, 22), "noise"), ((2, 4, 23, 31), "smooth"), ((1, 2, 1, 17), "noise"),
                                        ((1, 2, 13, 1), "smooth")])
def test_flow_gradient_reference_matches_cpu_autograd(sign, shape, kind):
    """Away from tap boundaries the float64 flow gradient (gix, giy with source_index_set_grad's multiplier) agrees
    with CPU autograd through ref_port.warp to 1e-6 of the largest gradient; grad_img likewise everywhere."""
    from oracle import ref_port
    B, C, H, W = shape
    rng = np.random.default_rng(sum(shape))
    img = rng.standard_normal(shape).astype(F32)
    gout = rng.standard_normal(shape).astype(F32)
    flow = make_flow(kind, rng, B, H, W)
    flow[0, :, 0, 0] = [-3.3 * W, 2.6 * H]     # several reflections
    ri, rf = torch.from_numpy(img).requires_grad_(), torch.from_numpy(flow).requires_grad_()
    ref_port.warp(ri, rf, "forward" if sign < 0 else "backward").backward(torch.from_numpy(gout))
    pos = exact_pos(flow[:, 0], flow[:, 1], sign)
    gi, _, lo, hi, _, _ = backward_ref(torch.from_numpy(img), torch.from_numpy(gout), pos, sign)
    assert torch.equal(lo, hi)
    scale = float(rf.grad.abs().max())
    frac = lambda a: np.abs(a - np.round(a))   # noqa: E731
    away = ((frac(pos.ix) > 1e-3) | (W == 1)) & ((frac(pos.iy) > 1e-3) | (H == 1))   # a one-pixel axis sits on 0
    err = (lo - rf.grad.double()).abs().numpy()
    assert away.mean() > 0.9
    assert (err * away[:, None]).max() <= 1e-6 * scale
    assert (gi - ri.grad.double()).abs().max() <= 1e-6 * float(ri.grad.abs().max())


def test_restated_tile_and_image_predicates():
    """route / in_tiles / tile_mix against hand-computed cases."""
    sms = 148
    assert route(2, 8, 90, 120, True, sms) == 1                    # 4-byte pitch multiple of 16: 4-D map
    assert route(2, 7, 90, 120, True, sms) is None                 # fewer than 8 channels: direct
    assert route(2, 16, 90, 120, False, sms) is None               # misaligned base: direct
    assert route(2, 16, 90, 120, True, sms, path_direct=True) is None
    # quad: 5 x 9 tiles x 2 groups = 90 CTAs per item; 3 * 148 = 444 -> 5 items are enough, 4 are not
    assert route(5, 128, 130, 149, True, sms) == 2 and route(4, 128, 130, 149, True, sms) is None
    assert route(4, 128, 130, 149, True, sms, quad_env="1") == 2 and route(5, 128, 130, 149, True, sms, quad_env="0") is None
    assert route(1, 32, 48, 41, True, sms, "1") == 1 and route(1, 32, 49, 41, True, sms, "1") == 4
    assert route(1, 48, 48, 41, True, sms, "1") is None            # C % 32 != 0
    assert route(1, 32, 48, 13, True, sms, "1") is None and route(1, 32, 22, 42, True, sms, "1") is None
    # image in the tiles: 4 x 6 tiles x 2 groups = 48 codes CTAs per item, more than 6 * 148 = 888 from 19 items
    assert in_tiles(192, 256, 19, 128, 96, 128, sms) and not in_tiles(192, 256, 18, 128, 96, 128, sms)
    assert not in_tiles(193, 256, 19, 128, 96, 128, sms) and not in_tiles(192, 256, 19, 128, 96, 128, sms, True)
    # tile box: identity taps fit; a 47-column spread fits the 48-wide box from a 4-aligned start, 45 columns in quad
    ix = np.tile(np.arange(64, dtype=F32), (1, 32, 1))
    iy = np.tile(np.arange(32, dtype=F32)[:, None], (1, 1, 64))
    assert tile_mix(ix, iy, False) == (4, 0)
    wide = np.full_like(ix, 10.0)
    wide[0, 0, 0], wide[0, 0, 31] = 4.0, 50.0      # taps 4 .. 51: 51 - 4 = 47 < 48
    assert tile_mix(wide, iy, False) == (4, 0)
    wide[0, 0, 0] = 3.0                            # box start 0 after the 4-float alignment: 51 - 0 >= 48
    assert tile_mix(wide, iy, False) == (3, 1)
    wide[0, 0, 31] = 46.0                          # quad keeps the start at 3: taps 3 .. 47, 44 < 45
    assert tile_mix(wide, iy, True) == (4, 0)
    wide[0, 0, 31] = 47.0                          # 48 - 3 = 45: does not fit
    assert tile_mix(wide, iy, True) == (3, 1)
    tall = np.full_like(iy, 2.0)
    tall[0, 0, 5] = 24.0                           # rows 2 .. 25: 23 < 24
    assert tile_mix(ix, tall, False) == (4, 0)
    tall[0, 0, 5] = 25.0                           # rows 2 .. 26
    assert tile_mix(ix, tall, False) == (3, 1)


def test_edge_flow_search_reaches_its_targets():
    """The edge flows land exactly on their targets for most positions (else the edge rows would test nothing).  The
    last pixel, 0 and the reflected span are always reached; about 40 % of the integers are not reachable through the
    fp32 position chain and stay within an ulp or two."""
    rng = np.random.default_rng(3)
    for sign in (-1.0, 1.0):
        flow, frac = edge_flow(rng, 2, 27, 45, sign, finite=False)
        assert frac > 0.75, frac
        ix, iy, mx, my = positions32(flow[:, 0], flow[:, 1], sign)
        assert (ix == 44).any() and (ix == 0).any() and (mx == 0).any() and (my == 0).any()
        assert np.isfinite(ix).all() and np.isfinite(iy).all()


# ===================================================================================================== GPU ===
def last_kernel():
    from cistaflow_b200 import _lib
    return _lib.load().cf_last_kernel().decode()


def dev_t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def input_view(a, dev, misalign):
    """a copy of ``a`` on the device, one float off a 16-byte boundary when ``misalign``."""
    if not misalign:
        return dev_t(a, dev)
    buf = torch.zeros(a.size + 8, device=dev)
    v = buf[1:1 + a.size].view(a.shape)
    v.copy_(torch.from_numpy(np.ascontiguousarray(a)))
    assert v.data_ptr() % 16 == 4
    return v


def pos_for(flow, H, W, sign):
    """Positions of a [B, 2, fH, fW] flow for an [H, W] output: exact at the same resolution, else the fused x0.5
    down-sampling with its delta."""
    if flow.shape[2:] == (H, W):
        return exact_pos(flow[:, 0], flow[:, 1], sign)
    f, e = half_flow64(flow, H, W)
    return approx_pos_with_pre(f[:, 0], f[:, 1], e[:, 0], e[:, 1], sign)


REPORT = {}


def report(parity_report, family, worst, **kw):
    REPORT[family] = max(REPORT.get(family, 0.0), worst)
    parity_report.add(f"warp_branches/{family}", worst_err_over_bound=worst, **kw)


# ------------------------------------------------------------------------------------- cf_warp forward table ---
WRow = namedtuple("WRow", "branch B C H W fH fW flow kernel P misalign quad_env mix")
_W = lambda branch, B, C, H, W, flow="noise", kernel="warp_gather_kernel", P=None, half=None, misalign=False, quad_env=None, mix=None: \
    WRow(branch, B, C, H, W, *(half or (H, W)), flow, kernel, P, misalign, quad_env, mix)   # noqa: E731
T = "warp_tma_kernel"
WARP_ROWS = [
    _W("direct CPT1, C=1", 2, 1, 20, 36),
    _W("direct CPT1, C=3", 2, 3, 33, 47),
    _W("direct CPT4, C=4", 2, 4, 20, 36),
    _W("direct CPT4, tail batch C=5", 2, 5, 21, 37),
    _W("direct CPT4, tail batch C=7", 2, 7, 17, 29),
    _W("direct CPT8, two groups + partial, C=33, 4-byte aligned", 2, 33, 18, 40, misalign=True),
    _W("direct CPT8, partial second group, C=40, 4-byte aligned", 2, 40, 19, 24, flow="smooth", misalign=True),
    _W("direct, H=1", 2, 3, 1, 50),
    _W("direct, W=1", 2, 5, 40, 1),
    _W("direct CPT8, plane smaller than one tile", 2, 9, 5, 7),
    _W("TMA 4-D, C=8, all tiles fit", 2, 8, 48, 64, "smooth", T, 1, mix="ring"),
    _W("TMA 4-D, C=13 (partial chunk), mixed tiles", 2, 13, 64, 96, "jump", T, 1, mix="both"),
    _W("TMA 4-D, C=64, noise: mostly fallback", 2, 64, 40, 64, "noise", T, 1, mix="fallback"),
    _W("TMA 4-D, C=70 (second group of 6), mixed tiles, B=3", 3, 70, 48, 72, "jump", T, 1, mix="both"),
    _W("TMA 4-D, C=128, all tiles fit", 2, 128, 40, 72, "smooth", T, 1, mix="ring"),
    _W("quad P=1 (H%4=0), W%4=1, C=32, forced", 3, 32, 48, 41, "jump", T, 1, quad_env="1", mix="both"),
    _W("quad P=2 (H%4=2), W%4=2, C=96, forced", 2, 96, 50, 42, "jump", T, 2, quad_env="1", mix="both"),
    _W("quad P=4 (H odd), W%4=3, C=128, forced", 2, 128, 49, 43, "jump", T, 4, quad_env="1", mix="both"),
    _W("quad P=4, above one wave at the default threshold", 0, 128, 65, 130, "jump", T, 4, mix="both"),
    _W("quad P=2, above one wave at the default threshold", 0, 96, 66, 129, "smooth", T, 2),
    _W("quad refused by CF_WARP_QUAD=0", 3, 32, 48, 41, "smooth", quad_env="0"),
    _W("quad refused: W < 16", 2, 32, 48, 13, "smooth", quad_env="1"),
    _W("quad refused: H < 24", 2, 32, 22, 42, "smooth", quad_env="1"),
    _W("x0.5 flow, direct CPT1", 2, 2, 20, 36, "smooth", half=(40, 72)),
    _W("x0.5 flow, direct CPT4", 2, 5, 20, 36, "noise", half=(40, 72)),
    _W("x0.5 flow, TMA 4-D", 2, 16, 32, 48, "smooth", T, 1, half=(64, 96), mix="ring"),
    _W("x0.5 flow, quad P=2", 2, 32, 30, 45, "smooth", T, 2, half=(60, 90), quad_env="1"),
    _W("x0.5 flow, odd flow size, direct", 2, 3, 20, 36, "smooth", half=(41, 73)),
    _W("x0.5 flow, odd flow size, TMA 4-D", 2, 16, 32, 48, "jump", T, 1, half=(65, 97), mix="both"),
    _W("x0.5 flow, H=1 (fH=2)", 2, 3, 1, 30, "smooth", half=(2, 60)),
    _W("x0.5 flow, H=1 (fH=3)", 2, 3, 1, 30, "noise", half=(3, 61)),
]


def _quad_batch(row, sms):
    """Items enough for 3 * SMs CTAs of the quad path (the default threshold)."""
    per = cdiv(row.W, TW) * cdiv(row.H, TH) * cdiv(row.C, CH_PER_CTA)
    return cdiv(3 * sms, per)


@gpu
@pytest.mark.parametrize("sign", [-1.0, 1.0], ids=["fwd", "bwd"])
@pytest.mark.parametrize("row", WARP_ROWS, ids=[r.branch for r in WARP_ROWS])
def test_warp_forward_branch(cuda_device, parity_report, monkeypatch, row, sign):
    import cistaflow_b200 as cf
    sms = sm_count(cuda_device)
    B = row.B or _quad_batch(row, sms)
    if row.quad_env is None:
        monkeypatch.delenv("CF_WARP_QUAD", raising=False)
    else:
        monkeypatch.setenv("CF_WARP_QUAD", row.quad_env)
    P = route(B, row.C, row.H, row.W, not row.misalign, sms, row.quad_env)
    assert P == row.P, f"{row.branch}: the host predicates pick P={P}"
    rng = np.random.default_rng(row.C * 1000 + row.H * 7 + row.W + (sign > 0))
    img = rng.standard_normal((B, row.C, row.H, row.W)).astype(F32)
    flow = make_flow(row.flow, rng, B, row.fH, row.fW)
    dimg = input_view(img, cuda_device, row.misalign)
    buf, (out,) = guarded([img.shape], cuda_device)
    cf.warp(dimg, dev_t(flow, cuda_device), sign, out=out)
    assert last_kernel() == row.kernel, f"{row.branch}: ran {last_kernel()}"
    torch.cuda.synchronize()
    assert_written_and_guarded(buf, [out], row.branch)
    pos = pos_for(flow, row.H, row.W, sign)
    if row.mix:
        ring, fallback = tile_mix(pos.ix, pos.iy, row.W % 4 != 0)
        want = {"ring": fallback == 0 and ring > 0, "both": ring > 0 and fallback > 0, "fallback": fallback > ring}[row.mix]
        assert want, f"{row.branch}: {ring} ring tiles, {fallback} fallback tiles"
    ref, bound = forward_ref(torch.from_numpy(img).to(cuda_device), pos)
    group = CH_PER_CTA if row.kernel == T else None
    worst = check(out, ref, bound, row.branch, group)
    family = "TMA quad" if row.kernel == T and row.W % 4 else ("TMA" if row.kernel == T else "direct")
    report(parity_report, family, worst, branch=row.branch, sign=sign, B=B)


# --------------------------------------------------------------------------------------- frame step table ---
FRow = namedtuple("FRow", "branch B Ci Cz H W flow kernel in_tiles misalign quad_env")
FRAME_ROWS = [
    FRow("TMA, separate image CTAs (few CTAs), Ci=1", 2, 1, 16, 64, 96, "smooth", T, False, False, None),
    FRow("TMA, separate image CTAs (odd image), Ci=3", 2, 3, 16, 65, 97, "jump", T, False, False, None),
    FRow("TMA, image in the codes tiles, Ci=1", 0, 1, 128, 192, 256, "jump", T, True, False, None),
    FRow("TMA, image in the codes tiles, Ci=3", 0, 3, 64, 192, 256, "smooth", T, True, False, None),
    FRow("quad, separate image CTAs, Ci=5", 2, 5, 32, 60, 90, "jump", T, False, False, "1"),
    FRow("direct frame kernel (misaligned codes), Ci=1", 2, 1, 16, 64, 96, "smooth", "warp_frame_and_codes_kernel", False, True, None),
    FRow("direct frame kernel, two image groups, Ci=5", 2, 5, 16, 63, 95, "noise", "warp_frame_and_codes_kernel", False, True, None),
    FRow("direct frame kernel, Cz < 8", 2, 3, 5, 40, 56, "jump", "warp_frame_and_codes_kernel", False, False, None),
]


def _tiles_batch(Cz, Hz, Wz, sms):
    per = cdiv(Wz, TW) * cdiv(Hz, TH) * cdiv(Cz, CH_PER_CTA)
    return 6 * sms // per + 1


def frame_inputs(rng, B, Ci, Cz, H, W, flow_kind):
    img = rng.standard_normal((B, Ci, H, W)).astype(F32)
    codes = rng.standard_normal((B, Cz, H // 2, W // 2)).astype(F32)
    codes[np.abs(codes) < 0.8] = 0      # sparse, like the codes: exact zeros demand exact zeros
    return img, codes, make_flow(flow_kind, rng, B, H, W)


def check_frame(img, codes, flow, wi, wz, sign, what, gate_open=True):
    """(worst image ratio, worst codes ratio) against float64."""
    dev = wi.device
    H, W = img.shape[2:]
    pi = exact_pos(flow[:, 0], flow[:, 1], sign)
    ri, bi = forward_ref(torch.from_numpy(img).to(dev), pi)
    pz = pos_for(flow, H // 2, W // 2, sign)
    rz, bz = forward_ref(torch.from_numpy(codes).to(dev), pz)
    return check(wi, ri, bi, what + ", image", 4), check(wz, rz, bz, what + ", codes", CH_PER_CTA), pz


@gpu
@pytest.mark.parametrize("mode", ["forward", "backward"])
@pytest.mark.parametrize("row", FRAME_ROWS, ids=[r.branch for r in FRAME_ROWS])
def test_frame_step_branch(cuda_device, parity_report, monkeypatch, row, mode):
    import cistaflow_b200 as cf
    sms = sm_count(cuda_device)
    Hz, Wz = row.H // 2, row.W // 2
    B = row.B or _tiles_batch(row.Cz, Hz, Wz, sms)
    if row.quad_env:
        monkeypatch.setenv("CF_WARP_QUAD", row.quad_env)
    else:
        monkeypatch.delenv("CF_WARP_QUAD", raising=False)
    P = route(B, row.Cz, Hz, Wz, not row.misalign, sms, row.quad_env)
    assert (P is not None) == (row.kernel == T), f"{row.branch}: the host predicates pick P={P}"
    assert in_tiles(row.H, row.W, B, row.Cz, Hz, Wz, sms) == row.in_tiles
    sign = -1.0 if mode == "forward" else 1.0
    rng = np.random.default_rng(row.H * row.W + row.Ci + row.Cz)
    img, codes, flow = frame_inputs(rng, B, row.Ci, row.Cz, row.H, row.W, row.flow)
    buf, (wi, wz) = guarded([img.shape, codes.shape], cuda_device)
    cf.warp_frame_and_codes(dev_t(img, cuda_device), input_view(codes, cuda_device, row.misalign), dev_t(flow, cuda_device),
                            mode, out=(wi, wz))
    assert last_kernel() == row.kernel
    torch.cuda.synchronize()
    assert_written_and_guarded(buf, [wi, wz], row.branch)
    w_i, w_z, _ = check_frame(img, codes, flow, wi, wz, sign, row.branch)
    report(parity_report, "frame step", max(w_i, w_z), branch=row.branch, mode=mode, B=B)


GATE_ROWS = [("TMA 4-D", 64, 96, False, None), ("TMA quad", 60, 90, False, "1"),
             ("direct frame kernel", 64, 96, True, None)]


@gpu
@pytest.mark.parametrize("kernel,H,W,misalign,quad_env", GATE_ROWS, ids=[r[0] for r in GATE_ROWS])
def test_zero_flow_gate_on_each_kernel(cuda_device, parity_report, monkeypatch, kernel, H, W, misalign, quad_env):
    """Gate closed (an all-zero flow, -0.0 included): a bitwise copy.  Gate open: the warp, held to the bound."""
    import cistaflow_b200 as cf
    if quad_env:
        monkeypatch.setenv("CF_WARP_QUAD", quad_env)
    else:
        monkeypatch.delenv("CF_WARP_QUAD", raising=False)
    rng = np.random.default_rng(H + W)
    img, codes, flow = frame_inputs(rng, 2, 1, 32, H, W, "smooth")
    name = "warp_frame_and_codes_kernel" if misalign else T
    zero = np.zeros_like(flow)
    zero[1, 0, 3, 4] = -0.0
    for f, closed in ((zero, True), (flow, False)):
        df = dev_t(f, cuda_device)
        gate = cf.flow_any(df)
        buf, (wi, wz) = guarded([img.shape, codes.shape], cuda_device)
        cf.warp_frame_and_codes(dev_t(img, cuda_device), input_view(codes, cuda_device, misalign), df, "forward",
                                out=(wi, wz), gate=gate)
        assert last_kernel() == name
        torch.cuda.synchronize()
        assert_written_and_guarded(buf, [wi, wz], f"gate {kernel}")
        if closed:
            assert torch.equal(wi.cpu(), torch.from_numpy(img)) and torch.equal(wz.cpu(), torch.from_numpy(codes))
        else:
            w_i, w_z, _ = check_frame(img, codes, f, wi, wz, -1.0, f"gate open, {kernel}")
            report(parity_report, "frame step", max(w_i, w_z), branch=f"gate open, {kernel}")


# ------------------------------------------------------------------------------------------------ upflow8 ---
URow = namedtuple("URow", "branch B Ci Cz lh lw pad_h pad_w kernel in_tiles misalign quad_env")
UPFLOW_ROWS = [
    URow("TMA, separate image CTAs, no padding", 2, 1, 16, 8, 12, 0, 0, T, False, False, None),
    URow("TMA, separate image CTAs, padded", 2, 3, 16, 8, 12, 8, 8, T, False, False, None),
    URow("TMA, image in the tiles, no padding", 0, 1, 64, 24, 32, 0, 0, T, True, False, None),
    URow("TMA, image in the tiles, padded", 0, 1, 64, 24, 32, 8, 8, T, True, False, None),
    URow("quad, padding on the columns only", 2, 1, 32, 8, 11, 0, 2, T, False, False, "1"),   # unpadded: W/2 % 4 == 0
    URow("quad, padded", 2, 1, 32, 8, 12, 4, 6, T, False, False, "1"),
    URow("direct frame kernel, no padding", 2, 1, 16, 8, 12, 0, 0, "warp_frame_and_codes_kernel", False, True, None),
    URow("direct frame kernel, padded", 2, 3, 16, 8, 12, 5, 3, "warp_frame_and_codes_kernel", False, True, None),
]


def upflow8_call(img, codes, lr, outs, B, Ci, Cz, H, W, lh, lw, pad_h, pad_w, sign, dev):
    from cistaflow_b200 import _lib
    lib = _lib.load()
    wi, wz, fo = outs
    rc = lib.cf_warp_frame_and_codes_upflow8(img.data_ptr(), codes.data_ptr(), lr.data_ptr(), wi.data_ptr(), wz.data_ptr(),
                                             _lib.ptr(fo), B, Ci, Cz, H, W, lh, lw, pad_h, pad_w, sign, _lib.stream_ptr(dev))
    _lib.check(rc, "cf_warp_frame_and_codes_upflow8")


@gpu
@pytest.mark.parametrize("return_flow", [True, False], ids=["flow_out", "no_flow_out"])
@pytest.mark.parametrize("row", UPFLOW_ROWS, ids=[r.branch for r in UPFLOW_ROWS])
def test_upflow8_branch(cuda_device, parity_report, monkeypatch, row, return_flow):
    """The fused upflow8 + unpad + frame step through the C ABI: image, codes and flow_out (fully written, once)
    against float64, and flow_out = null."""
    sms = sm_count(cuda_device)
    H, W = 8 * row.lh - row.pad_h, 8 * row.lw - row.pad_w
    Hz, Wz = H // 2, W // 2
    B = row.B or _tiles_batch(row.Cz, Hz, Wz, sms)
    if row.quad_env:
        monkeypatch.setenv("CF_WARP_QUAD", row.quad_env)
    else:
        monkeypatch.delenv("CF_WARP_QUAD", raising=False)
    assert (route(B, row.Cz, Hz, Wz, not row.misalign, sms, row.quad_env) is not None) == (row.kernel == T)
    assert in_tiles(H, W, B, row.Cz, Hz, Wz, sms) == row.in_tiles
    rng = np.random.default_rng(H * W + row.pad_h)
    img, codes, _ = frame_inputs(rng, B, row.Ci, row.Cz, H, W, "smooth")
    lr = (2.0 * rng.standard_normal((B, 2, row.lh, row.lw))).astype(F32)
    shapes = [img.shape, codes.shape] + ([(B, 2, H, W)] if return_flow else [])
    buf, views = guarded(shapes, cuda_device)
    outs = views + ([] if return_flow else [None])
    upflow8_call(dev_t(img, cuda_device), input_view(codes, cuda_device, row.misalign), dev_t(lr, cuda_device), outs,
                 B, row.Ci, row.Cz, H, W, row.lh, row.lw, row.pad_h, row.pad_w, -1.0, cuda_device)
    assert last_kernel() == row.kernel
    torch.cuda.synchronize()
    assert_written_and_guarded(buf, views, row.branch)
    up, uerr = upflow8_64(lr, H, W, row.pad_h, row.pad_w)
    worst = 0.0
    if return_flow:
        worst = check(views[2], torch.from_numpy(up).to(cuda_device), torch.from_numpy(uerr).to(cuda_device),
                      f"{row.branch}, flow_out")
    pi = approx_pos_with_pre(up[:, 0], up[:, 1], uerr[:, 0], uerr[:, 1], -1.0)
    ri, bi = forward_ref(torch.from_numpy(img).to(cuda_device), pi)
    worst = max(worst, check(views[0], ri, bi, f"{row.branch}, image", 4))
    hf, he = resample64(up, half_lambdas(Hz, H), half_lambdas(Wz, W), ferr=uerr)
    pz = approx_pos_with_pre(hf[:, 0], hf[:, 1], he[:, 0], he[:, 1], -1.0)
    rz, bz = forward_ref(torch.from_numpy(codes).to(cuda_device), pz)
    worst = max(worst, check(views[1], rz, bz, f"{row.branch}, codes", CH_PER_CTA))
    report(parity_report, "upflow8", worst, branch=row.branch, return_flow=return_flow, B=B)


# ------------------------------------------------------------------------------------------- static knobs ---
_KNOB_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
import torch
import cistaflow_b200 as cf
from cistaflow_b200 import _lib
img, codes, flow = torch.load(sys.argv[2])
dev = torch.device("cuda", 0)
wi, wz = cf.warp_frame_and_codes(img.to(dev), codes.to(dev), flow.to(dev), "forward")
wc = cf.warp(codes.to(dev), flow.to(dev), -1.0)
name = _lib.load().cf_last_kernel().decode()
torch.save((wi.cpu(), wz.cpu(), wc.cpu(), name), sys.argv[3])
"""


@gpu
def test_static_knobs_in_a_subprocess(cuda_device, parity_report, tmp_path):
    """CF_WARP_IMAGE_CTAS=1 (separate image CTAs) reproduces the in-tiles outputs bit for bit: the same block code.
    CF_WARP_PATH=direct (the plain gathers) is within the bound; whether it is also bitwise is reported."""
    import cistaflow_b200 as cf
    sms = sm_count(cuda_device)
    Cz, H, W = 64, 192, 256
    B = _tiles_batch(Cz, H // 2, W // 2, sms)
    rng = np.random.default_rng(99)
    img, codes, flow = frame_inputs(rng, B, 1, Cz, H, W, "jump")
    inp = tmp_path / "in.pt"
    torch.save(tuple(torch.from_numpy(a) for a in (img, codes, flow)), inp)
    wi, wz = cf.warp_frame_and_codes(dev_t(img, cuda_device), dev_t(codes, cuda_device), dev_t(flow, cuda_device), "forward")
    assert last_kernel() == T and in_tiles(H, W, B, Cz, H // 2, W // 2, sms)
    wc = cf.warp(dev_t(codes, cuda_device), dev_t(flow, cuda_device), -1.0)
    outs = {}
    flags = ["-s"] if sys.flags.no_user_site else []
    for knob in ("CF_WARP_IMAGE_CTAS=1", "CF_WARP_PATH=direct"):
        env = {k: v for k, v in os.environ.items() if k not in ("CF_WARP_IMAGE_CTAS", "CF_WARP_PATH", "CF_WARP_QUAD")}
        k, v = knob.split("=")
        env[k] = v
        path = tmp_path / f"{k}.pt"
        res = subprocess.run([sys.executable, *flags, "-c", _KNOB_SCRIPT, ROOT, str(inp), str(path)], env=env, cwd=ROOT,
                             capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, f"{knob}:\n{res.stdout}\n{res.stderr}"
        outs[k] = torch.load(path)
    si, sz, sc, name = outs["CF_WARP_IMAGE_CTAS"]
    assert name == T
    assert torch.equal(si.view(torch.int32), wi.cpu().view(torch.int32)), "separate image CTAs differ from the in-tiles image"
    assert torch.equal(sz.view(torch.int32), wz.cpu().view(torch.int32))
    di, dz, dc, name = outs["CF_WARP_PATH"]
    assert name == "warp_gather_kernel"
    w_i, w_z, _ = check_frame(img, codes, flow, di.to(cuda_device), dz.to(cuda_device), -1.0, "CF_WARP_PATH=direct")
    bitwise = bool(torch.equal(di, wi.cpu()) and torch.equal(dz, wz.cpu()) and torch.equal(dc, wc.cpu()))
    report(parity_report, "direct", max(w_i, w_z), branch="CF_WARP_PATH=direct", bitwise_equal_to_staged=bitwise)


# ---------------------------------------------------------------------------------------- edge positions ---
EDGE_ROWS = [("direct", 2, 3, 27, 45, "warp_gather_kernel", None), ("TMA 4-D", 2, 16, 40, 64, T, None),
             ("TMA quad", 2, 32, 48, 45, T, "1")]


@gpu
@pytest.mark.parametrize("finite", [True, False], ids=["finite", "nan_inf"])
@pytest.mark.parametrize("sign", [-1.0, 1.0], ids=["fwd", "bwd"])
@pytest.mark.parametrize("family,B,C,H,W,kernel,quad_env", EDGE_ROWS, ids=[r[0] for r in EDGE_ROWS])
def test_edge_positions_forward(cuda_device, parity_report, monkeypatch, family, B, C, H, W, kernel, quad_env, sign, finite):
    """Positions exactly on a tap, on the last pixel, on 0, on the span after one reflection, 2-10 spans out, at
    |x + u| = 1e6 and (nan_inf) at NaN and +-inf: every element written, no guard touched, values within the bound of
    the fmax-clip rule (non-finite positions go to 0)."""
    import cistaflow_b200 as cf
    if quad_env:
        monkeypatch.setenv("CF_WARP_QUAD", quad_env)
    else:
        monkeypatch.delenv("CF_WARP_QUAD", raising=False)
    rng = np.random.default_rng(C + H + (sign > 0))
    flow, _ = edge_flow(rng, B, H, W, sign, finite)
    img = rng.standard_normal((B, C, H, W)).astype(F32)
    buf, (out,) = guarded([img.shape], cuda_device)
    cf.warp(dev_t(img, cuda_device), dev_t(flow, cuda_device), sign, out=out)
    assert last_kernel() == kernel
    torch.cuda.synchronize()
    assert_written_and_guarded(buf, [out], family)
    ref, bound = forward_ref(torch.from_numpy(img).to(cuda_device), exact_pos(flow[:, 0], flow[:, 1], sign))
    worst = check(out, ref, bound, f"edge positions, {family}", CH_PER_CTA)
    report(parity_report, "TMA quad" if quad_env else ("TMA" if kernel == T else "direct"), worst,
           branch=f"edge positions ({'finite' if finite else 'NaN/inf'})", sign=sign)
    # the frame step's image part (its own block code) on the same flow
    if family == "TMA 4-D":
        codes = rng.standard_normal((B, 8, H // 2, W // 2)).astype(F32)
        bufi, (wi, wz) = guarded([(B, 1, H, W), codes.shape], cuda_device)
        cf.warp_frame_and_codes(dev_t(img[:, :1], cuda_device), dev_t(codes, cuda_device), dev_t(flow, cuda_device),
                                "forward" if sign < 0 else "backward", out=(wi, wz))
        torch.cuda.synchronize()
        assert_written_and_guarded(bufi, [wi, wz], "edge positions, frame step")
        check(wi, ref[:, :1], bound[:, :1], "edge positions, frame-step image")


# ------------------------------------------------------------------------------------------ adjoint sweep ---
ARow = namedtuple("ARow", "case B C H W fH fW flow")
ADJ_ROWS = [
    ARow("C=1, noise", 2, 1, 24, 36, 24, 36, "noise"),
    ARow("C=5, smooth", 2, 5, 23, 31, 23, 31, "smooth"),
    ARow("C=32, noise", 2, 32, 20, 28, 20, 28, "noise"),
    ARow("C=33, converge", 2, 33, 18, 26, 18, 26, "converge"),
    ARow("C=70, smooth", 2, 70, 17, 22, 17, 22, "smooth"),
    ARow("C=5, edge positions", 2, 5, 27, 45, 27, 45, "edge"),
    ARow("C=33, edge positions", 3, 33, 19, 23, 19, 23, "edge"),
    ARow("C=1, H=1", 2, 1, 1, 40, 1, 40, "noise"),
    ARow("half, C=5, smooth", 2, 5, 18, 24, 36, 48, "smooth"),
    ARow("half, C=33, noise", 2, 33, 18, 24, 36, 48, "noise"),
    ARow("half, C=5, odd flow", 2, 5, 18, 24, 37, 49, "smooth"),
    ARow("half, C=70, odd flow, jump", 2, 70, 15, 21, 31, 43, "jump"),
    ARow("half, C=3, H=1 (fH=3)", 2, 3, 1, 30, 3, 61, "smooth"),
    ARow("half, C=1, converge", 2, 1, 16, 20, 32, 40, "converge"),
]


def adjoint_inputs(row, sign):
    rng = np.random.default_rng(row.C * 100 + row.H + row.fW)
    img = rng.standard_normal((row.B, row.C, row.H, row.W)).astype(F32)
    gout = rng.standard_normal((row.B, row.C, row.H, row.W)).astype(F32)
    if row.flow == "edge":
        flow, _ = edge_flow(rng, row.B, row.H, row.W, sign, finite=True)
    else:
        flow = make_flow(row.flow, rng, row.B, row.fH, row.fW)
    return img, gout, flow


def adjoint_call(kind, img, gout, flow, want_img, want_flow, sign, dev, pass_img=True):
    """cf_warp_backward / cf_warp_backward_det into guarded outputs; a null pointer for a gradient not requested."""
    from cistaflow_b200 import _lib
    lib = _lib.load()
    B, C, H, W = img.shape
    fH, fW = flow.shape[2:]
    shapes = ([tuple(img.shape)] if want_img else []) + ([tuple(flow.shape)] if want_flow else [])
    buf, views = guarded(shapes, dev)
    gi = views[0] if want_img else None
    gf = views[-1] if want_flow else None
    ip = img.data_ptr() if pass_img else None
    s = _lib.stream_ptr(dev)
    if kind == "atomic":
        rc = lib.cf_warp_backward(gout.data_ptr(), ip, flow.data_ptr(), _lib.ptr(gi), _lib.ptr(gf), B, C, H, W, fH, fW, sign, s)
        _lib.check(rc, "cf_warp_backward")
    else:
        n = lib.cf_warp_backward_det_workspace_bytes(B, C, H, W, fH, fW)
        ws = torch.empty(n, dtype=torch.uint8, device=dev)
        rc = lib.cf_warp_backward_det(gout.data_ptr(), ip, flow.data_ptr(), _lib.ptr(gi), _lib.ptr(gf), B, C, H, W, fH, fW,
                                      sign, ws.data_ptr(), n, s)
        _lib.check(rc, "cf_warp_backward_det")
    name = last_kernel()
    torch.cuda.synchronize()
    assert_written_and_guarded(buf, views, f"{kind} adjoint")
    return gi, gf, name


ADJ_KERNELS = {("atomic", False): "warp_backward_kernel", ("atomic", True): "warp_backward_kernel",
               ("det", False): "warp_backward_det_gather_kernel", ("det", True): "warp_backward_det_flow_half_kernel"}


@gpu
@pytest.mark.parametrize("sign", [-1.0, 1.0], ids=["fwd", "bwd"])
@pytest.mark.parametrize("row", ADJ_ROWS, ids=[r.case for r in ADJ_ROWS])
def test_adjoint_sweep(cuda_device, parity_report, row, sign):
    """Both adjoints, each request (both gradients, grad_img only with img = null, grad_flow only), against float64;
    the atomic and the deterministic result agree within the sum of their bounds."""
    half = (row.fH, row.fW) != (row.H, row.W)
    img, gout, flow = adjoint_inputs(row, sign)
    dev = cuda_device
    di, dg, df = dev_t(img, dev), dev_t(gout, dev), dev_t(flow, dev)
    pos = pos_for(flow, row.H, row.W, sign)
    ri, bi, flo, fhi, bf, either = backward_ref(di, dg, pos, sign, (row.fH, row.fW))
    got = {}
    for kind in ("atomic", "det"):
        for want_img, want_flow in ((True, True), (True, False), (False, True)):
            gi, gf, name = adjoint_call(kind, di, dg, df, want_img, want_flow, sign, dev, pass_img=want_flow)
            if want_img and want_flow:
                assert name == ADJ_KERNELS[kind, half]
            what = f"{kind} adjoint, {row.case}, img={want_img} flow={want_flow}"
            worst = 0.0
            if want_img:
                worst = check(gi, ri, bi, what + ", grad_img", 32)
                got[kind, "img", want_flow] = gi
            if want_flow:
                worst = max(worst, check_interval(gf, flo, fhi, bf, what + ", grad_flow"))
                got[kind, "flow", want_img] = gf
            report(parity_report, f"{kind} adjoint", worst, case=row.case, sign=sign, grad_img=want_img,
                   grad_flow=want_flow, either_side_elements=either if want_flow else 0)
        assert torch.equal(got[kind, "img", True], got[kind, "img", False]) or kind == "atomic"
        assert torch.equal(got[kind, "flow", True], got[kind, "flow", False]) or kind == "atomic"
    # det against atomic: within the sum of the two bounds (each bound once per side)
    for key, ref_bound in (("img", bi), ("flow", bf)):
        a, d = got["atomic", key, True].double(), got["det", key, True].double()
        assert ((a - d).abs() <= 2 * ref_bound + 2 * (fhi - flo if key == "flow" else 0)).all(), f"det vs atomic, {key}"
    REPORT["either_side_elements"] = REPORT.get("either_side_elements", 0) + either


@gpu
@pytest.mark.parametrize("deterministic", [False, True], ids=["atomic", "det"])
def test_autograd_passes_the_same_pointers(cuda_device, parity_report, deterministic):
    """_WarpFunction.backward with the flag off and on: both gradients within the float64 bound, bitwise equal to the
    C call for the deterministic adjoint."""
    import cistaflow_b200 as cf
    row = ARow("autograd, half, C=33", 2, 33, 18, 24, 37, 49, "smooth")
    img, gout, flow = adjoint_inputs(row, -1.0)
    dev = cuda_device
    di, df = dev_t(img, dev).requires_grad_(), dev_t(flow, dev).requires_grad_()
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(deterministic)
    try:
        cf.warp(di, df, -1.0).backward(dev_t(gout, dev))
    finally:
        torch.use_deterministic_algorithms(prev)
    assert last_kernel() == ADJ_KERNELS["det" if deterministic else "atomic", True]
    pos = pos_for(flow, row.H, row.W, -1.0)
    ri, bi, flo, fhi, bf, _ = backward_ref(di.detach(), dev_t(gout, dev), pos, -1.0, (row.fH, row.fW))
    worst = max(check(di.grad, ri, bi, "autograd grad_img", 32), check_interval(df.grad, flo, fhi, bf, "autograd grad_flow"))
    report(parity_report, "det adjoint" if deterministic else "atomic adjoint", worst, case="autograd")
    if deterministic:
        gi, gf, _ = adjoint_call("det", di.detach(), dev_t(gout, dev), df.detach(), True, True, -1.0, dev)
        assert torch.equal(gi, di.grad) and torch.equal(gf, df.grad)


@gpu
def test_zz_report_worst_ratios(cuda_device, parity_report):
    """The largest err/bound per kernel family of this session, and the either-side count (reporting only)."""
    if REPORT:
        parity_report.add("warp_branches/summary", **REPORT)
        print("warp branches:", REPORT)
