"""From-scratch NumPy / C restatement of the hot path (no torch ops).

TEST INFRASTRUCTURE -- see ``oracle/__init__.py``.

``ref_port`` goes through the same library calls as the reference; this module
spells out what those calls *do*, element by element, so that the CUDA kernels
have a specification that does not depend on torch internals:

  * sequential accumulation order of the two voxelisers (C, ``voxel_seq.c``);
  * ``grid_sample(align_corners=True, padding_mode='reflection')`` behind the
    reference's ``2*(x/W - 0.5)`` normalisation (utils/flow_utils.py:114-119);
  * ``F.interpolate(scale_factor=0.5, bilinear, align_corners=True)``
    (e2v/e2v_model.py:190);
  * the 2x2 average-pool pyramid with floor on odd sizes and the transposed
    (2r+1)^2 zero-padded lookup window (ERAFT/corr.py:24-47).

Everything is float32 arithmetic in the same operation order as the torch CPU
kernels, so agreement with ``ref_port`` is ~1 ulp (asserted in
``tests/test_oracle_golden.py``).
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

F32 = np.float32


def build_c_oracle(force: bool = False) -> str:
    """Compile ``voxel_seq.c`` with the committed Makefile; returns the .so path."""
    so = os.path.join(_HERE, "_build", "libcf_oracle.so")
    src = os.path.join(_HERE, "voxel_seq.c")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.run(["make", "-C", _HERE], check=True, stdout=subprocess.DEVNULL)
    return so


def _lib():
    global _LIB
    if _LIB is None:
        _LIB = ctypes.CDLL(build_c_oracle())
        _LIB.cf_oracle_voxel_seq.restype = ctypes.c_int
        _LIB.cf_oracle_voxel_seq.argtypes = [
            ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
            ctypes.c_int, ctypes.c_void_p]
    return _LIB


# ---------------------------------------------------------------- part 1 ---
FLAVOUR_TORCH, FLAVOUR_NUMPY, FLAVOUR_POL = 0, 1, 2


def voxel_grid_sequential(events: np.ndarray, num_bins: int, width: int, height: int,
                          flavour: int = FLAVOUR_TORCH) -> np.ndarray:
    """Event-order sequential binning (see ``voxel_seq.c`` for the flavours)."""
    ev = np.ascontiguousarray(events, dtype=np.float64)
    assert ev.ndim == 2 and ev.shape[1] == 4
    shape = (num_bins, 2, height, width) if flavour == FLAVOUR_POL else (num_bins, height, width)
    grid = np.zeros(shape, np.float32)
    rc = _lib().cf_oracle_voxel_seq(ev.ctypes.data, ev.shape[0], num_bins, height, width,
                                    flavour, grid.ctypes.data)
    if rc != 0:
        raise ValueError(f"cf_oracle_voxel_seq failed with {rc} (event outside the grid?)")
    return grid


def preprocess(grid: np.ndarray, mode: str = "std", hot_threshold: float = 0.0) -> np.ndarray:
    """utils/event_process.py:193-239 with the threshold passed explicitly
    (25/nb for the NumPy variant, 20/nb for the torch one, <= 0 disables).
    Statistics in float64: the kernels accumulate them in fp64 as well, per
    thread and across threads (voxel_stats_kernel), or telescoped out of the
    scatter (the tiled path); only their per-cell map is fp32."""
    g = np.array(grid, dtype=np.float32, copy=True)
    if hot_threshold > 0:
        g[np.abs(g) > F32(hot_threshold)] = 0
    if mode == "maxmin":
        lo, hi = float(g.min()), float(g.max())
        return ((g.astype(np.float64) - lo) / (hi - lo + 1e-8)).astype(np.float32)
    assert mode == "std"
    nz = g != 0
    cnt = int(nz.sum())
    if cnt == 0:
        return g
    g64 = g.astype(np.float64)
    mean = g64.sum() / cnt
    std = np.sqrt((g64 * g64).sum() / cnt - mean * mean)
    return (nz * (g64 - mean) / (std + 1e-8)).astype(np.float32)


# ---------------------------------------------------------------- part 2 ---
def _reflect_clip(pos: np.ndarray, size: int) -> np.ndarray:
    """ATen ``reflect_coordinates(in, 0, 2*(size-1))`` + ``clip_coordinates``."""
    if size == 1:
        return np.zeros_like(pos)
    span = F32(size - 1)
    a = np.abs(pos)
    extra = np.fmod(a, span).astype(F32)
    flips = np.floor(a / span)
    out = np.where(np.mod(flips, 2) == 0, extra, span - extra).astype(F32)
    return np.minimum(F32(size - 1), np.maximum(out, F32(0)))


def _bilinear_gather(img: np.ndarray, ix: np.ndarray, iy: np.ndarray) -> np.ndarray:
    """img [C,H,W]; ix, iy [h,w] float32 pixel positions; taps outside the
    image contribute zero (ATen ``within_bounds_2d``)."""
    C, H, W = img.shape
    x0 = np.floor(ix)
    y0 = np.floor(iy)
    x1, y1 = x0 + 1, y0 + 1
    w_nw = ((x1 - ix) * (y1 - iy)).astype(F32)
    w_ne = ((ix - x0) * (y1 - iy)).astype(F32)
    w_sw = ((x1 - ix) * (iy - y0)).astype(F32)
    w_se = ((ix - x0) * (iy - y0)).astype(F32)
    out = np.zeros((C,) + ix.shape, F32)
    for xs, ys, wt in ((x0, y0, w_nw), (x1, y0, w_ne), (x0, y1, w_sw), (x1, y1, w_se)):
        ok = (xs >= 0) & (xs <= W - 1) & (ys >= 0) & (ys <= H - 1)
        xi = np.clip(xs, 0, W - 1).astype(np.int64)
        yi = np.clip(ys, 0, H - 1).astype(np.int64)
        out += (img[:, yi, xi] * (wt * ok)[None]).astype(F32)
    return out


def warp(img: np.ndarray, flow: np.ndarray, sign: float) -> np.ndarray:
    """utils/flow_utils.py:106-119 (sign=+1, backWarp) / :176-189 (sign=-1,
    forwardWarp).  img [B,C,H,W], flow [B,2,H,W], float32."""
    img = np.asarray(img, F32)
    flow = np.asarray(flow, F32)
    B, C, H, W = img.shape
    gx = np.arange(W, dtype=F32)[None, :]
    gy = np.arange(H, dtype=F32)[:, None]
    out = np.empty_like(img)
    for b in range(B):
        x = (gx + F32(sign) * flow[b, 0]).astype(F32)
        y = (gy + F32(sign) * flow[b, 1]).astype(F32)
        xn = (F32(2) * (x / F32(W) - F32(0.5))).astype(F32)
        yn = (F32(2) * (y / F32(H) - F32(0.5))).astype(F32)
        ix = (((xn + F32(1)) / F32(2)) * F32(W - 1)).astype(F32)
        iy = (((yn + F32(1)) / F32(2)) * F32(H - 1)).astype(F32)
        out[b] = _bilinear_gather(img[b], _reflect_clip(ix, W), _reflect_clip(iy, H))
    return out


def downsample_flow(flow: np.ndarray) -> np.ndarray:
    """``F.interpolate(flow, scale_factor=0.5, mode='bilinear',
    align_corners=True)`` (e2v/e2v_model.py:190), ATen upsample_bilinear2d."""
    flow = np.asarray(flow, F32)
    B, C, H, W = flow.shape
    h, w = int(np.floor(H * 0.5)), int(np.floor(W * 0.5))
    sy = F32((H - 1) / (h - 1)) if h > 1 else F32(0)
    sx = F32((W - 1) / (w - 1)) if w > 1 else F32(0)
    fy = (sy * np.arange(h, dtype=F32)).astype(F32)
    fx = (sx * np.arange(w, dtype=F32)).astype(F32)
    y0 = fy.astype(np.int64)
    x0 = fx.astype(np.int64)
    y1 = y0 + (y0 < H - 1)
    x1 = x0 + (x0 < W - 1)
    ly1 = (fy - y0).astype(F32)[:, None]
    lx1 = (fx - x0).astype(F32)[None, :]
    ly0, lx0 = F32(1) - ly1, F32(1) - lx1
    p00 = flow[:, :, y0][:, :, :, x0]
    p01 = flow[:, :, y0][:, :, :, x1]
    p10 = flow[:, :, y1][:, :, :, x0]
    p11 = flow[:, :, y1][:, :, :, x1]
    return (ly0 * (lx0 * p00 + lx1 * p01) + ly1 * (lx0 * p10 + lx1 * p11)).astype(F32)


# ---------------------------------------------------------------- part 3 ---
def corr_pyramid(fmap1: np.ndarray, fmap2: np.ndarray, num_levels: int = 4) -> list[np.ndarray]:
    """ERAFT/corr.py:13-27,52-60.  Level l: [B*h*w, 1, h>>l, w>>l].  The
    contraction is done in float64 and rounded once (the "true" value of the
    fp32 GEMM); pooling is the float32 a+b+c+d then /4 of ATen avg_pool2d."""
    B, D, h, w = fmap1.shape
    a = fmap1.reshape(B, D, h * w).astype(np.float64)
    b = fmap2.reshape(B, D, h * w).astype(np.float64)
    vol = np.einsum("bdi,bdj->bij", a, b) / np.sqrt(np.float32(D)).astype(np.float64)
    lvl = vol.astype(F32).reshape(B * h * w, 1, h, w)
    pyr = [lvl]
    for _ in range(num_levels - 1):
        hh, ww = lvl.shape[-2] // 2, lvl.shape[-1] // 2
        c = lvl[:, :, : 2 * hh, : 2 * ww]
        s = (c[:, :, 0::2, 0::2] + c[:, :, 0::2, 1::2]).astype(F32)
        s = (s + c[:, :, 1::2, 0::2]).astype(F32)
        s = (s + c[:, :, 1::2, 1::2]).astype(F32)
        lvl = (s / F32(4)).astype(F32)
        pyr.append(lvl)
    return pyr


def corr_lookup(pyramid: list[np.ndarray], coords: np.ndarray, radius: int = 4) -> np.ndarray:
    """ERAFT/corr.py:29-50 + ERAFT/utils.py:7-21.  coords [B,2,h,w] (ch0 = x).
    Output channel l*(2r+1)^2 + i*(2r+1) + j samples level l of query q at
    (cx/2^l + i - r, cy/2^l + j - r)  -- i moves along X (transposed window),
    bilinear, zero outside the map."""
    coords = np.asarray(coords, F32)
    B, _, h, w = coords.shape
    r = radius
    k = 2 * r + 1
    N = h * w
    out = np.zeros((B, len(pyramid) * k * k, h, w), F32)
    cx = coords[:, 0].reshape(B * N)
    cy = coords[:, 1].reshape(B * N)
    q = np.arange(B * N)
    for lvl, vol in enumerate(pyramid):
        Hl, Wl = vol.shape[-2:]
        px = (cx / F32(2 ** lvl)).astype(F32)
        py = (cy / F32(2 ** lvl)).astype(F32)
        for i in range(k):
            for j in range(k):
                x = (px + F32(i - r)).astype(F32)
                y = (py + F32(j - r)).astype(F32)
                # the reference normalises to [-1,1] and grid_sample maps back
                xg = (F32(2) * x / F32(Wl - 1) - F32(1)).astype(F32)
                yg = (F32(2) * y / F32(Hl - 1) - F32(1)).astype(F32)
                x = (((xg + F32(1)) / F32(2)) * F32(Wl - 1)).astype(F32)
                y = (((yg + F32(1)) / F32(2)) * F32(Hl - 1)).astype(F32)
                x0, y0 = np.floor(x), np.floor(y)
                acc = np.zeros(B * N, F32)
                for xs, ys, wt in ((x0, y0, (x0 + 1 - x) * (y0 + 1 - y)),
                                   (x0 + 1, y0, (x - x0) * (y0 + 1 - y)),
                                   (x0, y0 + 1, (x0 + 1 - x) * (y - y0)),
                                   (x0 + 1, y0 + 1, (x - x0) * (y - y0))):
                    ok = (xs >= 0) & (xs <= Wl - 1) & (ys >= 0) & (ys <= Hl - 1)
                    xi = np.clip(xs, 0, Wl - 1).astype(np.int64)
                    yi = np.clip(ys, 0, Hl - 1).astype(np.int64)
                    acc += (vol[q, 0, yi, xi] * (wt.astype(F32) * ok)).astype(F32)
                out[:, lvl * k * k + i * k + j] = acc.reshape(B, h, w)
    return out
