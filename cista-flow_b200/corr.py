"""All-pairs correlation pyramid + lookup: B200 mirror of ``ERAFT/corr.py`` and
``DCEIFlow/core/corr/raft_corr.py`` (the two reference ``CorrBlock`` classes are
bit-identical, SURVEY.md F7).

``CorrBlock(fmap1, fmap2, num_levels=4, radius=4)`` builds the pyramid with the
tcgen05 TF32 GEMM (``cf_corr_build``), exposes it as ``corr_pyramid`` (list of
``[B*h*w, 1, h>>l, w>>l]`` float32 tensors, as in the reference) and
``__call__(coords)`` returns ``[B, num_levels*(2r+1)^2, h, w]`` through one
fused lookup launch (``cf_corr_lookup``) instead of the reference's ~40 small
kernels + 4 host->device copies per call.
"""
from __future__ import annotations

import os

import torch

from . import _lib

# 'tf32' (tcgen05 tensor cores, default), 'fp32' (SIMT, the reference's arithmetic)
# "f16" = fp16 operand copies (kind::f16): same operand significands as "tf32", measured no faster (DESIGN.md)
# "auto" (default): tensor cores, operands carrying an 11-bit significand either way -- TF32 words rounded by the TMA, or
# fp16 copies scaled per batch item where that measured faster (wide maps); the two agree to fp32 summation-order noise
# and the end-to-end PSNR gate (tests/test_e2e_psnr.py) is taken with exactly this operand rounding.
# "3xtf32": tensor cores with each operand split into two TF32 terms (three MMAs per K step): the fp32 accuracy of the
# reference's matmul (held to the same 1e-5 as "fp32"), on the tensor cores instead of the SIMT kernel.
DEFAULT_PRECISION = os.environ.get("CISTAFLOW_CORR_PRECISION", "auto")
_PREC = {"tf32": _lib.CORR_TF32, "fp32": _lib.CORR_FP32, "f16": _lib.CORR_F16, "auto": _lib.CORR_AUTO,
         "3xtf32": _lib.CORR_3XTF32}
# Storage of the pyramid: "f32" (default) or "f16" (cf_corr_build_half: IEEE binary16, half the bytes; the lookup widens
# each tap to fp32; inference-only).  The fp16 pyramid is a precision decision the caller takes; the default stays fp32.
DEFAULT_STORAGE = os.environ.get("CISTAFLOW_CORR_STORAGE", "f32")
_STORAGE = {"f32": torch.float32, "f16": torch.float16}


def _storage(storage: str | None) -> str:
    st = storage or DEFAULT_STORAGE
    if st not in _STORAGE:
        raise ValueError(f"correlation storage {st!r} is not one of {sorted(_STORAGE)}")
    return st


def _check_half(prec: str, D: int, h: int, w: int) -> None:
    """The fp16 pyramid's preconditions (include/cistaflow_half.h), as ValueErrors naming the reason: no silent fp32."""
    if prec in ("fp32", "3xtf32"):
        raise ValueError(f"storage='f16' with precision {prec!r}: fp16 storage would lose its fp32 accuracy "
                         f"(use 'tf32', 'f16' or 'auto')")
    if D % 32 != 0:
        raise ValueError(f"storage='f16' needs D % 32 == 0 (got D={D})")
    if (h * w) % 8 != 0:
        raise ValueError(f"storage='f16' needs h*w % 8 == 0 for a 16-byte row pitch of the fp16 volume (got {h}x{w})")


def _check_no_grad(what: str, *tensors) -> None:
    if torch.is_grad_enabled() and any(t.requires_grad for t in tensors):
        raise RuntimeError(f"cistaflow_b200 {what} is inference-only: an input requires grad "
                           f"(run under torch.no_grad(), or use the default fp32 storage, which is differentiable)")


def coords_grid(batch, ht, wd, device=None):
    """ERAFT/utils.py:24-27 -- [B,2,ht,wd], channel 0 = x index, channel 1 = y index."""
    ys, xs = torch.meshgrid(torch.arange(ht, device=device), torch.arange(wd, device=device), indexing="ij")
    return torch.stack([xs, ys], dim=0).float()[None].repeat(batch, 1, 1, 1)


def _prep(t: torch.Tensor, name: str) -> torch.Tensor:
    _lib.require_cuda(t, name)
    return t.float().contiguous()


def build_pyramid(fmap1: torch.Tensor, fmap2: torch.Tensor, num_levels: int = 4, precision: str | None = None,
                  out: list[torch.Tensor] | None = None, storage: str | None = None):
    """The correlation pyramid.  storage "f32" (default: CISTAFLOW_CORR_STORAGE, else "f32"): float32 levels
    (cf_corr_build); "f16": float16 levels (cf_corr_build_half), which rejects precision "fp32" / "3xtf32" and shapes
    without D % 32 == 0 and h*w % 8 == 0 with a ValueError."""
    st = _storage(storage)
    prec = precision or DEFAULT_PRECISION
    if st == "f16":
        _check_half(prec, *fmap1.shape[1:])
    fmap1, fmap2 = _prep(fmap1, "fmap1"), _prep(fmap2, "fmap2")
    assert fmap1.shape == fmap2.shape and fmap1.dim() == 4
    B, D, h, w = fmap1.shape
    lib = _lib.load()
    if st == "f32" and prec in ("tf32", "f16", "auto", "3xtf32") and (D % 32 != 0 or (h * w) % 4 != 0):
        prec = "fp32"  # shapes the tensor-core tiling does not cover (never the model's: D=256, h,w % 4 == 0)
    dev = fmap1.device
    shapes = [(B * h * w, 1, h >> l, w >> l) for l in range(num_levels)]
    dtype = _STORAGE[st]
    if out is None:
        pyramid = [torch.empty(s, dtype=dtype, device=dev) for s in shapes]
    else:
        pyramid = list(out)
        assert len(pyramid) == num_levels
        for t, s in zip(pyramid, shapes):
            assert tuple(t.shape) == s and t.dtype == dtype and t.is_contiguous() and t.device == dev
    build = lib.cf_corr_build_half if st == "f16" else lib.cf_corr_build
    with torch.cuda.device(dev):
        ws_bytes = lib.cf_corr_workspace_bytes(B, D, h, w, num_levels, _PREC[prec])
        ws = _lib.workspace(ws_bytes, dev)
        rc = build(fmap1.data_ptr(), fmap2.data_ptr(), B, D, h, w, num_levels, _lib.pointer_array(pyramid),
                   _PREC[prec], _lib.ptr(ws), ws_bytes, _lib.stream_ptr(dev))
    _lib.check(rc, "cf_corr_build_half" if st == "f16" else "cf_corr_build")
    return pyramid


def lookup(pyramid, coords: torch.Tensor, radius: int, out: torch.Tensor | None = None) -> torch.Tensor:
    """cf_corr_lookup on a float32 pyramid, cf_corr_lookup_half on a float16 one (fp32 output either way)."""
    half = pyramid[0].dtype == torch.float16
    assert all(p.dtype == (torch.float16 if half else torch.float32) for p in pyramid), "pyramid levels of mixed dtypes"
    coords = _prep(coords, "coords")
    B, two, h, w = coords.shape
    assert two == 2
    levels = len(pyramid)
    assert pyramid[0].shape[0] == B * h * w, "coords do not match the pyramid"
    k = 2 * radius + 1
    if out is None:
        out = torch.empty((B, levels * k * k, h, w), dtype=torch.float32, device=coords.device)
    lib = _lib.load()
    with torch.cuda.device(coords.device):
        fn = lib.cf_corr_lookup_half if half else lib.cf_corr_lookup
        rc = fn(_lib.pointer_array(pyramid), coords.data_ptr(), B, h, w, levels, radius, out.data_ptr(),
                _lib.stream_ptr(coords.device))
    _lib.check(rc, "cf_corr_lookup_half" if half else "cf_corr_lookup")
    return out


class _PyramidFunction(torch.autograd.Function):
    """Forward: cf_corr_build.  Backward (training, SURVEY 8f rank 2): the level gradients are folded into the
    level-0 volume through the adjoint of avg_pool2d(2, 2) (each pooled cell spreads g/4 to its 2x2 window; a
    floored odd row/column gets nothing) and the two feature-map gradients are plain GEMMs
    (grad_f1 = f2 . G^T / sqrt(D), grad_f2 = f1 . G / sqrt(D)) -- torch.matmul, a library GEMM, like the reference's."""

    @staticmethod
    def forward(ctx, fmap1, fmap2, num_levels, precision):
        ctx.save_for_backward(fmap1, fmap2)
        pyramid = build_pyramid(fmap1, fmap2, num_levels, precision, storage="f32")
        return tuple(pyramid)

    @staticmethod
    def backward(ctx, *grads):
        fmap1, fmap2 = ctx.saved_tensors
        B, D, h, w = fmap1.shape
        N = h * w
        total = None
        for l in reversed(range(len(grads))):
            g = grads[l]
            if total is not None:   # adjoint of avg_pool2d: level l+1 -> level l
                hl, wl = h >> l, w >> l
                up = torch.nn.functional.interpolate(total, scale_factor=2, mode="nearest") * 0.25
                up = torch.nn.functional.pad(up, (0, wl - up.shape[3], 0, hl - up.shape[2]))
                total = up if g is None else up + g
            elif g is not None:
                total = g.float()
        if total is None:
            return None, None, None, None
        G = total.reshape(B, N, N) / float(D) ** 0.5          # d loss / d (f1^T f2)
        f1, f2 = fmap1.reshape(B, D, N).float(), fmap2.reshape(B, D, N).float()
        grad_f1 = torch.matmul(f2, G.transpose(1, 2)).reshape(B, D, h, w) if ctx.needs_input_grad[0] else None
        grad_f2 = torch.matmul(f1, G).reshape(B, D, h, w) if ctx.needs_input_grad[1] else None
        return grad_f1, grad_f2, None, None


class _LookupFunction(torch.autograd.Function):
    """Forward: cf_corr_lookup.  Backward: cf_corr_lookup_backward (patch gradients by gather, coordinate gradient)."""

    @staticmethod
    def forward(ctx, coords, radius, *pyramid):
        ctx.radius = radius
        ctx.save_for_backward(coords, *pyramid)
        return lookup(list(pyramid), coords, radius)

    @staticmethod
    def backward(ctx, grad_out):
        coords, *pyramid = ctx.saved_tensors
        B, _, h, w = coords.shape
        levels = len(pyramid)
        want_coords = ctx.needs_input_grad[0]
        want_pyr = any(ctx.needs_input_grad[2:])
        grad_out = grad_out.float().contiguous()
        grad_coords = torch.empty_like(coords) if want_coords else None
        grad_pyr = [torch.empty_like(p) for p in pyramid] if want_pyr else None
        lib = _lib.load()
        with torch.cuda.device(coords.device):
            rc = lib.cf_corr_lookup_backward(grad_out.data_ptr(), _lib.pointer_array(pyramid), coords.data_ptr(), B, h, w,
                                             levels, ctx.radius, _lib.pointer_array(grad_pyr) if want_pyr else None,
                                             _lib.ptr(grad_coords), _lib.stream_ptr(coords.device))
        _lib.check(rc, "cf_corr_lookup_backward")
        return (grad_coords, None, *(grad_pyr if want_pyr else [None] * levels))


class CorrBlock:
    """Drop-in for ``ERAFT/corr.py:12-60`` / ``raft_corr.py:15-65``.  Differentiable like the reference's:
    gradients reach the feature maps and the lookup coordinates when they are being recorded.

    ``storage="f16"`` (or CISTAFLOW_CORR_STORAGE=f16) keeps ``corr_pyramid`` as float16 tensors: half the memory, the
    reference's HalfCorrBlock choice.  That pyramid is inference-only (RuntimeError when an input requires grad while
    gradients are recorded); ``CorrBlock.corr`` is unaffected."""

    def __init__(self, fmap1, fmap2, num_levels=4, radius=4, precision=None, storage=None):
        self.num_levels = num_levels
        self.radius = radius
        self.storage = _storage(storage)
        if self.storage == "f16":
            _check_no_grad("CorrBlock with storage='f16'", fmap1, fmap2)
            with torch.no_grad():
                self.corr_pyramid = build_pyramid(fmap1, fmap2, num_levels, precision, storage="f16")
        elif torch.is_grad_enabled() and (fmap1.requires_grad or fmap2.requires_grad):
            self.corr_pyramid = list(_PyramidFunction.apply(_prep(fmap1, "fmap1"), _prep(fmap2, "fmap2"), num_levels, precision))
        else:
            with torch.no_grad():
                self.corr_pyramid = build_pyramid(fmap1, fmap2, num_levels, precision, storage="f32")

    def __call__(self, coords):
        if self.storage == "f16":
            _check_no_grad("CorrBlock with storage='f16'", coords)
        if torch.is_grad_enabled() and (coords.requires_grad or any(p.requires_grad for p in self.corr_pyramid)):
            return _LookupFunction.apply(_prep(coords, "coords"), self.radius, *self.corr_pyramid)
        with torch.no_grad():
            return lookup(self.corr_pyramid, coords, self.radius)

    @staticmethod
    def corr(fmap1, fmap2, precision=None):
        """[B, h, w, 1, h, w] = <fmap1, fmap2> / sqrt(D)  (ERAFT/corr.py:52-60).  Differentiable like the reference's
        when gradients are being recorded."""
        B, D, h, w = fmap1.shape
        if torch.is_grad_enabled() and (fmap1.requires_grad or fmap2.requires_grad):
            vol = _PyramidFunction.apply(_prep(fmap1, "fmap1"), _prep(fmap2, "fmap2"), 1, precision)[0]
        else:
            with torch.no_grad():
                vol = build_pyramid(fmap1, fmap2, 1, precision, storage="f32")[0]
        return vol.view(B, h, w, 1, h, w)


# AlternateCorrBlock: "tf32" / "f16" / "auto" run on the tensor cores (TF32 operands), "fp32" / "3xtf32" on the fp32
# SIMT kernel, so that an fp32-accurate request gets fp32 accuracy
_ALT_PREC = {"tf32": _lib.CORR_TF32, "f16": _lib.CORR_AUTO, "auto": _lib.CORR_AUTO, "fp32": _lib.CORR_FP32,
             "3xtf32": _lib.CORR_FP32}


class AlternateCorrBlock:
    """Drop-in for ``DCEIFlow/core/corr/raft_corr.py:175-203`` (RAFT's AlternateCorrBlock): the lookup of
    ``CorrBlock`` without the all-pairs volume.  The block keeps fmap1 and the average-pooled levels of fmap2
    (``cf_corr_alt_prepare``, O(B*D*h*w) bytes) and every call computes the dot products around each query on the
    tensor cores (``cf_corr_alt_lookup``).  The output equals ``CorrBlock(fmap1, fmap2, ...)(coords)`` up to fp32
    summation order and operand rounding.  Inference-only, like the reference's (it calls alt_cuda_corr.forward)."""

    def __init__(self, fmap1, fmap2, num_levels=4, radius=4, precision=None):
        self.num_levels = num_levels
        self.radius = radius
        prec = precision or DEFAULT_PRECISION
        if prec not in _ALT_PREC:
            raise ValueError(f"AlternateCorrBlock: precision {prec!r} is not one of {sorted(_ALT_PREC)}")
        self.precision = _ALT_PREC[prec]
        self._check_no_grad(fmap1, fmap2)
        fmap1, fmap2 = _prep(fmap1, "fmap1"), _prep(fmap2, "fmap2")
        assert fmap1.shape == fmap2.shape and fmap1.dim() == 4
        self.shape = tuple(fmap1.shape)
        B, D, h, w = self.shape
        lib = _lib.load()
        dev = fmap1.device
        with torch.cuda.device(dev):
            nbytes = lib.cf_corr_alt_workspace_bytes(B, D, h, w, num_levels, self.precision)
            self.state = _lib.workspace(nbytes, dev)
            rc = lib.cf_corr_alt_prepare(fmap1.data_ptr(), fmap2.data_ptr(), B, D, h, w, num_levels, self.precision,
                                         _lib.ptr(self.state), nbytes, _lib.stream_ptr(dev))
        _lib.check(rc, "cf_corr_alt_prepare")

    @staticmethod
    def _check_no_grad(*tensors):
        if torch.is_grad_enabled() and any(t.requires_grad for t in tensors):
            raise RuntimeError("cistaflow_b200 AlternateCorrBlock is inference-only: an input requires grad "
                               "(run under torch.no_grad(), or use CorrBlock, which is differentiable)")

    def __call__(self, coords):
        self._check_no_grad(coords)
        coords = _prep(coords, "coords")
        B, D, h, w = self.shape
        assert tuple(coords.shape) == (B, 2, h, w), "coords do not match the feature maps"
        k = 2 * self.radius + 1
        out = torch.empty((B, self.num_levels * k * k, h, w), dtype=torch.float32, device=coords.device)
        lib = _lib.load()
        with torch.cuda.device(coords.device):
            rc = lib.cf_corr_alt_lookup(_lib.ptr(self.state), coords.data_ptr(), B, D, h, w, self.num_levels, self.radius,
                                        self.precision, out.data_ptr(), _lib.stream_ptr(coords.device))
        _lib.check(rc, "cf_corr_alt_lookup")
        return out
