"""Flow-guided warp: B200 mirror of the reference's ``utils/flow_utils.py``.

Same classes and signatures (``backWarp(W, H)``, ``forwardWarp(W, H)``,
``FrameWarp(mode).warp_frame(I, flow)``, utils/flow_utils.py:40-221).  In the
reference both "modes" are a bilinear gather through ``grid_sample`` and differ
only in the sign of the flow (SURVEY.md F5); one CUDA kernel (``cf_warp``)
serves both.  ``warp_frame_and_codes`` is the fused per-frame step of
``e2v/e2v_model.py:188-191`` (image + sparse codes, x0.5 flow down-sampling
done inside the kernel).

Autograd: ``warp`` (hence ``backWarp`` / ``forwardWarp`` / ``FrameWarp.warp_frame``) is differentiable
w.r.t. both the image and the flow -- the backward is ``cf_warp_backward``, the bilinear splat (the
reference trains through these modules, loss.py:147,336,398).  Under ``torch.use_deterministic_algorithms(True)``
it is ``cf_warp_backward_det`` instead: the same gradients summed in a fixed order, bitwise reproducible.  The fused ``warp_frame_and_codes`` step is
inference-only (the evaluation drivers run under ``torch.no_grad()``).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib


def _prep(t: torch.Tensor, name: str, allow_grad: bool = False) -> torch.Tensor:
    _lib.require_cuda(t, name)
    if not allow_grad and torch.is_grad_enabled() and t.requires_grad:
        raise RuntimeError(f"cistaflow_b200 warp_frame_and_codes is inference-only: {name} requires grad "
                           f"(run under torch.no_grad(), or use warp() / FrameWarp.warp_frame, which are differentiable)")
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


class _WarpFunction(torch.autograd.Function):
    """cf_warp forward, cf_warp_backward (bilinear splat + flow gradient) backward; cf_warp_backward_det when
    torch.are_deterministic_algorithms_enabled()."""

    @staticmethod
    def forward(ctx, img, flow, sign):
        ctx.sign = float(sign)
        ctx.save_for_backward(img, flow)
        return _warp_forward(img, flow, sign, None)

    @staticmethod
    def backward(ctx, grad_out):
        img, flow = ctx.saved_tensors
        need_img, need_flow = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        grad_out = grad_out.float().contiguous()
        B, C, H, W = img.shape
        grad_img = torch.empty_like(img) if need_img else None
        grad_flow = torch.empty_like(flow) if need_flow else None
        lib = _lib.load()
        fH, fW = flow.shape[2], flow.shape[3]
        with torch.cuda.device(img.device):
            if torch.are_deterministic_algorithms_enabled():
                # torch.use_deterministic_algorithms(True): the sort + gather adjoint, no float atomics
                name = "cf_warp_backward_det"
                ws_bytes = lib.cf_warp_backward_det_workspace_bytes(B, C, H, W, fH, fW)
                ws = _lib.workspace(ws_bytes, img.device)
                rc = lib.cf_warp_backward_det(grad_out.data_ptr(), img.data_ptr(), flow.data_ptr(), _lib.ptr(grad_img),
                                              _lib.ptr(grad_flow), B, C, H, W, fH, fW, ctx.sign, _lib.ptr(ws), ws_bytes,
                                              _lib.stream_ptr(img.device))
            else:
                name = "cf_warp_backward"
                rc = lib.cf_warp_backward(grad_out.data_ptr(), img.data_ptr(), flow.data_ptr(), _lib.ptr(grad_img),
                                          _lib.ptr(grad_flow), B, C, H, W, fH, fW, ctx.sign, _lib.stream_ptr(img.device))
        _lib.check(rc, name)
        return grad_img, grad_flow, None


def warp(img: torch.Tensor, flow: torch.Tensor, sign: float, out: torch.Tensor | None = None) -> torch.Tensor:
    """Differentiable front end of ``cf_warp`` (see ``_warp_forward`` for the maths)."""
    if torch.is_grad_enabled() and (img.requires_grad or flow.requires_grad):
        assert out is None, "out= is not supported when gradients are recorded"
        return _WarpFunction.apply(_prep(img, "img", True), _prep(flow, "flow", True), sign)
    return _warp_forward(img, flow, sign, out)


def _warp_forward(img: torch.Tensor, flow: torch.Tensor, sign: float, out: torch.Tensor | None = None) -> torch.Tensor:
    """out[b,c,y,x] = bilinear(img[b,c], reflect((x+sign*u)(W-1)/W, (y+sign*v)(H-1)/H)).

    ``flow`` is either at the image's resolution or at twice the resolution
    (then the reference's x0.5 bilinear align_corners=True down-sampling is
    fused, values not rescaled)."""
    img, flow = _prep(img, "img", True), _prep(flow, "flow", True)
    assert img.dim() == 4 and flow.dim() == 4 and flow.shape[1] == 2 and flow.shape[0] == img.shape[0]
    assert img.device == flow.device
    B, C, H, W = img.shape
    if out is None:
        out = torch.empty_like(img)
    lib = _lib.load()
    with torch.cuda.device(img.device):
        rc = lib.cf_warp(img.data_ptr(), flow.data_ptr(), out.data_ptr(), B, C, H, W, flow.shape[2], flow.shape[3],
                         float(sign), _lib.stream_ptr(img.device))
    _lib.check(rc, "cf_warp")
    return out


def flow_any(flow: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """``flow.any()`` as a device-side int32 flag (1 = some element is non-zero), no host synchronisation.
    The reference reads this predicate on the host in every frame (e2v/e2v_model.py:184, 236)."""
    flow = _prep(flow, "flow")
    if out is None:
        out = torch.empty(1, dtype=torch.int32, device=flow.device)
    assert out.dtype == torch.int32 and out.numel() >= 1 and out.device == flow.device
    lib = _lib.load()
    with torch.cuda.device(flow.device):
        rc = lib.cf_flow_any(flow.data_ptr(), flow.numel(), out.data_ptr(), _lib.stream_ptr(flow.device))
    _lib.check(rc, "cf_flow_any")
    return out


def warp_frame_and_codes(img: torch.Tensor, codes: torch.Tensor, flow: torch.Tensor, mode: str = "forward",
                         out: tuple[torch.Tensor, torch.Tensor] | None = None, skip_zero_flow: bool = False,
                         gate: torch.Tensor | None = None):
    """One launch for ``e2v/e2v_model.py:188-191``: returns (warped image, warped codes).
    img [B,Ci,H,W], codes [B,Cz,H//2,W//2], flow [B,2,H,W].

    ``skip_zero_flow=True`` reproduces the whole branch of ``e2v_model.py:184-191`` -- when the flow is all zero
    the reference skips the warp and keeps ``rec_img0`` / ``states[1]`` -- with the predicate evaluated on the
    device (``cf_flow_any`` + a gated kernel that copies instead of warping): no ``.any()`` read-back, so the frame
    step stays asynchronous and can be captured in a CUDA graph.  ``gate`` passes a flag computed earlier."""
    img, codes, flow = _prep(img, "img"), _prep(codes, "codes"), _prep(flow, "flow")
    B, Ci, H, W = img.shape
    assert flow.shape == (B, 2, H, W), "flow must be [B,2,H,W] at the image resolution"
    assert codes.shape[0] == B and codes.shape[2] == H // 2 and codes.shape[3] == W // 2, \
        "codes must be [B,C,H//2,W//2]"
    if out is None:
        img_out, codes_out = torch.empty_like(img), torch.empty_like(codes)
    else:
        img_out, codes_out = out
        for o, ref in ((img_out, img), (codes_out, codes)):
            assert o.shape == ref.shape and o.dtype == torch.float32 and o.is_contiguous() and o.device == ref.device
    sign = -1.0 if mode == "forward" else 1.0
    if skip_zero_flow and gate is None:
        gate = flow_any(flow)
    if gate is not None:
        assert gate.dtype == torch.int32 and gate.device == img.device
    lib = _lib.load()
    with torch.cuda.device(img.device):
        rc = lib.cf_warp_frame_and_codes_gated(img.data_ptr(), codes.data_ptr(), flow.data_ptr(), img_out.data_ptr(),
                                               codes_out.data_ptr(), B, Ci, codes.shape[1], H, W, sign,
                                               _lib.ptr(gate), _lib.stream_ptr(img.device))
    _lib.check(rc, "cf_warp_frame_and_codes")
    return img_out, codes_out


def warp_frame_and_codes_upflow8(img: torch.Tensor, codes: torch.Tensor, flow_lr: torch.Tensor, mode: str = "forward",
                                 pad: tuple[int, int] | None = None, return_flow: bool = True):
    """The whole tail of the reference's frame step in ONE launch (SURVEY 8f rank 1): ``upflow8`` of the flow network's
    1/8-resolution output (DCEIFlow/utils/sample_utils.py:66-68), ``ImagePadder.unpad`` (utils/image_process.py:103-107),
    warp of the previous frame, x0.5 down-sampling of the flow and warp of the sparse codes (e2v/e2v_model.py:188-191).

    img [B,Ci,H,W], codes [B,Cz,H//2,W//2], flow_lr [B,2,lh,lw] with 8*lh = H + pad_h, 8*lw = W + pad_w (top/left
    padding; ``pad`` defaults to what ImagePadder(min_size=32) adds).  Returns (warped image, warped codes, flow_final
    [B,2,H,W] or None)."""
    img, codes, flow_lr = _prep(img, "img"), _prep(codes, "codes"), _prep(flow_lr, "flow_lr")
    B, Ci, H, W = img.shape
    lh, lw = flow_lr.shape[2], flow_lr.shape[3]
    if pad is None:
        pad = (8 * lh - H, 8 * lw - W)
    pad_h, pad_w = int(pad[0]), int(pad[1])
    if not (tuple(flow_lr.shape[:2]) == (B, 2) and 8 * lh - pad_h == H and 8 * lw - pad_w == W):
        raise ValueError(f"flow_lr must be [B,2,(H+pad_h)/8,(W+pad_w)/8]: got {tuple(flow_lr.shape)} for a {H}x{W} frame "
                         f"with padding ({pad_h}, {pad_w})")
    assert codes.shape[0] == B and codes.shape[2] == H // 2 and codes.shape[3] == W // 2, "codes must be [B,C,H//2,W//2]"
    img_out, codes_out = torch.empty_like(img), torch.empty_like(codes)
    flow_out = torch.empty((B, 2, H, W), dtype=torch.float32, device=img.device) if return_flow else None
    sign = -1.0 if mode == "forward" else 1.0
    lib = _lib.load()
    with torch.cuda.device(img.device):
        rc = lib.cf_warp_frame_and_codes_upflow8(img.data_ptr(), codes.data_ptr(), flow_lr.data_ptr(), img_out.data_ptr(),
                                                 codes_out.data_ptr(), _lib.ptr(flow_out), B, Ci, codes.shape[1], H, W, lh, lw,
                                                 pad_h, pad_w, sign, _lib.stream_ptr(img.device))
    _lib.check(rc, "cf_warp_frame_and_codes_upflow8")
    return img_out, codes_out, flow_out


class backWarp(nn.Module):
    """I0 = backwarp(I1, F_0_1): gather at (x+u, y+v)  (utils/flow_utils.py:40-120).
    Note the (W, H) argument order of the reference."""

    def __init__(self, W, H):
        super().__init__()
        self.W, self.H = W, H

    def forward(self, img, flow):
        return warp(img, flow, +1.0)


class forwardWarp(nn.Module):
    """I1 = forwardwarp(I0, F_0_1): gather at (x-u, y-v)  (utils/flow_utils.py:123-190)."""

    def __init__(self, W, H):
        super().__init__()
        self.W, self.H = W, H

    def forward(self, img, flow):
        return warp(img, flow, -1.0)


class FrameWarp(object):
    """utils/flow_utils.py:193-221: dispatch on mode, one cached module per (W, H)."""

    def __init__(self, mode):
        self.mode = mode
        self.flowWarp_dict = dict()

    def get_flowWarp_module(self, width: int, height: int):
        module = self.flowWarp_dict.get((width, height))
        if module is None:
            module = forwardWarp(width, height) if self.mode == "forward" else backWarp(width, height)
            self.flowWarp_dict[(width, height)] = module
        return module

    def warp_frame(self, I, flow):
        height, width = I.shape[-2:]
        return self.get_flowWarp_module(width, height)(I, flow)

    def warp_frame_and_codes(self, I, Z, flow, skip_zero_flow: bool = False):
        """Fused image + codes step (extension; not in the reference)."""
        return warp_frame_and_codes(I, Z, flow, self.mode, skip_zero_flow=skip_zero_flow)
