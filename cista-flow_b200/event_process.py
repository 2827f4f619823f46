"""Event stream -> voxel grid: B200 mirror of the reference's ``utils/event_process.py``.

Same names, argument meaning and return types as the reference, so that
``from utils.event_process import events_to_voxel_grid, event_preprocess`` can
be re-pointed here (see ``install.py``):

  events_to_voxel_grid(events, num_bins, width, height, is_reverse=False)
        -> np.ndarray float32 [nb,H,W]            (utils/event_process.py:15-72)
  events_to_voxel_grid_pol(events, num_bins, width, height)
        -> np.ndarray float32 [nb,2,H,W]          (utils/event_process.py:75-123)
  events_to_voxel_grid_pytorch(events, num_bins, width, height)
        -> torch.Tensor float32 [nb,H,W] on events.device   (:127-190)
  event_preprocess(grid, mode='std', filter_hot_pixel=False)          (:193-216)
  event_preprocess_pytorch(grid, mode='std', filter_hot_pixel=False)  (:219-239)

plus the batched device-resident form the GPU path is designed around
(``events_to_voxel_grid_batched``): many windows per launch, fused statistics
and normalisation, result stays in HBM for the network.

All arithmetic runs in ``libcistaflow.so`` on the GPU (NumPy/CPU inputs are
staged to the current CUDA device and the result copied back, so the drop-in
contract "result lives where the input lived" is kept).  Differences from the
reference, all deliberate:
  * inputs are never mutated (the reference rewrites ``events[:,3]`` and
    ``events[:,0]`` in place, :51/:159);
  * ``event_preprocess`` returns float32 (the reference silently returns
    float64 under NumPy >= 2, SURVEY.md F9);
  * events with x >= width or y >= height (or a negative coordinate) are DROPPED.  The reference does not check: its
    NumPy variants scatter into the flattened grid at ``x + y*W + ti*W*H`` (:61-66), so an event with x == W silently
    lands on column 0 of the next row (or of the next bin for the last row) and only an index past the end of the array
    raises; its callers filter first (``event_window[event_window[:,1] < self.width]``, data_readers/video_readers.py:
    208-209).  Feed pre-filtered events -- ``filter_events`` does the reader's filter on the device -- and the results
    are identical; the divergence on unfiltered input is pinned by
    tests/test_gpu_parity_r2.py::test_out_of_grid_events_are_dropped_where_the_reference_wraps.
"""
from __future__ import annotations

import os
import warnings

import numpy as np
import torch

from . import _lib

# 'atomic' (fast, <=1e-5 rel.) or 'deterministic' (bit-exact vs the reference's
# sequential accumulation).  Override per call with mode=... or globally here;
# torch.use_deterministic_algorithms(True) makes the default 'deterministic' (resolve_mode).
DEFAULT_MODE = os.environ.get("CISTAFLOW_VOXEL_MODE", "atomic")

_MODES = {"atomic": _lib.VOXEL_ATOMIC, "deterministic": _lib.VOXEL_DETERMINISTIC,
          # 'atomic' with the data path forced (tests / experiments): RED.ADD into the L2-resident grid, or
          # partition + shared-memory tiles (no global atomics)
          "atomic_l2": _lib.VOXEL_ATOMIC_L2, "atomic_tiled": _lib.VOXEL_ATOMIC_TILED}
_PRE = {None: _lib.PRE_NONE, "none": _lib.PRE_NONE, "std": _lib.PRE_STD, "maxmin": _lib.PRE_MAXMIN}
_FLAVOURS = {"torch": _lib.FLAVOUR_TORCH, "numpy": _lib.FLAVOUR_NUMPY, "pol": _lib.FLAVOUR_POL,
             "mvsec": _lib.FLAVOUR_MVSEC}


def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("cistaflow_b200 needs a CUDA device (B200); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def resolve_mode(mode: str | None) -> str:
    """The voxel mode a call runs: an explicit ``mode`` wins; otherwise 'deterministic' while
    ``torch.use_deterministic_algorithms(True)`` is in force, else ``DEFAULT_MODE``."""
    if mode:
        return mode
    return "deterministic" if torch.are_deterministic_algorithms_enabled() else DEFAULT_MODE


def _check_args(events, num_bins, width, height):
    # same asserts as the reference (utils/event_process.py:23-26)
    assert events.shape[1] == 4
    assert num_bins > 0
    assert width > 0
    assert height > 0


def events_to_voxel_grid_batched(events: torch.Tensor, offsets: torch.Tensor, num_bins: int, width: int,
                                 height: int, normalize: str | None = None, filter_hot_pixel: bool = False,
                                 hot_threshold: float | None = None, flavour: str = "numpy",
                                 mode: str | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
    """B windows in one launch.

    events   float64 CUDA tensor [sum N_b, 4] rows (t, x, y, p), windows concatenated
    offsets  int64 CUDA tensor [B+1]
    returns  float32 [B, nb, H, W] ([B, nb, 2, H, W] for flavour='pol') on the same device

    ``normalize`` fuses ``event_preprocess`` ('std' / 'maxmin'); the hot-pixel
    threshold defaults to the reference's 25/nb (flavour numpy/pol) or 20/nb
    (flavour torch) when ``filter_hot_pixel`` is set.
    """
    _lib.require_cuda(events, "events")
    _lib.require_cuda(offsets, "offsets")
    _check_args(events, num_bins, width, height)
    if events.dtype != torch.float64:
        events = events.double()
    events = events.contiguous()
    offsets = offsets.to(torch.int64).contiguous()
    B = offsets.numel() - 1
    mode_id = _MODES[resolve_mode(mode)]
    flav = _FLAVOURS[flavour]
    pre = _PRE[normalize]
    thr = 0.0
    if filter_hot_pixel:
        thr = hot_threshold if hot_threshold is not None else (20.0 if flavour == "torch" else 25.0) / num_bins
    shape = (B, num_bins, 2, height, width) if flavour == "pol" else (B, num_bins, height, width)
    dev = events.device
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=dev)
    else:
        assert out.shape == shape and out.dtype == torch.float32 and out.is_contiguous() and out.device == dev
    lib = _lib.load()
    total = events.shape[0]
    with torch.cuda.device(dev):
        ws_bytes = lib.cf_voxel_workspace_bytes(total, B, num_bins, height, width, mode_id, flav, pre)
        ws = _lib.workspace(ws_bytes, dev)
        rc = lib.cf_voxel_bin(_lib.ptr(events) if total else None, offsets.data_ptr(), total, B, num_bins, height,
                              width, mode_id, flav, pre, thr, out.data_ptr(), _lib.ptr(ws), ws_bytes,
                              _lib.stream_ptr(dev))
    _lib.check(rc, "cf_voxel_bin")
    return out


# ---- packed event ingest (8 bytes per event; include/cistaflow.h part 1b) ---------------------------------
def pack_events_host(events: np.ndarray, offsets: np.ndarray | None = None) -> np.ndarray:
    """NumPy packer for the host side of the ingest path: float64 [N,4] rows (t, x, y, p) -> uint64 [N],
    low word = float32 (t - t_first_of_window) (fp64 subtraction first), high word = x | y << 16 | p << 31.
    Pack on the host, upload 8 B/event instead of 32 B/event.  Same bits as the device packer
    (``pack_events`` on a CUDA tensor)."""
    ev = np.ascontiguousarray(events, dtype=np.float64)
    assert ev.ndim == 2 and ev.shape[1] == 4
    n = ev.shape[0]
    if offsets is None:
        offsets = np.array([0, n], dtype=np.int64)
    offsets = np.asarray(offsets, dtype=np.int64)
    t0 = np.zeros(n, dtype=np.float64)
    for b in range(len(offsets) - 1):
        if offsets[b + 1] > offsets[b]:
            t0[offsets[b]:offsets[b + 1]] = ev[offsets[b], 0]
    # a row outside [offsets[0], offsets[B]) belongs to no window: the invalid record (x = 0xffff, t_rel = 0)
    inside = np.zeros(n, dtype=bool)
    inside[offsets[0]:offsets[-1]] = True
    t_rel = np.where(inside, ev[:, 0] - t0, 0.0).astype(np.float32).view(np.uint32).astype(np.uint64)
    ok = inside & (ev[:, 1] >= 0) & (ev[:, 1] < 65535) & (ev[:, 2] >= 0) & (ev[:, 2] < 32768)
    x = np.where(ok, ev[:, 1], 65535).astype(np.uint64)      # truncation like the kernels' (int) conversion
    y = np.where(ok, ev[:, 2], 0).astype(np.uint64)
    p = (inside & (ev[:, 3] > 0)).astype(np.uint64)
    return t_rel | ((x | (y << np.uint64(16)) | (p << np.uint64(31))) << np.uint64(32))


def pack_events(events: torch.Tensor, offsets: torch.Tensor) -> torch.Tensor:
    """Device packer: CUDA float64 [N,4] + int64 offsets [B+1] -> int64 [N] (the bits of the uint64 records)."""
    _lib.require_cuda(events, "events")
    _lib.require_cuda(offsets, "offsets")
    assert events.dim() == 2 and events.shape[1] == 4
    events = events.double().contiguous()
    offsets = offsets.to(torch.int64).contiguous()
    packed = torch.empty(events.shape[0], dtype=torch.int64, device=events.device)
    lib = _lib.load()
    with torch.cuda.device(events.device):
        rc = lib.cf_events_pack(_lib.ptr(events) if events.shape[0] else None, offsets.data_ptr(), events.shape[0],
                                offsets.numel() - 1, packed.data_ptr(), _lib.stream_ptr(events.device))
    _lib.check(rc, "cf_events_pack")
    return packed


def events_to_voxel_grid_packed(packed: torch.Tensor, offsets: torch.Tensor, num_bins: int, width: int, height: int,
                                normalize: str | None = None, filter_hot_pixel: bool = False,
                                hot_threshold: float | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
    """``events_to_voxel_grid_batched`` for packed events (int64/uint64 CUDA tensor [sum N_b]): reads 8 B per
    event.  Atomic-mode numerics; polarity and the 25/nb hot-pixel default follow ``events_to_voxel_grid``.
    There is no deterministic form: under ``torch.use_deterministic_algorithms(True)`` it raises RuntimeError (warns
    with ``warn_only=True``), as torch does for its ops without a deterministic implementation."""
    if torch.are_deterministic_algorithms_enabled():
        msg = ("events_to_voxel_grid_packed does not have a deterministic implementation (it accumulates with fp32 "
               "atomics), but you set 'torch.use_deterministic_algorithms(True)'. Unpacked events through "
               "events_to_voxel_grid_batched(..., mode='deterministic') are bit-exact.")
        if not torch.is_deterministic_algorithms_warn_only_enabled():
            raise RuntimeError(msg)
        warnings.warn(msg)
    _lib.require_cuda(packed, "packed")
    _lib.require_cuda(offsets, "offsets")
    assert packed.dim() == 1 and packed.element_size() == 8
    assert num_bins > 0 and width > 0 and height > 0
    packed = packed.contiguous()
    offsets = offsets.to(torch.int64).contiguous()
    B = offsets.numel() - 1
    thr = 0.0
    if filter_hot_pixel:
        thr = hot_threshold if hot_threshold is not None else 25.0 / num_bins
    dev = packed.device
    shape = (B, num_bins, height, width)
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=dev)
    else:
        assert out.shape == shape and out.dtype == torch.float32 and out.is_contiguous() and out.device == dev
    lib = _lib.load()
    with torch.cuda.device(dev):
        ws_bytes = lib.cf_preprocess_workspace_bytes(B, num_bins * height * width) if normalize else 0
        ws = _lib.workspace(ws_bytes, dev)
        rc = lib.cf_voxel_bin_packed(_lib.ptr(packed) if packed.numel() else None, offsets.data_ptr(), packed.numel(), B,
                                     num_bins, height, width, _PRE[normalize], thr, out.data_ptr(), _lib.ptr(ws), ws_bytes,
                                     _lib.stream_ptr(dev))
    _lib.check(rc, "cf_voxel_bin_packed")
    return out


# ---- device-side windowing (include/cistaflow.h: cf_events_filter, cf_event_window_offsets) -----------------------------
def filter_events(events: torch.Tensor, width: int, height: int):
    """``event_window[event_window[:,1] < width]`` then ``[:,2] < height`` (data_readers/video_readers.py:208-209) on the
    device, stable, without a read-back: returns (compacted float64 [N,4] buffer, device int64 scalar = rows kept).
    Rows past the kept count are unspecified."""
    _lib.require_cuda(events, "events")
    assert events.dim() == 2 and events.shape[1] == 4
    events = events.double().contiguous()
    n = events.shape[0]
    out = torch.empty_like(events)
    kept = torch.empty(1, dtype=torch.int64, device=events.device)
    lib = _lib.load()
    with torch.cuda.device(events.device):
        ws_bytes = lib.cf_events_filter_workspace_bytes(n)
        ws = _lib.workspace(ws_bytes, events.device)
        rc = lib.cf_events_filter(_lib.ptr(events) if n else None, n, int(width), int(height), _lib.ptr(out) if n else None,
                                  kept.data_ptr(), _lib.ptr(ws), ws_bytes, _lib.stream_ptr(events.device))
    _lib.check(rc, "cf_events_filter")
    return out, kept


def window_offsets(count: torch.Tensor, param: int, max_windows: int, policy: str = "fixed"):
    """Window boundaries from a device-resident event count: policy 'fixed' = windows of ``param`` events, the last keeps
    the remainder (FixedSizeEventReader, data_readers/event_readers.py:6-47); 'split' = ``np.array_split`` into
    ``max(1, round(count / param))`` windows (limit_num_events, video_readers.py:219-224).  Returns (offsets int64
    [max_windows + 1] with trailing empty windows, device int32 scalar = number of windows) -- both stay on the device."""
    _lib.require_cuda(count, "count")
    assert count.dtype == torch.int64 and count.numel() == 1
    offsets = torch.empty(max_windows + 1, dtype=torch.int64, device=count.device)
    n_windows = torch.empty(1, dtype=torch.int32, device=count.device)
    pol = {"fixed": _lib.WINDOWS_FIXED, "split": _lib.WINDOWS_SPLIT}[policy]
    lib = _lib.load()
    with torch.cuda.device(count.device):
        rc = lib.cf_event_window_offsets(count.data_ptr(), pol, int(param), offsets.data_ptr(), int(max_windows),
                                         n_windows.data_ptr(), _lib.stream_ptr(count.device))
    _lib.check(rc, "cf_event_window_offsets")
    return offsets, n_windows


def _single_window(events_dev: torch.Tensor, num_bins, width, height, flavour, mode, **kw) -> torch.Tensor:
    n = events_dev.shape[0]
    offsets = torch.tensor([0, n], dtype=torch.int64, device=events_dev.device)
    return events_to_voxel_grid_batched(events_dev, offsets, num_bins, width, height, flavour=flavour, mode=mode, **kw)[0]


def events_to_voxel_grid(events, num_bins, width, height, is_reverse=False, mode=None):
    """Drop-in for ``utils/event_process.py:15-72`` (NumPy in, NumPy float32 out)."""
    _check_args(events, num_bins, width, height)
    ev = np.ascontiguousarray(events, dtype=np.float64)
    if is_reverse:
        # :33-34 flips the stream; :51-54 then maps EVERY polarity to -1 (sic)
        ev = ev[::-1].copy()
        ev[:, 3] = -1.0
    dev = _device()
    ev_dev = torch.from_numpy(ev).to(dev)
    return _single_window(ev_dev, num_bins, width, height, "numpy", mode).cpu().numpy()


def events_to_voxel_grid_pol(events, num_bins, width, height, mode=None):
    """Drop-in for ``utils/event_process.py:75-123`` -> float32 [nb,2,H,W]."""
    _check_args(events, num_bins, width, height)
    ev_dev = torch.from_numpy(np.ascontiguousarray(events, dtype=np.float64)).to(_device())
    return _single_window(ev_dev, num_bins, width, height, "pol", mode).cpu().numpy()


def events_to_voxel_grid_pytorch(events, num_bins, width, height, mode=None):
    """Drop-in for ``utils/event_process.py:127-190``: result on ``events.device``."""
    _check_args(events, num_bins, width, height)
    with torch.no_grad():
        src = events.device
        ev_dev = events if events.is_cuda else events.to(_device())
        grid = _single_window(ev_dev, num_bins, width, height, "torch", mode)
        return grid if src == grid.device else grid.to(src)


def event_preprocess_batched(grids: torch.Tensor, mode: str = "std", filter_hot_pixel: bool = False,
                             hot_threshold: float | None = None, variant: str = "numpy",
                             out: torch.Tensor | None = None) -> torch.Tensor:
    """``event_preprocess`` on a CUDA batch [B, nb, H, W]; statistics per window."""
    _lib.require_cuda(grids, "grids")
    assert mode in ("std", "maxmin"), "mode must be 'maxmin' or 'std'"
    g = grids.float().contiguous()
    B = g.shape[0]
    cells = g[0].numel()
    nb = g.shape[1]
    thr = 0.0
    if filter_hot_pixel:
        thr = hot_threshold if hot_threshold is not None else (20.0 if variant == "torch" else 25.0) / nb
    if out is None:
        out = torch.empty_like(g)
    lib = _lib.load()
    with torch.cuda.device(g.device):
        ws_bytes = lib.cf_preprocess_workspace_bytes(B, cells)
        ws = _lib.workspace(ws_bytes, g.device)
        rc = lib.cf_voxel_preprocess(g.data_ptr(), out.data_ptr(), B, cells, _PRE[mode], thr, _lib.ptr(ws), ws_bytes,
                                     _lib.stream_ptr(g.device))
    _lib.check(rc, "cf_voxel_preprocess")
    return out


def event_preprocess(event_voxel_grid, mode="std", filter_hot_pixel=False):
    """Drop-in for ``utils/event_process.py:193-216`` (NumPy in/out, 25/nb threshold)."""
    assert mode == "maxmin" or mode == "std"
    g = torch.from_numpy(np.ascontiguousarray(event_voxel_grid, dtype=np.float32)).to(_device())
    return event_preprocess_batched(g[None], mode, filter_hot_pixel, variant="numpy")[0].cpu().numpy()


def event_preprocess_pytorch(event_voxel_grid, mode="std", filter_hot_pixel=False):
    """Drop-in for ``utils/event_process.py:219-239`` (torch in/out, 20/nb threshold).
    Like the reference, an unknown ``mode`` returns the (hot-pixel filtered) input."""
    src = event_voxel_grid.device
    g = event_voxel_grid if event_voxel_grid.is_cuda else event_voxel_grid.to(_device())
    if mode not in ("std", "maxmin"):
        g = g.clone()
        if filter_hot_pixel:
            g[abs(g) > 20.0 / g.shape[0]] = 0
        return g.to(src)
    res = event_preprocess_batched(g[None], mode, filter_hot_pixel, variant="torch")[0]
    return res if src == res.device else res.to(src)
