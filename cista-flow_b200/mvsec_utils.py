"""The second voxeliser: B200 mirror of ``data_readers/MVSEC_utils.py`` (253-303, 306-343, 384-403; the same code
lives in ``DCEIFlow/utils/event_uitls.py``), SURVEY.md section 8f rank 4.

Same names and signatures:

  events_to_voxel_torch(xs, ys, ts, ps, B, device=None, sensor_size=(180, 240), temporal_bilinear=True) -> [B,H,W]
  events_to_neg_pos_voxel_torch(...)                                                   -> ([B,H,W], [B,H,W])
  eventsToVoxelTorch(events[x,y,t,p], num_bins=5, height=None, width=None, event_polarity=False, ...)
  eventsToVoxel(...)                                                                   -> numpy

It differs from ``events_to_voxel_grid`` in details that change bits: rows are (x, y, t, p); the time axis is
normalised as ((t - t0) / dT) * (B - 1) (divide first); the polarity is used AS GIVEN (the MVSEC reader stores
0 / 1, so negative events contribute nothing, MVSEC_utils.py:355,364); the weights are fp64 products cast to fp32 and
summed in fp32 by one ``index_put_(accumulate=True)`` per bin.  All of that is ``CF_FLAVOUR_MVSEC`` of
``cf_voxel_bin``; this module only arranges the arguments.  The reference's ``temporal_bilinear=False`` branch is not
mirrored: no caller uses it, and its bin edges (``tend = tstart + dt``, the whole duration) put every event in bin 0.

``mode`` is that of ``events_to_voxel_grid_batched``: None means 'deterministic' under
``torch.use_deterministic_algorithms(True)`` and ``event_process.DEFAULT_MODE`` otherwise.

Results come back where the inputs lived (CPU tensors for CPU / NumPy inputs, like the reference) unless ``device``
says otherwise.  Deliberate differences: out-of-range coordinates are dropped (the reference raises IndexError); a
window whose events all share one time stamp uses dT = 1 (the reference divides by zero and returns NaN).
"""
from __future__ import annotations

import numpy as np
import torch

from . import event_process


def _as_tensor(a):
    return torch.from_numpy(np.ascontiguousarray(a)) if isinstance(a, np.ndarray) else a


def _binary_search(t, l, r, x):
    """binary_search_torch_tensor (MVSEC_utils.py:184-201, side='left') on a host tensor."""
    while l <= r:
        mid = l + (r - l) // 2
        midval = t[mid]
        if midval == x:
            return mid
        if midval < x:
            l = mid + 1
        else:
            r = mid - 1
    return l


def _voxel(xs, ys, ts, weights, B, sensor_size, mode):
    """[B,H,W] float32 on the current CUDA device from per-event columns (any device, any real dtype)."""
    dev = event_process._device()
    n = xs.shape[0]
    height, width = int(sensor_size[0]), int(sensor_size[1])
    if n == 0:
        return torch.zeros((B, height, width), dtype=torch.float32, device=dev)
    rows = torch.stack([ts.to(dev, torch.float64), xs.to(dev, torch.float64), ys.to(dev, torch.float64),
                        weights.to(dev, torch.float64)], dim=1)
    offsets = torch.tensor([0, n], dtype=torch.int64, device=dev)
    return event_process.events_to_voxel_grid_batched(rows, offsets, B, width, height, flavour="mvsec", mode=mode)[0]


def events_to_voxel_torch(xs, ys, ts, ps, B, device=None, sensor_size=(180, 240), temporal_bilinear=True, mode=None):
    """MVSEC_utils.py:253-303 (temporal bilinear): voxel[b, y, x] = sum_e ps_e * max(0, 1 - |t*_e - b|)."""
    xs, ys, ts, ps = (_as_tensor(a) for a in (xs, ys, ts, ps))
    assert len(xs) == len(ys) and len(ys) == len(ts) and len(ts) == len(ps)
    where = torch.device(device) if device is not None else xs.device
    if not temporal_bilinear:
        # MVSEC_utils.py:292-300: bin bi takes the events with ts in [ts[0] + dt*bi, ts[0] + dt*(bi+1)), dt the WHOLE
        # window (sic), their polarities accumulated per pixel.  The index range comes from the reference's own binary
        # search (host side, on the time column); each bin is one single-bin voxelisation on the GPU.
        n = len(ts)
        if n == 0:
            return torch.zeros((int(B), int(sensor_size[0]), int(sensor_size[1])), dtype=torch.float32, device=where)
        tc = ts.detach().cpu()
        dt = tc[-1] - tc[0]
        bins = []
        for bi in range(int(B)):
            tstart = tc[0] + dt * bi
            beg, end = _binary_search(tc, 0, n - 1, tstart), _binary_search(tc, 0, n - 1, tstart + dt)
            bins.append(_voxel(xs[beg:end], ys[beg:end], ts[beg:end], ps[beg:end], 1, sensor_size, mode)[0])
        return torch.stack(bins).to(where)
    return _voxel(xs, ys, ts, ps, int(B), sensor_size, mode).to(where)


def events_to_neg_pos_voxel_torch(xs, ys, ts, ps, B, device=None, sensor_size=(180, 240), temporal_bilinear=True, mode=None):
    """MVSEC_utils.py:306-343: positive (p > 0) and non-positive events in separate grids, unit weights."""
    xs, ys, ts, ps = (_as_tensor(a) for a in (xs, ys, ts, ps))
    pos = (ps > 0).to(torch.float64)
    neg = (ps <= 0).to(torch.float64)
    return (events_to_voxel_torch(xs, ys, ts, pos, B, device, sensor_size, temporal_bilinear, mode),
            events_to_voxel_torch(xs, ys, ts, neg, B, device, sensor_size, temporal_bilinear, mode))


def eventsToXYTP(events, process=False):
    """MVSEC_utils.py:348-364: rows (x, y, t, p) -> int32 x, y, p and (optionally [0,1]-normalised) fp64 t."""
    event_x = events[:, 0].astype(np.int32)
    event_y = events[:, 1].astype(np.int32)
    event_pols = events[:, 3].astype(np.int32)
    event_timestamps = events[:, 2]
    if process:
        first_stamp, last_stamp = event_timestamps[0], event_timestamps[-1]
        event_timestamps = (event_timestamps - first_stamp) / (last_stamp - first_stamp)
    return event_x, event_y, event_timestamps, event_pols


def eventsToVoxelTorch(events, num_bins=5, height=None, width=None, event_polarity=False, temporal_bilinear=True, mode=None):
    """MVSEC_utils.py:388-403: [num_bins,H,W], or [2*num_bins,H,W] (positive grids, then negative) with event_polarity."""
    xs, ys, ts, ps = eventsToXYTP(events, process=True)
    if height is None or width is None:
        width = xs.max() + 1
        height = ys.max() + 1
    if not event_polarity:
        return events_to_voxel_torch(xs, ys, ts, ps, num_bins, sensor_size=(height, width),
                                     temporal_bilinear=temporal_bilinear, mode=mode)
    pos, neg = events_to_neg_pos_voxel_torch(xs, ys, ts, ps, num_bins, sensor_size=(height, width),
                                             temporal_bilinear=temporal_bilinear, mode=mode)
    return torch.cat([pos, neg], 0)


def eventsToVoxel(events, num_bins=5, height=None, width=None, event_polarity=False, temporal_bilinear=True, mode=None):
    """MVSEC_utils.py:384-385 (call site data_readers/MVSEC.py:178)."""
    return eventsToVoxelTorch(events, num_bins, height, width, event_polarity, temporal_bilinear, mode).numpy()
