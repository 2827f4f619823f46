"""NaN-filled output buffers with guard regions, shared by the branch sweeps (test_gpu_corr_branches.py,
test_gpu_warp_branches.py).  An element a kernel skipped stays NaN, and a write outside an output changes a guard."""
import math

import numpy as np
import torch

GUARD = 64           # floats of NaN in front of and behind every output view
NAN_BITS = 0x7FC00000


def guarded(shapes, device, misalign=None):
    """Views of the given shapes inside one NaN-filled float32 buffer, GUARD floats of NaN around each.  Views start
    on 16-byte boundaries, except view ``misalign``, which starts one float later."""
    offs, pos = [], GUARD
    for k, s in enumerate(shapes):
        o = pos + (1 if k == misalign else 0)
        offs.append(o)
        pos = -(-(o + math.prod(s)) // 4) * 4 + GUARD
    buf = torch.full((pos,), float("nan"), dtype=torch.float32, device=device)
    views = [buf[o:o + math.prod(s)].view(s) for o, s in zip(offs, shapes)]
    return buf, views


def assert_written_and_guarded(buf, views, what):
    """Every element of every view written (no NaN left), every float outside the views unchanged."""
    inside = torch.zeros(buf.numel(), dtype=torch.bool, device=buf.device)
    base = buf.data_ptr()
    for k, v in enumerate(views):
        o = (v.data_ptr() - base) // 4
        inside[o:o + v.numel()] = True
        nan = torch.isnan(v)
        if nan.any():
            first = np.unravel_index(int(nan.reshape(-1).nonzero()[0]), tuple(v.shape))
            raise AssertionError(f"{what}: view {k} has {int(nan.sum())} unwritten elements, first at {first}")
    bits = buf.view(torch.int32)[~inside]
    bad = bits != NAN_BITS
    assert not bad.any(), f"{what}: {int(bad.sum())} guard floats overwritten"
