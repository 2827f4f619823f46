#!/usr/bin/env python
"""Generate golden input/output fixtures from the REFERENCE ITSELF.

Run with a checkout of the original project (no test reads it at run time):

    CISTA_REFERENCE=<checkout> PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

The reference is imported read-only from ``$CISTA_REFERENCE``; every array stored
below is either a seeded synthetic input or the output of an unmodified
reference function on that input.  The reference has no tests or golden vectors
of its own (SURVEY.md F3), so these files are what pins the oracle.

Files
-----
voxel.npz   utils/event_process.py   all voxelisers + both preprocess variants
warp.npz    utils/flow_utils.py      forwardWarp / backWarp / FrameWarp, + the
                                     image+codes step of e2v/e2v_model.py:188-191
corr.npz    ERAFT/corr.py, DCEIFlow/core/corr/raft_corr.py   pyramid + lookup
fwl.npz     loss.py                  voxel_warping_flow_loss (FWL metric), both time directions
mvsec.npz   data_readers/MVSEC_utils.py   eventsToVoxel / events_to_voxel_torch / events_to_neg_pos_voxel_torch
                                     (the second voxeliser, temporal bilinear)
trace_eiflow.npz / trace_eraft.npz
            hot-path calls recorded inside DCEIFlowCistaNet / ERAFTCistaNet
            (seeded random-init weights, base_channels=16 to keep the files
            small) on the 3rd recurrent frame of a synthetic 128x160 stream.
trace3_eiflow.npz / trace3_eraft.npz
            three CONSECUTIVE recurrent frames (4th-6th) of the default-size models
            (180x240, base_channels 64): hot-path inputs + reference outputs per frame.
"""
import argparse
import os
import sys
import types

import numpy as np
import torch

REF = os.environ.get("CISTA_REFERENCE", "")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.dont_write_bytecode = True
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

from cistaflow_b200 import synth  # noqa: E402  (host-only helper, no CUDA needed)


def _stub_optional_imports():
    """e2v.e2v_model pulls in matplotlib and omegaconf only for plotting /
    IDNet config (SURVEY.md section 8c); neither is used on the hot path."""
    mpl = types.ModuleType("matplotlib")
    plt = types.ModuleType("matplotlib.pyplot")
    mpl.pyplot = plt
    sys.modules.setdefault("matplotlib", mpl)
    sys.modules.setdefault("matplotlib.pyplot", plt)
    oc = types.ModuleType("omegaconf")

    class OmegaConf:
        @staticmethod
        def create(d):
            return types.SimpleNamespace(**d)
    oc.OmegaConf = OmegaConf
    sys.modules.setdefault("omegaconf", oc)


def save(name, **arrays):
    path = os.path.join(HERE, name)
    arrays = compact(name, arrays)
    np.savez_compressed(path, **arrays)
    print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB, {len(arrays)} arrays")


# ---------------------------------------------------------------- sampling ---
# Every fixture stays below 1 MB.  The correlation, trace and multi-frame trace fixtures therefore keep a fixed sample
# of their large arrays: KEY#values holds the elements at the set bits of KEY#mask (np.packbits of a boolean array of
# shape KEY#shape); tests/conftest.py expands them to zero-filled arrays of the full shape, and the tests compare
# outputs only where the fixture stores them.  A sample is chosen so that the stored outputs depend only on stored
# inputs: a correlation row depends on its query's fmap1 column and all of fmap2, a lookup on its query's rows, a warped
# pixel on the flow there and on the source within MARGIN pixels (|flow| < 10 px in these traces), a warped code channel
# on that channel alone.  Event streams that synth.events() regenerates from a seed are stored as the seed.
MARGIN = 12


def _sparse(out, key, keep):
    a = out.pop(key)
    keep = np.broadcast_to(keep, a.shape)
    out[key + "#shape"] = np.array(a.shape)
    out[key + "#mask"] = np.packbits(keep.ravel())
    out[key + "#values"] = a[keep]


def _queries(rng, b, h, w, frac, extra=()):
    """Sampled correlation queries, bool [b, h, w]."""
    q = rng.random((b, h, w)) < frac
    for idx in extra:
        q[idx] = True
    return q


def _rows(q):
    """Pyramid level [b*h*w, 1, hl, wl]: the rows of the sampled queries."""
    return q.reshape(-1, 1, 1, 1)


def _positions(q):
    """[b, c, h, w] maps (fmap1, lookup outputs): every channel at the sampled queries."""
    return q[:, None]


def _box(shape, r0, r1, c0, c1, channels=None):
    """[b, c, h, w]: rows r0:r1, columns c0:c1 (clipped to the map), channels :channels."""
    keep = np.zeros(shape, bool)
    keep[:, :channels, max(r0, 0):r1, max(c0, 0):c1] = True
    return keep


def _warp_boxes(out, h, w, frame_in, frame_out, flows, codes_in, codes_out, half_flow, channels):
    """Frame warp: outputs in the central box (a third of each side), flow there (+4 px for the x0.5 down-sampling),
    source within MARGIN.  Codes warp (half resolution): outputs in that box halved and shrunk by 2 px, the first
    `channels` channels."""
    r0, r1, c0, c1 = h // 3, 2 * h // 3, w // 3, 2 * w // 3
    _sparse(out, frame_out, _box(out[frame_out].shape, r0, r1, c0, c1))
    _sparse(out, frame_in, _box(out[frame_in].shape, r0 - MARGIN, r1 + MARGIN, c0 - MARGIN, c1 + MARGIN))
    for key in flows:
        _sparse(out, key, _box(out[key].shape, r0 - 4, r1 + 4, c0 - 4, c1 + 4))
    s0, s1, t0, t1 = r0 // 2 + 2, r1 // 2 - 2, c0 // 2 + 2, c1 // 2 - 2
    _sparse(out, codes_out, _box(out[codes_out].shape, s0, s1, t0, t1, channels))
    _sparse(out, codes_in, _box(out[codes_in].shape, s0 - MARGIN, s1 + MARGIN, t0 - MARGIN, t1 + MARGIN, channels))
    if half_flow:
        _sparse(out, half_flow, _box(out[half_flow].shape, s0, s1, t0, t1))


def compact(name, out):
    out = dict(out)
    rng = np.random.default_rng(0)
    if name == "corr.npz":
        q = _queries(rng, 1, 16, 24, 0.25, extra=[(0, 0, 0), (0, 1, 1)])   # the two hand-placed queries
        for l in range(4):
            _sparse(out, f"pyr{l}", _rows(q))
        _sparse(out, "lookup", _positions(q))
        q = _queries(rng, 2, 15, 20, 0.25)
        for l in range(3):
            _sparse(out, f"odd/pyr{l}", _rows(q))
        _sparse(out, "odd/lookup", _positions(q))
    elif name.startswith("trace_"):
        H, W, _, n_lookup, _ = (int(v) for v in out["meta"])
        ev = out.pop("voxel/events")
        out["voxel/seed"] = np.array(synth.seed_for(9, 2))
        assert np.array_equal(synth.events(len(ev), H, W, int(out["voxel/seed"])), ev)
        del out["rec_img0"]                                   # == warp0/in
        cells = rng.random(out["voxel/grid"].shape) < 0.25
        _sparse(out, "voxel/grid", cells)
        _sparse(out, "voxel/normalised", cells)
        q = _queries(rng, *out["corr/fmap1"].shape[:1], *out["corr/fmap1"].shape[2:], 0.2)
        _sparse(out, "corr/fmap1", _positions(q))
        for l in range(4):
            _sparse(out, f"corr/pyr{l}", _rows(q))
        for k in range(n_lookup):
            if f"lookup{k}/out" in out:
                _sparse(out, f"lookup{k}/out", _positions(q))
        _warp_boxes(out, H, W, "warp0/in", "warp0/out", ("warp0/flow", "flow_final"), "warp1/in", "warp1/out",
                    "warp1/flow", channels=4)
    elif name.startswith("trace3_"):
        H, W, _, frames, _, _ = (int(v) for v in out["meta"])
        for f in range(frames):
            n_lookup = int(out[f"f{f}/counts"][0])
            ev_t = out.pop(f"f{f}/ev_t")
            ev = np.stack([ev_t] + [out.pop(f"f{f}/ev_{c}").astype(np.float64) for c in "xyp"], axis=1)
            out[f"f{f}/seed"] = np.array(synth.seed_for(1, 3 + f))
            assert np.array_equal(synth.events(len(ev), H, W, int(out[f"f{f}/seed"])), ev)
            for k in range(n_lookup - 1):                     # only the last lookup's output is stored
                del out[f"f{f}/coords{k}"]
            q = _queries(rng, *out[f"f{f}/fmap1"].shape[:1], *out[f"f{f}/fmap1"].shape[2:], 0.2)
            _sparse(out, f"f{f}/fmap1", _positions(q))
            _sparse(out, f"f{f}/lookup_last", _positions(q))
            _warp_boxes(out, H, W, f"f{f}/warp0_in", f"f{f}/warp0_out", (f"f{f}/flow_final",), f"f{f}/warp1_in",
                        f"f{f}/warp1_out", None, channels=2)
    return out


# ------------------------------------------------------------------ voxel ---
def make_voxel():
    from utils import event_process as ep
    out = {}
    cases = {
        "base": synth.events(3000, 30, 40, 11),
        "dense_hot": synth.events(6000, 12, 16, 12, hot_fraction=0.6, hot_pixels=0.02),
        "single": synth.events(1, 30, 40, 13),
        "two_same_t": np.array([[5.0, 3, 4, 1], [5.0, 7, 2, 0]], np.float64),
        "empty": np.zeros((0, 4), np.float64),
    }
    dims = {"base": (5, 40, 30), "dense_hot": (5, 16, 12), "single": (5, 40, 30),
            "two_same_t": (3, 40, 30), "empty": (5, 40, 30)}
    for name, ev in cases.items():
        nb, w, h = dims[name]
        out[f"{name}/events"] = ev
        out[f"{name}/dims"] = np.array([nb, w, h])
        out[f"{name}/numpy"] = ep.events_to_voxel_grid(ev.copy(), nb, w, h)
        out[f"{name}/torch"] = ep.events_to_voxel_grid_pytorch(torch.from_numpy(ev.copy()), nb, w, h).numpy()
        out[f"{name}/pol"] = ep.events_to_voxel_grid_pol(ev.copy(), nb, w, h)
        g = out[f"{name}/numpy"]
        for mode in ("std", "maxmin"):
            for hot in (False, True):
                key = f"{name}/pre_numpy_{mode}_{int(hot)}"
                out[key] = np.asarray(ep.event_preprocess(g.copy(), mode, hot), np.float32)
                key = f"{name}/pre_torch_{mode}_{int(hot)}"
                out[key] = ep.event_preprocess_pytorch(torch.from_numpy(out[f"{name}/torch"].copy()), mode, hot).numpy()
    save("voxel.npz", **out)


# ------------------------------------------------------------------- warp ---
def make_warp():
    from utils.flow_utils import FrameWarp, backWarp, forwardWarp
    out = {}
    rng = np.random.default_rng(21)
    img = rng.random((2, 3, 18, 22), dtype=np.float32)
    flow = (6.0 * rng.standard_normal((2, 2, 18, 22))).astype(np.float32)
    flow[0, :, 0, 0] = 0.0
    flow[1, :, 3, 4] = (-40.0, 55.0)          # several reflections
    out["img"], out["flow"] = img, flow
    ti, tf = torch.from_numpy(img), torch.from_numpy(flow)
    out["forward"] = forwardWarp(22, 18)(ti, tf).numpy()
    out["backward"] = backWarp(22, 18)(ti, tf).numpy()
    out["zero_flow_forward"] = forwardWarp(22, 18)(ti, torch.zeros_like(tf)).numpy()

    # the per-frame step: e2v/e2v_model.py:188-191
    i1, z1, f1 = synth.warp_inputs(1, 36, 44, 22, code_channels=6)
    fw = FrameWarp("forward")
    ds = torch.nn.functional.interpolate(torch.from_numpy(f1), scale_factor=0.5, mode="bilinear", align_corners=True)
    out["step/img"], out["step/codes"], out["step/flow"] = i1, z1, f1
    out["step/flow_half"] = ds.numpy()
    out["step/img_warped"] = fw.warp_frame(torch.from_numpy(i1), torch.from_numpy(f1)).numpy()
    out["step/codes_warped"] = fw.warp_frame(torch.from_numpy(z1), ds).numpy()
    bw = FrameWarp("backward")
    out["step/codes_warped_backward"] = bw.warp_frame(torch.from_numpy(z1), ds).numpy()

    # the same step from the flow network's 1/8-resolution output: upflow8 (DCEIFlow/utils/sample_utils.py:66-68) +
    # ImagePadder.unpad (utils/image_process.py:103-107, padding on the top/left) + the warps (SURVEY 8f rank 1)
    from DCEIFlow.utils.sample_utils import upflow8
    from utils.image_process import ImagePadder
    padder = ImagePadder((36, 44), min_size=32)
    lr = (0.6 * np.random.default_rng(23).standard_normal((1, 2, 8, 8))).astype(np.float32)     # (36+28)/8 x (44+20)/8
    up = padder.unpad(upflow8(torch.from_numpy(lr)))
    assert tuple(up.shape) == (1, 2, 36, 44) and (padder.pad_height, padder.pad_width) == (28, 20)
    ds8 = torch.nn.functional.interpolate(up, scale_factor=0.5, mode="bilinear", align_corners=True)
    out["up8/flow_lr"], out["up8/pad"] = lr, np.array([padder.pad_height, padder.pad_width])
    out["up8/flow_final"] = up.numpy().copy()
    out["up8/img_warped"] = fw.warp_frame(torch.from_numpy(i1), up).numpy()
    out["up8/codes_warped"] = fw.warp_frame(torch.from_numpy(z1), ds8).numpy()
    save("warp.npz", **out)


# -------------------------------------------------------------------- fwl ---
def make_fwl():
    """loss.voxel_warping_flow_loss (FWL metric).  loss.py imports plotting / perceptual-metric packages
    that are absent here and unused by this function: they are stubbed with attribute-less modules."""
    class _Any(types.ModuleType):
        def __getattr__(self, k):
            if k.startswith("__"):
                raise AttributeError(k)
            return object
    for name in ("pytorch_msssim", "lpips", "skimage", "skimage.metrics"):
        sys.modules.setdefault(name, _Any(name))
    import loss as ref_loss
    rng = np.random.default_rng(61)
    ev = [synth.events(4000, 36, 44, 70 + b) for b in range(2)]
    from utils import event_process as ep
    voxel = np.stack([ep.events_to_voxel_grid(e.copy(), 5, 44, 36) for e in ev]).astype(np.float32)
    disp = (3.0 * rng.standard_normal((2, 2, 36, 44))).astype(np.float32)
    disp[0, :, :3, :3] = 40.0          # samples far outside the image: zeros padding
    out = {"voxel": voxel, "disp": disp}
    for rev in (False, True):
        loss, extra = ref_loss.voxel_warping_flow_loss(torch.from_numpy(voxel), torch.from_numpy(disp), output_images=True,
                                                       reverse_time=rev)
        out[f"loss_{int(rev)}"] = np.float32(loss.item())
        out[f"warped_{int(rev)}"] = extra["voxel_grid_warped"].numpy()
    zero = ref_loss.voxel_warping_flow_loss(torch.from_numpy(voxel), torch.zeros(2, 2, 36, 44))
    out["loss_zero_flow"] = np.float32(zero.item())
    save("fwl.npz", **out)


# ------------------------------------------------------------------ mvsec ---
def make_mvsec():
    """The second voxeliser (data_readers/MVSEC_utils.py:253-303, 306-343, 384-403).  Its index_put_(accumulate=True)
    is sequential on the CPU below 32768 elements (or with one thread): the fixtures stay below that size and pin
    the thread count, so the outputs are deterministic."""
    from data_readers import MVSEC_utils as mu
    torch.set_num_threads(1)
    out = {}
    cases = {
        "base": (3000, 30, 40, 21, "pm1"),        # polarities -1 / +1
        "binary": (3000, 30, 40, 22, "01"),       # polarities 0 / 1 as stored by the MVSEC reader: 0 contributes nothing
        "dense": (6000, 12, 16, 23, "pm1"),
        "two": (2, 30, 40, 24, "pm1"),
    }
    for name, (n, h, w, seed, pol) in cases.items():
        ev = synth.events(n, h, w, seed)                      # rows (t, x, y, p in {0,1})
        p = ev[:, 3].copy() if pol == "01" else np.where(ev[:, 3] > 0, 1.0, -1.0)
        xytp = np.stack([ev[:, 1], ev[:, 2], ev[:, 0], p], axis=1)       # MVSEC row order (x, y, t, p)
        out[f"{name}/events_xytp"] = xytp
        out[f"{name}/dims"] = np.array([5, h, w])
        out[f"{name}/voxel"] = mu.eventsToVoxel(xytp.copy(), num_bins=5, height=h, width=w, event_polarity=False)
        out[f"{name}/voxel_pol"] = mu.eventsToVoxel(xytp.copy(), num_bins=5, height=h, width=w, event_polarity=True)
        xs, ys, ts, ps = mu.eventsToXYTP(xytp.copy(), process=True)
        out[f"{name}/direct"] = mu.events_to_voxel_torch(xs, ys, ts, ps, 5, sensor_size=(h, w)).numpy()
        # temporal_bilinear=False (MVSEC_utils.py:292-300): bin bi takes the events in [ts[0] + dt*bi, ts[0] + dt*(bi+1)) with
        # dt the WHOLE window (sic), found by the reference's own binary search
        out[f"{name}/naive"] = mu.events_to_voxel_torch(torch.from_numpy(xs), torch.from_numpy(ys), torch.from_numpy(ts),
                                                        torch.from_numpy(ps), 5, sensor_size=(h, w), temporal_bilinear=False).numpy()
    save("mvsec.npz", **out)


# ------------------------------------------------------------------- corr ---
def make_corr():
    from ERAFT.corr import CorrBlock as ECorr
    from DCEIFlow.core.corr.raft_corr import CorrBlock as DCorr
    out = {}
    rng = np.random.default_rng(31)
    h, w, d = 16, 24, 64
    f1 = rng.standard_normal((1, d, h, w), dtype=np.float32)
    f2 = rng.standard_normal((1, d, h, w), dtype=np.float32)
    ys, xs = np.meshgrid(np.arange(h, dtype=np.float32), np.arange(w, dtype=np.float32), indexing="ij")
    coords = (np.stack([xs, ys])[None] + 3.0 * rng.standard_normal((1, 2, h, w))).astype(np.float32)
    coords[0, :, 0, 0] = (-30.0, 50.0)         # far outside: all-zero window
    coords[0, :, 1, 1] = (w - 1.0, h - 1.0)    # exactly on the corner
    out["fmap1"], out["fmap2"], out["coords"] = f1, f2, coords
    e = ECorr(torch.from_numpy(f1), torch.from_numpy(f2), num_levels=4, radius=4)
    dblk = DCorr(torch.from_numpy(f1.copy()), torch.from_numpy(f2.copy()), num_levels=4, radius=4)
    for l in range(4):
        out[f"pyr{l}"] = e.corr_pyramid[l].numpy()
        assert torch.equal(e.corr_pyramid[l], dblk.corr_pyramid[l]), "ERAFT/DCEIFlow CorrBlock differ"
    out["lookup"] = e(torch.from_numpy(coords)).numpy()
    assert torch.equal(e(torch.from_numpy(coords)), dblk(torch.from_numpy(coords)))
    # odd feature-map size: avg_pool2d floors (15x20 -> 7x10 -> 3x5 -> 1x2)
    h2, w2 = 15, 20
    g1 = rng.standard_normal((2, 32, h2, w2), dtype=np.float32)
    g2 = rng.standard_normal((2, 32, h2, w2), dtype=np.float32)
    ys, xs = np.meshgrid(np.arange(h2, dtype=np.float32), np.arange(w2, dtype=np.float32), indexing="ij")
    c2 = (np.stack([xs, ys])[None] + 2.0 * rng.standard_normal((2, 2, h2, w2))).astype(np.float32)
    e2 = ECorr(torch.from_numpy(g1), torch.from_numpy(g2), num_levels=3, radius=3)
    out["odd/fmap1"], out["odd/fmap2"], out["odd/coords"] = g1, g2, c2
    for l in range(3):
        out[f"odd/pyr{l}"] = e2.corr_pyramid[l].numpy()
    out["odd/lookup"] = e2(torch.from_numpy(c2)).numpy()
    save("corr.npz", **out)


# ------------------------------------------------------------------ trace ---
def make_trace(model_mode: str, fname: str):
    """Record the inputs/outputs of every hot-path call made by the reference
    model on the 3rd recurrent frame."""
    _stub_optional_imports()
    from utils.configs import set_configs
    from utils import event_process as ep
    import e2v.e2v_model as em
    import utils.flow_utils as fu

    H, W, NEV = 128, 160, 9000
    parser = argparse.ArgumentParser()
    set_configs(parser)
    cfgs = parser.parse_args(["--image_dim", str(H), str(W), "--model_mode", model_mode, "--base_channels", "16"])
    torch.manual_seed(0)
    if model_mode == "cista-eiflow":
        model = em.DCEIFlowCistaNet(cfgs)
        import DCEIFlow.DCEIFlow as host
    else:
        model = em.ERAFTCistaNet(cfgs)
        import ERAFT.eraft as host
    model.eval()

    rec = {"on": False, "n_lookup": 0, "n_warp": 0}
    out = {}
    RefCorr = host.CorrBlock

    class TapCorr(RefCorr):
        def __init__(self, fmap1, fmap2, num_levels=4, radius=4):
            super().__init__(fmap1.clone(), fmap2.clone(), num_levels=num_levels, radius=radius)
            if rec["on"]:
                out["corr/fmap1"], out["corr/fmap2"] = fmap1.numpy().copy(), fmap2.numpy().copy()
                for l, p in enumerate(self.corr_pyramid):
                    out[f"corr/pyr{l}"] = p.numpy().copy()

        def __call__(self, coords):
            res = super().__call__(coords)
            if rec["on"]:
                k = rec["n_lookup"]
                out[f"lookup{k}/coords"] = coords.numpy().copy()
                out[f"lookup{k}/out"] = res.numpy().copy()
                rec["n_lookup"] += 1
            return res

    host.CorrBlock = TapCorr
    ref_warp_frame = fu.FrameWarp.warp_frame

    def tap_warp(self, I, flow):
        res = ref_warp_frame(self, I, flow)
        if rec["on"]:
            k = rec["n_warp"]
            out[f"warp{k}/in"], out[f"warp{k}/flow"] = I.numpy().copy(), flow.numpy().copy()
            out[f"warp{k}/out"] = res.numpy().copy()
            rec["n_warp"] += 1
        return res

    fu.FrameWarp.warp_frame = tap_warp
    try:
        states, prev, vox_old = None, torch.zeros(1, 1, H, W), torch.zeros(1, 5, H, W)
        with torch.no_grad():
            for frame in range(3):
                ev = synth.events(NEV, H, W, synth.seed_for(9, frame))
                rec["on"] = frame == 2
                grid = ep.events_to_voxel_grid(ev.copy(), 5, W, H)
                vox = np.asarray(ep.event_preprocess(grid.copy(), "std", True), np.float32)
                if rec["on"]:
                    out["voxel/events"], out["voxel/grid"], out["voxel/normalised"] = ev, grid, vox
                vox_t = torch.from_numpy(vox)[None]
                if model_mode == "cista-eiflow":
                    batch = {"event_voxel": vox_t, "rec_img0": prev}
                else:
                    batch = {"event_voxel": vox_t, "event_voxel_old": vox_old, "rec_img0": prev}
                pred, flow_out, states = model(batch, states)
                if rec["on"]:
                    out["flow_final"] = flow_out["flow_final"].numpy().copy()
                    out["rec_img0"] = prev.numpy().copy()
                prev, vox_old = pred.clone(), vox_t
    finally:
        host.CorrBlock = RefCorr
        fu.FrameWarp.warp_frame = ref_warp_frame
    out["meta"] = np.array([H, W, NEV, rec["n_lookup"], rec["n_warp"]])
    # keep the file small: only every other lookup output, pyramid levels >= 1 are
    # re-derivable from level 0 but cheap (1/3 of it) so they stay.
    for k in range(rec["n_lookup"]):
        if k % 2 == 1 and k != rec["n_lookup"] - 1:
            del out[f"lookup{k}/out"]
    save(fname, **out)


def make_trace_multi(model_mode: str, fname: str, first: int = 3, frames: int = 3):
    """Consecutive recurrent frames `first .. first+frames-1` (the drivers skip the first 3 too) of the reference model
    at its DEFAULT size (180x240, base_channels 64): the hot-path INPUTS of every frame -- events, the feature maps the
    encoder produced (first 32 of 256 channels: the contraction is linear in channels and D = 32 is a valid CorrBlock
    call), every lookup's coords, the previous reconstruction, the final flow, the first 8 of 128 code channels -- and
    the reference's own OUTPUTS for the last lookup (recomputed by the reference CorrBlock on the stored channel
    subset; every 4th output channel kept), the warped frame and the warped code channels.  Events are stored as
    (t f64, x u16, y u16, p u8); the voxel grid is checked against the oracle (pinned bit-exact by voxel.npz).  The GPU tests replay frame by frame."""
    _stub_optional_imports()
    from utils.configs import set_configs
    from utils import event_process as ep
    import e2v.e2v_model as em
    import utils.flow_utils as fu

    H, W, NEV, DSUB, CSUB = 180, 240, 15000, 32, 8
    parser = argparse.ArgumentParser()
    set_configs(parser)
    cfgs = parser.parse_args(["--image_dim", str(H), str(W), "--model_mode", model_mode])
    torch.manual_seed(0)
    if model_mode == "cista-eiflow":
        model = em.DCEIFlowCistaNet(cfgs)
        import DCEIFlow.DCEIFlow as host
    else:
        model = em.ERAFTCistaNet(cfgs)
        import ERAFT.eraft as host
    model.eval()
    rec = {"frame": -1, "n_lookup": 0, "n_warp": 0}
    out = {}
    RefCorr = host.CorrBlock

    class TapCorr(RefCorr):
        def __init__(self, fmap1, fmap2, num_levels=4, radius=4):
            super().__init__(fmap1, fmap2, num_levels=num_levels, radius=radius)
            if rec["frame"] >= 0:
                f = rec["frame"]
                out[f"f{f}/fmap1"], out[f"f{f}/fmap2"] = fmap1[:, :DSUB].numpy().copy(), fmap2[:, :DSUB].numpy().copy()
                self.sub = RefCorr(fmap1[:, :DSUB].contiguous(), fmap2[:, :DSUB].contiguous(), num_levels=num_levels, radius=radius)

        def __call__(self, coords):
            res = super().__call__(coords)
            if rec["frame"] >= 0:
                f, k = rec["frame"], rec["n_lookup"]
                out[f"f{f}/coords{k}"] = coords.numpy().copy()
                out[f"f{f}/lookup_last"] = self.sub(coords)[:, ::4].numpy().copy()   # overwritten until the last call
                rec["n_lookup"] += 1
            return res

    host.CorrBlock = TapCorr
    ref_warp_frame = fu.FrameWarp.warp_frame

    def tap_warp(self, I, flow):
        res = ref_warp_frame(self, I, flow)
        if rec["frame"] >= 0:
            f, k = rec["frame"], rec["n_warp"]
            sub = slice(0, CSUB) if I.shape[1] > CSUB else slice(None)
            out[f"f{f}/warp{k}_in"], out[f"f{f}/warp{k}_out"] = I[:, sub].numpy().copy(), res[:, sub].numpy().copy()
            rec["n_warp"] += 1
        return res

    fu.FrameWarp.warp_frame = tap_warp
    try:
        states, prev, vox_old = None, torch.zeros(1, 1, H, W), torch.zeros(1, 5, H, W)
        with torch.no_grad():
            for frame in range(first + frames):
                ev = synth.events(NEV, H, W, synth.seed_for(1, frame))
                f = frame - first
                rec["frame"], rec["n_lookup"], rec["n_warp"] = (f if f >= 0 else -1), 0, 0
                grid = ep.events_to_voxel_grid(ev.copy(), 5, W, H)
                vox = np.asarray(ep.event_preprocess(grid.copy(), "std", True), np.float32)
                if f >= 0:
                    out[f"f{f}/ev_t"], out[f"f{f}/ev_x"] = ev[:, 0].copy(), ev[:, 1].astype(np.uint16)
                    out[f"f{f}/ev_y"], out[f"f{f}/ev_p"] = ev[:, 2].astype(np.uint16), ev[:, 3].astype(np.uint8)
                vox_t = torch.from_numpy(vox)[None]
                if model_mode == "cista-eiflow":
                    batch = {"event_voxel": vox_t, "rec_img0": prev}
                else:
                    batch = {"event_voxel": vox_t, "event_voxel_old": vox_old, "rec_img0": prev}
                pred, flow_out, states = model(batch, states)
                if f >= 0:
                    out[f"f{f}/flow_final"] = flow_out["flow_final"].numpy().copy()
                    out[f"f{f}/counts"] = np.array([rec["n_lookup"], rec["n_warp"]])
                prev, vox_old = pred.clone(), vox_t
    finally:
        host.CorrBlock = RefCorr
        fu.FrameWarp.warp_frame = ref_warp_frame
    out["meta"] = np.array([H, W, NEV, frames, DSUB, CSUB])
    save(fname, **out)


if __name__ == "__main__":
    assert os.path.isdir(REF), f"reference checkout not found at {REF}"
    only = sys.argv[1:]
    if not only or "voxel" in only:
        make_voxel()
    if not only or "warp" in only:
        make_warp()
    if not only or "fwl" in only:
        make_fwl()
    if not only or "mvsec" in only:
        make_mvsec()
    if not only or "corr" in only:
        make_corr()
    if not only or "trace" in only:
        make_trace("cista-eiflow", "trace_eiflow.npz")
        make_trace("cista-eraft", "trace_eraft.npz")
    if not only or "trace3" in only:
        make_trace_multi("cista-eiflow", "trace3_eiflow.npz")
        make_trace_multi("cista-eraft", "trace3_eraft.npz")
