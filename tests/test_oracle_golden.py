"""Pins the CPU oracle against outputs of the reference itself.

The fixtures under tests/golden/ were produced by importing /root/reference in
the build container (tests/golden/make_golden.py).  Both layers of the oracle
are checked: ``ref_port`` (same library calls as the reference -> bit-exact)
and ``explicit`` (from-scratch NumPy/C -> ~1 ulp, bit-exact for the sequential
voxel accumulation).  Runs on CPU.
"""
import numpy as np
import pytest
import torch

from cistaflow_b200 import synth
from oracle import explicit, ref_port

VOXEL_CASES = ["base", "dense_hot", "single", "two_same_t", "empty"]


@pytest.mark.parametrize("case", VOXEL_CASES)
def test_voxel_ref_port_bit_exact(golden, case):
    g = golden("voxel")
    ev = g[f"{case}/events"]
    nb, w, h = (int(v) for v in g[f"{case}/dims"])
    assert np.array_equal(ref_port.voxel_grid_numpy(ev, nb, w, h), g[f"{case}/numpy"])
    assert np.array_equal(ref_port.voxel_grid_torch(torch.from_numpy(ev), nb, w, h).numpy(), g[f"{case}/torch"])
    assert np.array_equal(ref_port.voxel_grid_pol_numpy(ev, nb, w, h), g[f"{case}/pol"])
    assert ev.dtype == np.float64  # inputs are not mutated (the reference rewrites them in place)


@pytest.mark.parametrize("case", VOXEL_CASES)
def test_voxel_sequential_c_oracle_bit_exact(golden, case):
    """The plain-C event-order accumulation IS what np.add.at / index_add_ do."""
    g = golden("voxel")
    ev = g[f"{case}/events"]
    nb, w, h = (int(v) for v in g[f"{case}/dims"])
    for flavour, key in ((explicit.FLAVOUR_TORCH, "torch"), (explicit.FLAVOUR_NUMPY, "numpy"), (explicit.FLAVOUR_POL, "pol")):
        got = explicit.voxel_grid_sequential(ev, nb, w, h, flavour)
        ref = g[f"{case}/{key}"]
        assert got.shape == ref.shape
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), f"{case}/{key} differs bitwise"


def test_voxel_flavours_differ_by_at_most_an_ulp_or_so(golden):
    g = golden("voxel")
    assert not np.array_equal(g["base/numpy"], g["base/torch"])  # they are NOT the same function
    assert np.abs(g["base/numpy"] - g["base/torch"]).max() < 2e-6


@pytest.mark.parametrize("case", VOXEL_CASES)
@pytest.mark.parametrize("mode", ["std", "maxmin"])
@pytest.mark.parametrize("hot", [False, True])
def test_preprocess(golden, case, mode, hot):
    g = golden("voxel")
    nb = int(g[f"{case}/dims"][0])
    ref_np = g[f"{case}/pre_numpy_{mode}_{int(hot)}"]
    ref_t = g[f"{case}/pre_torch_{mode}_{int(hot)}"]
    got_np = ref_port.preprocess_numpy(g[f"{case}/numpy"], mode, hot)
    got_t = ref_port.preprocess_torch(torch.from_numpy(g[f"{case}/torch"]), mode, hot).numpy()
    assert got_np.dtype == np.float32
    np.testing.assert_allclose(got_np, ref_np, rtol=0, atol=1e-6)
    assert np.array_equal(got_t, ref_t, equal_nan=True)
    # explicit restatement with the threshold spelled out (25/nb vs 20/nb)
    ex_np = explicit.preprocess(g[f"{case}/numpy"], mode, 25.0 / nb if hot else 0.0)
    ex_t = explicit.preprocess(g[f"{case}/torch"], mode, 20.0 / nb if hot else 0.0)
    np.testing.assert_allclose(ex_np, ref_np, rtol=1e-5, atol=1e-5)
    if np.isfinite(ref_t).all():
        np.testing.assert_allclose(ex_t, ref_t, rtol=1e-5, atol=1e-5)


def test_warp_ref_port_and_explicit(golden):
    g = golden("warp")
    img, flow = torch.from_numpy(g["img"]), torch.from_numpy(g["flow"])
    assert np.array_equal(ref_port.warp(img, flow, "forward").numpy(), g["forward"])
    assert np.array_equal(ref_port.warp(img, flow, "backward").numpy(), g["backward"])
    np.testing.assert_allclose(explicit.warp(g["img"], g["flow"], -1.0), g["forward"], rtol=0, atol=2e-6)
    np.testing.assert_allclose(explicit.warp(g["img"], g["flow"], +1.0), g["backward"], rtol=0, atol=2e-6)
    # SURVEY F6: zero flow is NOT the identity under the reference's normalisation
    zero = explicit.warp(g["img"], np.zeros_like(g["flow"]), -1.0)
    np.testing.assert_allclose(zero, g["zero_flow_forward"], rtol=0, atol=2e-6)
    assert np.abs(zero - g["img"]).max() > 1e-2


def test_warp_frame_and_codes_step(golden):
    g = golden("warp")
    img, codes, flow = (torch.from_numpy(g[f"step/{k}"]) for k in ("img", "codes", "flow"))
    wi, wz = ref_port.warp_frame_and_codes(img, codes, flow, "forward")
    assert np.array_equal(wi.numpy(), g["step/img_warped"])
    assert np.array_equal(wz.numpy(), g["step/codes_warped"])
    half = explicit.downsample_flow(g["step/flow"])
    np.testing.assert_allclose(half, g["step/flow_half"], rtol=0, atol=2e-6)
    np.testing.assert_allclose(explicit.warp(g["step/codes"], half, -1.0), g["step/codes_warped"], rtol=0, atol=1e-5)
    np.testing.assert_allclose(explicit.warp(g["step/codes"], half, +1.0), g["step/codes_warped_backward"], rtol=0, atol=1e-5)


@pytest.mark.parametrize("prefix,levels,radius", [("", 4, 4), ("odd/", 3, 3)])
def test_corr_pyramid_and_lookup(golden, prefix, levels, radius):
    g = golden("corr")
    f1, f2, coords = g[prefix + "fmap1"], g[prefix + "fmap2"], g[prefix + "coords"]
    pyr = ref_port.corr_pyramid(torch.from_numpy(f1), torch.from_numpy(f2), levels)
    for l in range(levels):
        assert np.array_equal(*g.pick(f"{prefix}pyr{l}", pyr[l].numpy()))
    out = ref_port.corr_lookup(pyr, torch.from_numpy(coords), radius)
    assert np.array_equal(*g.pick(prefix + "lookup", out.numpy()))
    # explicit: fp64 contraction rounded once, explicit pooling + transposed window
    ex = explicit.corr_pyramid(f1, f2, levels)
    for l in range(levels):
        assert ex[l].shape == g[f"{prefix}pyr{l}"].shape
        np.testing.assert_allclose(*g.pick(f"{prefix}pyr{l}", ex[l]), rtol=0, atol=2e-5)
    # (a sampled query's lookup reads only its own, stored, pyramid rows)
    ex_out = explicit.corr_lookup([g[f"{prefix}pyr{l}"] for l in range(levels)], coords, radius)
    np.testing.assert_allclose(*g.pick(prefix + "lookup", ex_out), rtol=0, atol=2e-5)


def test_lookup_window_is_transposed(golden):
    """SURVEY F7: channel i*(2r+1)+j moves i along X.  Swapping the roles must NOT match."""
    g = golden("corr")
    pyr = [g[f"pyr{l}"] for l in range(4)]
    coords = g["coords"]
    good = explicit.corr_lookup(pyr, coords, 4)
    k = 9
    swapped = good.reshape(1, 4, k, k, 16, 24).transpose(0, 1, 3, 2, 4, 5).reshape(good.shape)
    assert np.abs(np.subtract(*g.pick("lookup", good))).max() < 2e-5
    assert np.abs(np.subtract(*g.pick("lookup", swapped))).max() > 0.1


@pytest.mark.parametrize("trace", ["trace_eiflow", "trace_eraft"])
def test_model_trace_replay_through_oracle(golden, trace):
    """Hot-path calls recorded inside the reference models replay through the oracle."""
    g = golden(trace)
    H, W, nev, n_lookup, n_warp = (int(v) for v in g["meta"])
    grid = ref_port.voxel_grid_numpy(synth.events(nev, H, W, int(g["voxel/seed"])), 5, W, H)
    assert np.array_equal(*g.pick("voxel/grid", grid))
    np.testing.assert_allclose(*g.pick("voxel/normalised", ref_port.preprocess_numpy(grid, "std", True)), rtol=0, atol=1e-6)
    pyr = ref_port.corr_pyramid(torch.from_numpy(g["corr/fmap1"]), torch.from_numpy(g["corr/fmap2"]), 4)
    for l in range(4):
        assert np.array_equal(*g.pick(f"corr/pyr{l}", pyr[l].numpy()))
    for k in range(n_lookup):
        if f"lookup{k}/out" in g:
            out = ref_port.corr_lookup(pyr, torch.from_numpy(g[f"lookup{k}/coords"]), 4)
            assert np.array_equal(*g.pick(f"lookup{k}/out", out.numpy()))
    assert n_warp == 2
    for k in range(n_warp):
        out = ref_port.warp(torch.from_numpy(g[f"warp{k}/in"]), torch.from_numpy(g[f"warp{k}/flow"]), "forward")
        assert np.array_equal(*g.pick(f"warp{k}/out", out.numpy()))
    # the codes were warped with the x0.5 down-sampled flow (e2v/e2v_model.py:190)
    half = ref_port.downsample_flow(torch.from_numpy(g["flow_final"]))
    assert np.array_equal(*g.pick("warp1/flow", half.numpy()))


MVSEC_CASES = ["base", "binary", "dense", "two"]


@pytest.mark.parametrize("case", MVSEC_CASES)
def test_mvsec_voxeliser_ref_port_bit_exact(golden, case):
    """The second voxeliser (data_readers/MVSEC_utils.py eventsToVoxel): the port reproduces the reference's own
    outputs bit for bit (sequential index_put_: one thread, < 32768 events)."""
    import torch
    g = golden("mvsec")
    ev = g[f"{case}/events_xytp"]
    nb, h, w = (int(v) for v in g[f"{case}/dims"])
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        got = ref_port.mvsec_events_to_voxel(ev, nb, h, w, False)
        got_pol = ref_port.mvsec_events_to_voxel(ev, nb, h, w, True)
    finally:
        torch.set_num_threads(threads)
    assert got.dtype == np.float32 and got.shape == (nb, h, w) and got_pol.shape == (2 * nb, h, w)
    assert np.array_equal(got.view(np.uint32), g[f"{case}/voxel"].view(np.uint32))
    assert np.array_equal(got_pol.view(np.uint32), g[f"{case}/voxel_pol"].view(np.uint32))
    assert np.array_equal(g[f"{case}/direct"], g[f"{case}/voxel"])
    xs_, ys_, ps_ = (torch.from_numpy(ev[:, k].astype(np.int32)) for k in (0, 1, 3))
    ts_ = torch.from_numpy((ev[:, 2] - ev[0, 2]) / (ev[-1, 2] - ev[0, 2]))
    naive = ref_port.mvsec_voxel_naive_torch(xs_, ys_, ts_, ps_, nb, h, w).numpy()
    assert np.array_equal(naive, g[f"{case}/naive"])
    if case == "binary":   # 0 / 1 polarities: negative events contribute nothing (MVSEC_utils.py:355,364)
        assert (g[f"{case}/voxel"] >= 0).all()


def test_fwl_ref_port_bit_exact(golden):
    """loss.voxel_warping_flow_loss (FWL metric): the port reproduces the reference's warped channels and
    variance bit for bit, both time directions, and its zero-flow denominator."""
    g = golden("fwl")
    voxel, disp = torch.from_numpy(g["voxel"]), torch.from_numpy(g["disp"])
    for rev in (False, True):
        var, summed, warped = ref_port.voxel_flow_warp(voxel, disp, reverse_time=rev)
        assert np.array_equal(warped.numpy(), g[f"warped_{int(rev)}"])
        assert np.float32(var.item()) == g[f"loss_{int(rev)}"]
    var0, _, _ = ref_port.voxel_flow_warp(voxel, torch.zeros_like(disp))
    assert np.float32(var0.item()) == g["loss_zero_flow"]



def trace3_events(g, f):
    H, W, nev = (int(v) for v in g["meta"][:3])
    return synth.events(nev, H, W, int(g[f"f{f}/seed"]))


@pytest.mark.parametrize("trace", ["trace3_eiflow", "trace3_eraft"])
def test_multi_frame_trace_through_oracle(golden, trace):
    """Three consecutive recurrent frames of the default-size reference models (tests/golden/make_golden.py
    make_trace_multi): the oracle port reproduces the stored reference outputs (warps bit for bit, lookups to sgemm blocking order)."""
    g = golden(trace)
    H, W, nev, frames, dsub, csub = (int(v) for v in g["meta"])
    for f in range(frames):
        n_lookup, n_warp = (int(v) for v in g[f"f{f}/counts"])
        assert n_lookup in (6, 12) and n_warp == 2
        pyr = ref_port.corr_pyramid(torch.from_numpy(g[f"f{f}/fmap1"]), torch.from_numpy(g[f"f{f}/fmap2"]), 4)
        out = ref_port.corr_lookup(pyr, torch.from_numpy(g[f"f{f}/coords{n_lookup - 1}"]), 4)
        # (the stored lookups came from a CorrBlock built inside the running model: same calls, but the sgemm blocking of
        #  a D = 32 product differs between the two contexts -- 1e-7 relative, not bit-exact)
        got, ref = g.pick(f"f{f}/lookup_last", out[:, ::4].numpy())
        assert np.abs(got - ref).max() <= 1e-6 * np.abs(ref).max()
        flow = torch.from_numpy(g[f"f{f}/flow_final"])
        wi, wz = ref_port.warp_frame_and_codes(torch.from_numpy(g[f"f{f}/warp0_in"]), torch.from_numpy(g[f"f{f}/warp1_in"]),
                                               flow, "forward")
        assert np.array_equal(*g.pick(f"f{f}/warp0_out", wi.numpy())) and np.array_equal(*g.pick(f"f{f}/warp1_out", wz.numpy()))
        ev = trace3_events(g, f)
        assert ev.shape == (nev, 4) and np.all(np.diff(ev[:, 0]) >= 0)
    # the recurrence is live: consecutive frames warp different states with different flows
    assert not np.array_equal(g["f0/warp1_in"], g["f1/warp1_in"]) and not np.array_equal(g["f0/flow_final"], g["f1/flow_final"])


def test_upflow8_unpad_warp_step(golden):
    """upflow8 + ImagePadder.unpad + warps (DCEIFlow.py:222-227, e2v_model.py:188-191): oracle port == reference."""
    g = golden("warp")
    pad_h, pad_w = (int(v) for v in g["up8/pad"])
    wi, wz, flow = ref_port.warp_frame_and_codes_upflow8(torch.from_numpy(g["step/img"]), torch.from_numpy(g["step/codes"]),
                                                         torch.from_numpy(g["up8/flow_lr"]), pad_h, pad_w, "forward")
    assert np.array_equal(flow.numpy(), g["up8/flow_final"])
    assert np.array_equal(wi.numpy(), g["up8/img_warped"]) and np.array_equal(wz.numpy(), g["up8/codes_warped"])
