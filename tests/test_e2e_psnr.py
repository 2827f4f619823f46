"""End-to-end PSNR gate (north_star: "reconstructions must agree within 0.01 dB PSNR"), run where the reference lives.

The UNMODIFIED reference models (e2v/e2v_model.py:144-196 DCEIFlowCistaNet, :206-248 ERAFTCistaNet; default
base_channels = 64, 180x240, 10 recurrent frames, seeded random-init weights -- the pretrained files are not in the
reference checkout, SURVEY F4) are run twice on the same synthetic event stream:

  stock      the reference's own hot path;
  perturbed  the same model with every deviation the CUDA path is allowed to introduce injected at the reference's
             own call sites, at the magnitude the GPU parity tests measure:
               * CorrBlock operands rounded to TF32 (round-to-nearest-even to 10 mantissa bits -- exactly what the
                 TFLOAT32 tensor map does to the feature maps on their way into shared memory);
               * the voxel grid accumulated in a DIFFERENT event order (what the atomic mode is: fp32 sums of the same
                 weights in an unspecified order), then normalised by the reference;
               * warped frame / codes and lookup outputs perturbed by fp32 rounding noise (relative 2^-22), the
                 measured level of the CUDA kernels' op-order differences (the parity tests allow 1e-4 absolute).

PSNR is loss.py:15-24's formula against a fixed synthetic ground-truth sequence; the gate is |dPSNR| <= 0.01 dB per
frame for BOTH model modes, and the perturbed reconstruction itself must sit >= 50 dB from the stock one.
This runs the original project's networks, which are not part of this repository: set CISTA_REFERENCE to a checkout of
it; without one the test is skipped, and tests/test_gpu_parity*.py replay the recorded multi-frame traces through the
real kernels instead.
"""
import argparse
import math
import os
import sys
import types

import numpy as np
import pytest
import torch

REF = os.environ.get("CISTA_REFERENCE", "")
pytestmark = pytest.mark.skipif(not os.path.isdir(REF), reason="CISTA_REFERENCE does not name a checkout of the original project")

H, W, NEV, FRAMES = 180, 240, 15000, 10


def _stub_optional_imports():
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


def round_to_tf32(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> nearest TF32 (10 explicit mantissa bits, ties to even), returned as fp32."""
    u = x.contiguous().view(torch.int32)
    bias = ((u >> 13) & 1) + 0x0FFF
    return ((u + bias) & ~0x1FFF).view(torch.float32)


def psnr(a: torch.Tensor, b: torch.Tensor) -> float:
    """loss.py:15-24"""
    mse = float(((a.double() - b.double()) ** 2).mean())
    return 100.0 if mse < 1e-10 else 20.0 * math.log10(1.0 / math.sqrt(mse))


def fp32_noise(t: torch.Tensor, gen: torch.Generator) -> torch.Tensor:
    return t * (1.0 + (torch.rand(t.shape, generator=gen) - 0.5) * 2.0 ** -21)


def run_model(model_mode: str, perturbed: bool):
    if REF not in sys.path:
        sys.path.insert(0, REF)
    sys.dont_write_bytecode = True
    _stub_optional_imports()
    from cistaflow_b200 import synth
    from utils.configs import set_configs
    from utils import event_process as ep
    import e2v.e2v_model as em
    import utils.flow_utils as fu

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
    gen = torch.Generator().manual_seed(99)
    rng = np.random.default_rng(7)
    RefCorr = host.CorrBlock
    ref_warp_frame = fu.FrameWarp.warp_frame

    class Tf32Corr(RefCorr):
        def __init__(self, fmap1, fmap2, num_levels=4, radius=4):
            super().__init__(round_to_tf32(fmap1), round_to_tf32(fmap2), num_levels=num_levels, radius=radius)

        def __call__(self, coords):
            return fp32_noise(super().__call__(coords), gen)

    def noisy_warp(self, I, flow):
        return fp32_noise(ref_warp_frame(self, I, flow), gen)

    if perturbed:
        host.CorrBlock = Tf32Corr
        fu.FrameWarp.warp_frame = noisy_warp
    recs, flows = [], []
    try:
        states, prev, vox_old = None, torch.zeros(1, 1, H, W), torch.zeros(1, 5, H, W)
        with torch.no_grad():
            for frame in range(FRAMES):
                ev = synth.events(NEV, H, W, synth.seed_for(1, frame))
                if perturbed:
                    # same events, same weights, another accumulation order: rows 1..n-2 permuted (rows 0 and n-1
                    # define t0 and dT in the reference, utils/event_process.py:39-44)
                    perm = np.concatenate([[0], 1 + rng.permutation(len(ev) - 2), [len(ev) - 1]])
                    ev = ev[perm]
                grid = ep.events_to_voxel_grid(ev.copy(), 5, W, H)
                vox = np.asarray(ep.event_preprocess(grid.copy(), "std", True), np.float32)
                vox_t = torch.from_numpy(vox)[None]
                if model_mode == "cista-eiflow":
                    batch = {"event_voxel": vox_t, "rec_img0": prev}
                else:
                    batch = {"event_voxel": vox_t, "event_voxel_old": vox_old, "rec_img0": prev}
                pred, flow_out, states = model(batch, states)
                recs.append(pred.clone())
                flows.append(flow_out["flow_final"].clone())
                prev, vox_old = pred.clone(), vox_t
    finally:
        host.CorrBlock = RefCorr
        fu.FrameWarp.warp_frame = ref_warp_frame
    return recs, flows


@pytest.mark.parametrize("model_mode", ["cista-eiflow", "cista-eraft"])
def test_e2e_psnr_within_0p01_db(model_mode):
    from cistaflow_b200 import synth
    stock, flow_s = run_model(model_mode, perturbed=False)
    pert, flow_p = run_model(model_mode, perturbed=True)
    rng = np.random.default_rng(3)
    rows = []
    for k in range(FRAMES):
        gt = torch.from_numpy(synth.smooth_field(rng, 1, 1, H, W, 0.25, cell=24)).clamp(-0.5, 0.5) + 0.5
        p_s, p_p = psnr(stock[k], gt), psnr(pert[k], gt)
        rows.append((k, p_s, p_p, psnr(pert[k], stock[k]), float((flow_p[k] - flow_s[k]).abs().max()),
                     float(flow_s[k].abs().max())))
    for k, p_s, p_p, p_x, df, fmax in rows:
        print(f"{model_mode} frame {k}: PSNR stock {p_s:.4f} dB, perturbed {p_p:.4f} dB, dPSNR {p_p - p_s:+.5f} dB, "
              f"perturbed-vs-stock {p_x:.1f} dB, max|dflow| {df:.2e} px (|flow|max {fmax:.1f})")
    assert max(r[5] for r in rows) > 0.5, "degenerate run: the flow network predicts no motion"
    assert all(abs(p_p - p_s) <= 0.01 for _, p_s, p_p, _, _, _ in rows[3:]), rows   # the drivers skip the first 3 frames too
    assert all(abs(p_p - p_s) <= 0.01 for _, p_s, p_p, _, _, _ in rows), rows
    assert min(r[3] for r in rows) >= 50.0, rows
