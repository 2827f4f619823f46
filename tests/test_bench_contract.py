"""bench.py's contract with the driver, checked on CPU (no GPU needed): the workload is BASELINE.json configs[4], both arms
print the same `config`, the byte model is SURVEY.md 8(d)'s, the 64-stream job is split 64/N, and the reference arm
runs on rank 0 only."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_headline_workload_is_configs4(bench):
    cfg = bench.make_cfg("configs[4]")
    assert (cfg["H"], cfg["W"], cfg["streams"], cfg["events"], cfg["lookups"]) == (480, 640, 64, 100000, 6)
    baseline = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "64 independent 480x640" in baseline["configs"][4] and cfg["workload"].startswith("configs[4]")
    for world in (1, 2, 4, 8):
        pc = bench.public_config(cfg, world)
        assert pc["streams_total"] == 64 and pc["streams_per_gpu"] == 64 // world
        json.dumps(pc)


def test_byte_model_matches_survey_8d(bench):
    cfg = bench.make_cfg("configs[4]")
    m = bench.bytes_model(cfg, 1)
    assert m["N"] == 4800 and (m["h"], m["w"]) == (60, 80)
    assert m["voxel"] == 32 * 100000 + 4 * 5 * 480 * 640                     # SURVEY: ~9.3 MB per window
    assert abs(m["warp"] - 83.6e6) < 0.1e6                                   # 83.6 MB per stream
    assert m["lookup"] == 4800 * 2904                                        # 13.9 MB per call
    assert m["corr_build_flops"] == 2 * 4800 * 4800 * 256                    # 11.8 GF per stream
    cfg1 = bench.make_cfg("configs[1]")
    m1 = bench.bytes_model(cfg1, 8)
    assert m1["N"] == 768 and abs(m1["warp"] / 8 - 11.7e6) < 0.1e6 and m1["lookup"] == 8 * 768 * 2904


def test_tiling_helpers(bench):
    ev = torch.arange(40, dtype=torch.float64).reshape(10, 4)
    off = torch.tensor([0, 3, 10])
    e, o = bench.tile_events(ev, off, 5)
    assert o.tolist() == [0, 3, 10, 13, 20, 23] and e.shape == (23, 4)
    assert torch.equal(e[10:13], ev[0:3]) and torch.equal(e[13:20], ev[3:10])
    rows = bench.tile_rows(torch.arange(6.).reshape(3, 2), 7)
    assert rows.shape == (7, 2) and torch.equal(rows[3], rows[0]) and torch.equal(rows[6], rows[0])


def test_reference_arm_prints_the_same_config_and_honours_steps(bench, tmp_path):
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert res.returncode == 0, res.stderr
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["steps"] == 1 and line["warmup"] == 3 and line["scaling"] == "strong"
    assert line["config"] == bench.public_config(bench.make_cfg("configs[4]"), 1)
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0 and line["gpu_launches"] == 0
    assert line["value"] > 0 and line["unit"] == "frames/s"
    names = sorted(os.listdir(tmp_path))
    assert names == sorted(["voxel.npy", "warped_frame.npy", "warped_codes.npy"] + [f"lookup{k}.npy" for k in range(6)])
    assert all(np.load(tmp_path / n).dtype == np.float32 for n in names)
    # under torchrun only rank 0 runs the CPU arm; the other ranks exit 0 without a line
    env2 = dict(env, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res2 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                          capture_output=True, text=True, timeout=120, env=env2, cwd=ROOT)
    assert res2.returncode == 0 and res2.stdout.strip() == ""


def test_dump_outputs_is_a_fixed_bounded_sample(bench, tmp_path):
    big = torch.arange(3 * 10 ** 6, dtype=torch.float32).reshape(3, 10 ** 6)
    outs = [torch.full((2, 3), float(k)) for k in range(6)]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), [np.ones((2, 2), np.float32)] * 2, outs, big, big + 1)
    names = sorted(os.listdir(tmp_path / "a"))
    assert len(names) == 9 and sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 20
    for n in names:
        a = np.load(tmp_path / "a" / n)
        assert a.dtype == np.float32 and np.array_equal(a, np.load(tmp_path / "b" / n))
    assert np.array_equal(np.load(tmp_path / "a" / "lookup3.npy"), np.full(6, 3.0, np.float32))     # small: whole
    assert np.array_equal(np.load(tmp_path / "a" / "voxel.npy"), np.ones(8, np.float32))
    frame = np.load(tmp_path / "a" / "warped_frame.npy")                                            # large: sampled
    assert 0 < frame.size < big.numel() and np.all(np.diff(frame) >= 0)
    assert np.array_equal(np.load(tmp_path / "a" / "warped_codes.npy"), frame + 1)                 # same positions


def test_stock_torch_comparator_restates_the_reference_ops():
    """scripts/stock_torch_gpu.py (the same-GPU stock-PyTorch comparator of SURVEY.md 8d) must compute what the
    reference computes: its op sequences against the pinned oracle, on CPU at a small size."""
    sys.path.insert(0, ROOT)
    from cistaflow_b200 import synth
    from oracle import ref_port
    spec = importlib.util.spec_from_file_location("stock_torch_gpu", os.path.join(ROOT, "scripts", "stock_torch_gpu.py"))
    st = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(st)
    H, W, nb = 64, 96, 5
    ev, off = synth.event_windows(2, 3000, H, W, 77)
    got = st.voxel_step(torch.from_numpy(ev.copy()), off.tolist(), nb, W, H)
    for b in range(2):
        want = ref_port.preprocess_torch(ref_port.voxel_grid_torch(torch.from_numpy(ev[off[b]:off[b + 1]].copy()), nb, W, H), "std", True)
        assert torch.equal(got[b], want)
    img, codes, flow = synth.warp_inputs(2, H, W, 78, 16, flow_kind="smooth")
    img, codes, flow = map(torch.from_numpy, (img, codes, flow))
    for mode, sign in (("forward", -1.0), ("backward", 1.0)):
        wi, wz = st.warp_step(img, codes, flow, (st.StockWarp(W, H, sign), st.StockWarp(W // 2, H // 2, sign)))
        ri, rz = ref_port.warp_frame_and_codes(img, codes, flow, mode)
        assert torch.equal(wi, ri) and torch.equal(wz, rz)
    f1, f2, c0 = synth.corr_inputs(2, 128, 192, 79)     # 16x24 map: the coarsest level is 2x3 (1x1 divides by zero)
    f1, f2, c0 = map(torch.from_numpy, (f1, f2, c0))
    pyr = st.pyramid_step(f1, f2, 4)
    ref = ref_port.corr_pyramid(f1, f2, 4)
    assert all(torch.equal(a, b) for a, b in zip(pyr, ref))
    assert torch.allclose(st.lookup_step(pyr, c0, 4), ref_port.corr_lookup(ref, c0, 4), rtol=0, atol=1e-5)
