"""CPU-side checks: the C-ABI library loads and exports every symbol the header
declares, the product fails loudly without a GPU (no CPU fallback), install()
rebinding, synthetic generators, stream sharding incl. a world_size-2 gloo run."""
import os
import re
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built_lib():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as entry
    entry.build()
    from cistaflow_b200 import _lib
    return _lib


def header_symbols():
    text = open(os.path.join(ROOT, "include", "cistaflow.h")).read()
    return sorted(set(re.findall(r"CF_API\s+[\w\s\*]+?\b(cf_\w+)\s*\(", text)))


def test_header_declares_the_expected_entry_points():
    syms = header_symbols()
    for s in ("cf_voxel_bin", "cf_warp", "cf_warp_frame_and_codes", "cf_corr_build", "cf_corr_lookup",
              "cf_voxel_preprocess", "cf_last_error", "cf_version", "cf_device_check"):
        assert s in syms
    assert len(syms) == 26


def test_library_exports_every_header_symbol(built_lib):
    lib = built_lib.load()
    for name in header_symbols():
        assert hasattr(lib, name), f"libcistaflow.so does not export {name}"
        assert name in built_lib.SYMBOLS, f"ctypes table lacks {name}"
    assert sorted(built_lib.SYMBOLS) == header_symbols()
    assert lib.cf_version() == 100
    # no undefined references to torch / python: the boundary is plain C
    out = subprocess.run(["nm", "-D", "--undefined-only", built_lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "torch" not in out.lower() and "Py" not in out


def test_sass_contains_blackwell_tensor_and_tma_instructions(built_lib):
    """tcgen05.mma -> UTC*MMA, tcgen05.ld -> LDTM, TMA -> UTMALDG, fp32 atomics -> REDG."""
    cuobjdump = "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", built_lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG", "REDG.E.ADD.F32"):
        assert mnemonic in sass, mnemonic


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_ops_fail_loudly_without_gpu(built_lib):
    import cistaflow_b200 as cf
    lib = built_lib.load()
    assert lib.cf_device_check() != 0
    assert b"no CPU fallback" in lib.cf_last_error()
    ev = np.zeros((4, 4))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cf.events_to_voxel_grid(ev, 5, 8, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cf.forwardWarp(8, 8)(torch.zeros(1, 1, 8, 8), torch.zeros(1, 2, 8, 8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        cf.CorrBlock(torch.zeros(1, 32, 8, 8), torch.zeros(1, 32, 8, 8))
    # direct C-ABI call with no device: an error code, never a computed result
    rc = lib.cf_warp(1, 1, 1, 1, 1, 8, 8, 8, 8, -1.0, None)
    assert rc < 0


def test_missing_library_is_an_error(monkeypatch, built_lib):
    monkeypatch.setattr(built_lib, "_lib", None)
    monkeypatch.setattr(built_lib, "LIB_PATH", "/nonexistent/libcistaflow.so")
    with pytest.raises(RuntimeError, match="no CPU / PyTorch fallback"):
        built_lib.load()


def test_product_does_not_import_the_oracle():
    src_dir = os.path.join(ROOT, "cista-flow_b200")
    for dirpath, _, files in os.walk(src_dir):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), f"{f} imports the oracle"
                assert "/root/reference" not in text


def test_install_rebinds_importers(monkeypatch):
    import importlib
    import cistaflow_b200 as cf
    inst = importlib.import_module("cistaflow_b200.install")  # the module (cf.install is the function)
    sentinel = object()
    fake_fu = types.ModuleType("utils.flow_utils")
    fake_fu.FrameWarp = fake_fu.backWarp = fake_fu.forwardWarp = sentinel
    fake_model = types.ModuleType("e2v.e2v_model")
    fake_model.FrameWarp = sentinel
    fake_eraft = types.ModuleType("ERAFT.eraft")
    fake_eraft.CorrBlock = sentinel
    fake_vr = types.ModuleType("data_readers.video_readers")
    fake_vr.events_to_voxel_grid = fake_vr.event_preprocess = sentinel
    fake_vr.unrelated = sentinel
    for m in (fake_fu, fake_model, fake_eraft, fake_vr):
        monkeypatch.setitem(sys.modules, m.__name__, m)
    done = inst.install(import_missing=False)
    assert fake_model.FrameWarp is cf.FrameWarp and fake_fu.backWarp is cf.backWarp
    assert fake_eraft.CorrBlock is cf.CorrBlock
    assert fake_vr.events_to_voxel_grid is cf.events_to_voxel_grid and fake_vr.event_preprocess is cf.event_preprocess
    assert fake_vr.unrelated is sentinel
    assert "e2v.e2v_model.FrameWarp" in done and "ERAFT.eraft.CorrBlock" in done
    inst.uninstall()
    assert fake_model.FrameWarp is sentinel and fake_eraft.CorrBlock is sentinel


def test_reference_signatures_are_mirrored():
    import inspect
    import cistaflow_b200 as cf
    sig = inspect.signature
    assert list(sig(cf.events_to_voxel_grid).parameters)[:5] == ["events", "num_bins", "width", "height", "is_reverse"]
    assert list(sig(cf.events_to_voxel_grid_pytorch).parameters)[:4] == ["events", "num_bins", "width", "height"]
    assert list(sig(cf.event_preprocess).parameters) == ["event_voxel_grid", "mode", "filter_hot_pixel"]
    assert sig(cf.event_preprocess).parameters["mode"].default == "std"
    assert list(sig(cf.backWarp.__init__).parameters)[1:] == ["W", "H"]
    assert list(sig(cf.FrameWarp.warp_frame).parameters)[1:] == ["I", "flow"]
    p = sig(cf.CorrBlock.__init__).parameters
    assert list(p)[1:5] == ["fmap1", "fmap2", "num_levels", "radius"] and p["num_levels"].default == 4 and p["radius"].default == 4
    g = cf.coords_grid(2, 3, 4)
    assert g.shape == (2, 2, 3, 4) and g[0, 0, 1, 2] == 2 and g[0, 1, 1, 2] == 1  # ch0 = x, ch1 = y
    # the second voxeliser (data_readers/MVSEC_utils.py:253, 306, 384, 388)
    p = sig(cf.events_to_voxel_torch).parameters
    assert list(p)[:8] == ["xs", "ys", "ts", "ps", "B", "device", "sensor_size", "temporal_bilinear"]
    assert p["sensor_size"].default == (180, 240) and p["temporal_bilinear"].default is True
    assert list(sig(cf.events_to_neg_pos_voxel_torch).parameters)[:8] == list(p)[:8]
    for fn in (cf.eventsToVoxel, cf.eventsToVoxelTorch):
        q = sig(fn).parameters
        assert list(q)[:6] == ["events", "num_bins", "height", "width", "event_polarity", "temporal_bilinear"]
        assert q["num_bins"].default == 5 and q["event_polarity"].default is False


def test_synth_generators_are_seeded_and_well_formed():
    from cistaflow_b200 import synth
    a, b = synth.events(5000, 30, 40, 7), synth.events(5000, 30, 40, 7)
    assert np.array_equal(a, b) and a.dtype == np.float64 and a.shape == (5000, 4)
    assert (np.diff(a[:, 0]) >= 0).all() and a[:, 0].min() >= synth.T_BASE
    assert a[:, 1].max() < 40 and a[:, 2].max() < 30 and set(np.unique(a[:, 3])) <= {0.0, 1.0}
    assert np.float32(a[1, 0]) == np.float32(a[0, 0])  # stamps really do NOT survive fp32 (SURVEY F10)
    ev, off = synth.event_windows(3, 100, 8, 8, 1)
    assert ev.shape == (300, 4) and list(off) == [0, 100, 200, 300]
    img, codes, flow = synth.warp_inputs(2, 36, 44, 3)
    assert img.shape == (2, 1, 36, 44) and codes.shape == (2, 128, 18, 22) and flow.shape == (2, 2, 36, 44)
    assert 0.4 < (codes == 0).mean() < 0.8
    f1, f2, c = synth.corr_inputs(1, 180, 240, 3)
    assert f1.shape == (1, 256, 24, 32) and c.shape == (1, 2, 24, 32)
    assert synth.padded_dims(260, 346) == (288, 352) and synth.padded_dims(480, 640) == (480, 640)


def test_pack_events_host_layout():
    """The host packer's record layout (include/cistaflow.h part 1b): low word float32 t - t_first_of_window,
    high word x | y << 16 | p << 31; out-of-range coordinates are marked with x = 0xffff."""
    import cistaflow_b200 as cf
    ev = np.array([[1000.0, 3, 4, 1], [1000.0 + 2.5e-3, 239, 179, 0], [2000.0, 7, 8, 1], [2000.25, -1, 2, 0]])
    off = np.array([0, 2, 4])
    rec = cf.pack_events_host(ev, off)
    assert rec.dtype == np.uint64 and rec.shape == (4,)
    lo = (rec & np.uint64(0xffffffff)).astype(np.uint32).view(np.float32)
    hi = (rec >> np.uint64(32)).astype(np.uint32)
    np.testing.assert_array_equal(lo, np.array([0.0, 2.5e-3, 0.0, 0.25], np.float32))   # stamps relative to each window
    assert lo[1] == np.float32(np.float64(1000.0 + 2.5e-3) - 1000.0) != np.float32(1000.0 + 2.5e-3) - np.float32(1000.0)
    assert list(hi & 0xffff) == [3, 239, 7, 0xffff] and list((hi >> 16) & 0x7fff) == [4, 179, 8, 0]
    assert list(hi >> 31) == [1, 0, 1, 0]


def test_shard_streams_partition():
    from cistaflow_b200 import sharding
    for n, world in ((64, 1), (64, 8), (10, 4), (3, 8)):
        parts = [sharding.shard_streams(n, world, r) for r in range(world)]
        assert sorted(sum(parts, [])) == list(range(n))
        assert [len(p) for p in parts] == sharding.streams_per_rank(n, world)
        assert max(map(len, parts)) - min(map(len, parts)) <= 1
    table = sharding.gather_stream_metrics([0, 1], torch.tensor([[1.0, 2.0], [3.0, 4.0]]), 2)
    assert table.tolist() == [[1.0, 2.0], [3.0, 4.0]]
    assert sharding.max_over_ranks(1.5, torch.device("cpu")) == 1.5


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from cistaflow_b200 import sharding
rank, local, world = sharding.env_rank_world()
dist.init_process_group("gloo", rank=rank, world_size=world)
n = 5
mine = sharding.shard_streams(n, world, rank)
rows = torch.tensor([[float(s), 10.0 * s + rank] for s in mine], dtype=torch.float64).reshape(len(mine), 2)
table = sharding.gather_stream_metrics(mine, rows, n)
assert table.shape == (n, 2)
for s in range(n):
    assert table[s, 0] == s and table[s, 1] == 10.0 * s + (s % world), (s, table[s])
t = sharding.max_over_ranks(1.0 + rank, torch.device("cpu"))
assert t == float(world)
dist.barrier()
dist.destroy_process_group()
os.write(1, f"OK {rank}\n".encode())  # one write(2): atomic on a pipe, the two ranks cannot interleave
"""


def test_sharding_world_size_2_gloo(tmp_path):
    """The N>1 path on CPU: two ranks, gloo, uneven shard (5 streams), metric gather + max-over-ranks."""
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    import socket
    with socket.socket() as sock:  # a free port: a fixed one can collide with a lingering run
        sock.bind(("127.0.0.1", 0))
        port = sock.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(port), str(script), ROOT]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "OK 0" in res.stdout and "OK 1" in res.stdout


REF = os.environ.get("CISTA_REFERENCE", "")


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "e2v")), reason="CISTA_REFERENCE does not name a checkout of the original project")
def test_install_against_the_real_reference_modules():
    """install() rebinds the names inside the reference's own modules (CPU: import + rebind only)."""
    code = r"""
import sys, types
sys.dont_write_bytecode = True
sys.path.insert(0, %r); sys.path.insert(0, %r)
mpl = types.ModuleType("matplotlib"); plt = types.ModuleType("matplotlib.pyplot"); mpl.pyplot = plt
sys.modules["matplotlib"] = mpl; sys.modules["matplotlib.pyplot"] = plt
oc = types.ModuleType("omegaconf")
class OmegaConf:
    create = staticmethod(lambda d: types.SimpleNamespace(**d))
oc.OmegaConf = OmegaConf; sys.modules["omegaconf"] = oc
import e2v.e2v_model, ERAFT.eraft, DCEIFlow.DCEIFlow, data_readers.video_readers, data_readers.MVSEC_utils
import cistaflow_b200 as cf
done = cf.install()
assert data_readers.MVSEC_utils.eventsToVoxel is cf.eventsToVoxel          # the second voxeliser
assert data_readers.MVSEC_utils.events_to_voxel_torch is cf.events_to_voxel_torch
assert e2v.e2v_model.FrameWarp is cf.FrameWarp
assert ERAFT.eraft.CorrBlock is cf.CorrBlock and DCEIFlow.DCEIFlow.CorrBlock is cf.CorrBlock
assert data_readers.video_readers.events_to_voxel_grid is cf.events_to_voxel_grid
assert data_readers.video_readers.event_preprocess is cf.event_preprocess
import argparse
from utils.configs import set_configs
p = argparse.ArgumentParser(); set_configs(p)
m = e2v.e2v_model.ERAFTCistaNet(p.parse_args(["--model_mode", "cista-eraft", "--base_channels", "8"]))
assert isinstance(m.frame_warp, cf.FrameWarp)       # the model now owns OUR FrameWarp
cf.uninstall()
assert e2v.e2v_model.FrameWarp is not cf.FrameWarp
print("OK", len(done))
""" % (REF, ROOT)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "OK" in res.stdout, res.stdout + res.stderr


@pytest.mark.parametrize("H,W", [(130, 173), (33, 51), (312, 485), (35, 22), (36, 27)])
def test_quad_row_view_index_math(H, W):
    """The odd-pitch warp stages codes through a tensor map over the buffer seen as [groups of P channels][P*H/4 rows]
    [4*W floats] (warp_tma.cu, QUAD).  This restates the index arithmetic of the issue side (four [48 x 6 x 8] boxes per
    stage at 16-byte aligned columns) and of the consumer side (box k%4, row k/4, column shift) in NumPy and checks
    that every (channel, source row, column) of a stage is found where the consumer looks for it."""
    B, C, BW, BH, CC = 2, 64, 48, 24, 8
    P = 1 if H % 4 == 0 else (4 if H % 2 else 2)
    rng = np.random.default_rng(H * 1000 + W)
    buf = rng.standard_normal((B, C, H, W)).astype(np.float32)
    view = buf.reshape(B * C // P, P * H // 4, 4 * W)          # the 3-D tensor map: dims (4W, P*H/4, B*C/P)

    def box(col, row, grp):                                       # TMA tile load, zero fill outside the map
        out = np.zeros((CC, BH // 4, BW), np.float32)
        for ci in range(CC):
            for ri in range(BH // 4):
                for xi in range(BW):
                    g, r, x = grp + ci, row + ri, col + xi
                    if g < view.shape[0] and r < view.shape[1] and x < view.shape[2]:
                        out[ci, ri, xi] = view[g, r, x]
        return out

    for b, c_begin, chunk, by, bx in [(0, 0, 0, 0, 0), (1, 0, 1, 5, 7), (1, 0, 3, H - 20, max(W - 45, 0)), (0, 0, 7, 17, 2)]:
        pp = chunk % P
        first_channel = c_begin + pp + P * CC * (chunk // P)
        group = (b * C + c_begin) // P + CC * (chunk // P)
        r0 = pp * H + by
        stage = np.stack([box((((r0 + j) & 3) * W + bx) & ~3, (r0 + j) >> 2, group) for j in range(4)])   # [4][8][6][48]
        flat = stage.reshape(-1)
        q = ((b * C + first_channel) * H + by) & 3
        assert q == r0 & 3
        for k in range(min(BH, H - by)):
            shift = (((k + q) & 3) * W + bx) & 3
            row = ((k & 3) * (CC * (BH // 4)) + (k >> 2)) * BW + shift
            for i in range(CC):
                c = first_channel + P * i
                n = min(BW - 3, W - bx)
                got = flat[i * (BH // 4) * BW + row: i * (BH // 4) * BW + row + n]
                assert np.array_equal(got, buf[b, c, by + k, bx:bx + n]), (b, c, k)
