import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with `-m gpu` on the GPU box")


class Fixture(dict):
    """The arrays of one fixture.  An array stored as a fixed sample (KEY#values / KEY#mask / KEY#shape, see
    tests/golden/make_golden.py) is expanded to a zero-filled array of its full shape; ``pick`` restricts a computed
    output and the stored one to the sampled elements."""

    def __init__(self, z):
        super().__init__()
        self.masks = {}
        for k in z.files:
            if k.endswith("#values"):
                key = k[: -len("#values")]
                shape = tuple(int(s) for s in z[key + "#shape"])
                mask = np.unpackbits(z[key + "#mask"], count=int(np.prod(shape))).astype(bool).reshape(shape)
                full = np.zeros(shape, z[k].dtype)
                full[mask] = z[k]
                self[key], self.masks[key] = full, mask
            elif "#" not in k:
                self[k] = z[k]

    def pick(self, key, got):
        """(got, stored) where the fixture stores ``key``."""
        got, ref = np.asarray(got), self[key]
        assert got.shape == ref.shape, (key, got.shape, ref.shape)
        mask = self.masks.get(key)
        return (got, ref) if mask is None else (got[mask], ref[mask])


@pytest.fixture(scope="session")
def golden():
    """Loader for the fixtures generated from the reference (tests/golden/make_golden.py)."""
    cache = {}

    def load(name):
        if name not in cache:
            with np.load(os.path.join(GOLDEN, name + ".npz")) as z:
                cache[name] = Fixture(z)
        return cache[name]
    return load


@pytest.fixture(scope="session")
def cuda_device():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


class _ParityReport:
    """Collects the agreement fractions the GPU parity tests measure (north_star: ">= 95 % tolerance-agreement")
    and writes them to gpurun_out/parity_report.json at the end of the session."""

    def __init__(self):
        self.rows = []

    def add(self, test, **kw):
        self.rows.append({"test": test, **{k: (float(v) if isinstance(v, (float, np.floating)) else v) for k, v in kw.items()}})


@pytest.fixture(scope="session")
def parity_report():
    rep = _ParityReport()
    yield rep
    if rep.rows:
        import json
        out = os.path.join(ROOT, "gpurun_out")
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "parity_report.json"), "w") as fh:
            json.dump(rep.rows, fh, indent=1)
