"""pytest fixtures.  `-m "not gpu"` runs here (no GPU): oracle pinning, host logic, C-ABI
exports.  `-m gpu` tests are the parity tests proper and call through the C-ABI on a B200."""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import __graft_entry__ as ge  # noqa: E402


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def pkg():
    os.environ.setdefault("PK_SKIP_REF_BUILD", "1")
    p = ge.load_package()
    if not os.path.exists(p.lib_path()):
        ge.build()
    return p


@pytest.fixture(scope="session")
def O():
    return ge.load_oracle()


@pytest.fixture(scope="session")
def synth(pkg):
    from parakeet_cpp_b200 import synth as s
    return s


class Model:
    """A seeded synthetic checkpoint on disk + both config views + vocab."""

    def __init__(self, tmpdir, pkg, O, synth, kind, seed):
        self.kind = kind
        if kind == "tiny":
            self.ocfg, self.cfg = O.make_tiny_config(), pkg.make_tiny_config()
        elif kind == "110m":
            self.ocfg, self.cfg = O.make_110m_config(), pkg.make_110m_config(max_batch=8)
        else:
            raise ValueError(kind)
        self.W = synth.make_weights(self.ocfg, seed=seed)
        self.weights_path = os.path.join(tmpdir, f"{kind}_{seed}.safetensors")
        synth.save_safetensors(self.weights_path, self.W)
        self.pieces = synth.make_vocab(self.ocfg.vocab - 1, seed=seed)
        self.vocab_path = os.path.join(tmpdir, f"{kind}_{seed}.vocab.txt")
        synth.save_vocab(self.vocab_path, self.pieces)


@pytest.fixture(scope="session")
def tiny(tmp_path_factory, pkg, O, synth):
    return Model(str(tmp_path_factory.mktemp("tiny")), pkg, O, synth, "tiny", 3)


@pytest.fixture(scope="session")
def m110(tmp_path_factory, pkg, O, synth):
    return Model(str(tmp_path_factory.mktemp("m110")), pkg, O, synth, "110m", 0)


@pytest.fixture(scope="session")
def golden():
    """The reference's outputs on the tiny model's clips and the 110m clip (two files, each below 1 MB)."""
    d = {}
    for name in ("golden_v1.npz", "golden_110m_v1.npz"):
        with np.load(os.path.join(ROOT, "tests", "golden", name), allow_pickle=False) as z:
            d.update(z)
    return d


@pytest.fixture(scope="session")
def golden_refcalls():
    """Single calls into the compiled reference that the oracle and resampler tests compare with."""
    with np.load(os.path.join(ROOT, "tests", "golden", "golden_refcalls_v1.npz"), allow_pickle=False) as z:
        return dict(z)
