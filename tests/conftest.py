import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA (sm_100a) device; run with `-m gpu` on the B200 box")


def load_npz(name):
    z = np.load(os.path.join(GOLDEN, name))
    meta = json.loads(bytes(z["meta"]).decode("utf-8"))
    return z, meta


@pytest.fixture(scope="session")
def fbank_golden():
    return load_npz("fbank_golden.npz")


@pytest.fixture(scope="session")
def conformer_golden():
    return load_npz("conformer_golden.npz")


@pytest.fixture(scope="session")
def predictor_golden():
    with open(os.path.join(GOLDEN, "predictor_golden.json"), encoding="utf-8") as f:
        return json.load(f)


def make_audio(kind, seed, n, scale=1.0):
    from masr_b200 import synth
    x = synth.noise_audio(seed, n) if kind == "noise" else synth.speechlike_audio(seed, n)
    return (x * np.float32(scale)).astype(np.float32)


_SD_CACHE = {}


def synth_weights(seed):
    """numpy state dict for weight seed `seed` (cached per session: 34 M parameters)."""
    from masr_b200 import synth
    if seed not in _SD_CACHE:
        _SD_CACHE[seed] = synth.conformer_state_dict(seed)
    return _SD_CACHE[seed]


@pytest.fixture(scope="session")
def gpu_engines():
    """Engines keyed by (weight seed, streaming); built lazily, shared by the GPU tests."""
    cache = {}

    def get(seed=0, streaming=True, gemm="tc"):
        from masr_b200.engine import ConformerEngine
        key = (seed, streaming, gemm)
        if key not in cache:
            cache[key] = ConformerEngine(synth_weights(seed), streaming=streaming, gemm=gemm)
        return cache[key]

    return get
