import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


def rel_err(got: np.ndarray, ref: np.ndarray) -> float:
    """The parity metric of BASELINE.md: max|got - ref| / max|ref| over one blob."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    denom = max(float(np.abs(ref).max()), 1e-30)
    return float(np.abs(got - ref).max()) / denom


def sample_index(size: int, n: int = 512) -> np.ndarray:
    """n flat indices spread over an array of `size` elements (a fixed stride modulo a prime), or all of them."""
    if size <= n:
        return np.arange(size)
    return np.arange(n, dtype=np.int64) * 1000003 % size


def sample_of(ref: np.ndarray) -> dict:
    """What tests/golden/ keeps of a large reference output: its values at sample_index and max|ref| over the whole
    array (the denominator of rel_err)."""
    ref = np.asarray(ref, np.float32).reshape(-1)
    return {"val": ref[sample_index(ref.size)], "amax": np.float32(np.abs(ref).max())}


def sampled_rel_err(got: np.ndarray, gold, key: str) -> float:
    """rel_err against a stored sample (sample_of, saved under `key`/val and `key`/amax): max|got - ref| over the
    sampled elements / max|ref| over the whole reference array."""
    got = np.asarray(got, np.float64).reshape(-1)
    want = gold[key + "/val"]
    got = got[sample_index(got.size)]
    assert got.shape == want.shape, (got.shape, want.shape)
    return float(np.abs(got - want).max()) / max(float(gold[key + "/amax"]), 1e-30)


def digest(*arrays) -> str:
    """sha256 of the arrays' bytes: pins the regenerated inputs of a golden comparison to the ones it was made from."""
    import hashlib
    h = hashlib.sha256()
    for a in arrays:
        if a is not None:
            h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as O
    O.build(ref=True)
    return O


@pytest.fixture(scope="session")
def restatement(oracle):
    return oracle.restatement()


@pytest.fixture(scope="session")
def model_dir(tmp_path_factory):
    return tmp_path_factory.mktemp("models")


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


@pytest.fixture(autouse=True)
def _default_precision():
    """Every test starts in the engine's default arithmetic mode (FP32_SPLIT); tests that pin a mode set it themselves."""
    try:
        from feathercnn_b200 import booster
        booster.set_precision(booster.PRECISION_FP32_SPLIT)
    except Exception:  # libraries not built (pure-oracle CPU tests)
        pass
    yield
