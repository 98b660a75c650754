"""Shared fixtures.  `-m gpu` tests need a B200; everything else runs on CPU."""
from __future__ import annotations

import json
import os
import sys
from pathlib import Path

import numpy as np
import pytest

REPO = Path(__file__).resolve().parents[1]
if str(REPO) not in sys.path:
    sys.path.insert(0, str(REPO))
GOLDEN = REPO / "tests" / "golden"
# A checkout of the original Python project, for the few tests that import its modules (optional)
REFERENCE = Path(os.environ["DSP_REF_PATH"]) if os.environ.get("DSP_REF_PATH") else None


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "needs_reference: imports the original project from DSP_REF_PATH")


def pytest_collection_modifyitems(config, items):
    have_ref = REFERENCE is not None and (REFERENCE / "src" / "dsp" / "fft.py").exists()
    skip_ref = pytest.mark.skip(reason="DSP_REF_PATH does not name a checkout of the original project")
    for item in items:
        if "needs_reference" in item.keywords and not have_ref:
            item.add_marker(skip_ref)


def rel_err(a, b) -> float:
    """Reference parity metric (scripts/tools/compare_librosa.py:37-38)."""
    a = np.asarray(a)
    b = np.asarray(b)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-8))


@pytest.fixture(scope="session")
def golden_small():
    z = np.load(GOLDEN / "features_small.npz")
    meta = json.loads(bytes(z["meta_json"]).decode())
    return z, meta


@pytest.fixture(scope="session")
def golden_config1():
    return np.load(GOLDEN / "config1_clip.npz")


@pytest.fixture(scope="session")
def golden_real():
    return np.load(GOLDEN / "real_clip.npz")


@pytest.fixture(scope="session")
def golden_fft():
    return np.load(GOLDEN / "fft_cases.npz")


@pytest.fixture(scope="session")
def golden_retrieval():
    return np.load(GOLDEN / "retrieval.npz")


@pytest.fixture(scope="session")
def known_answers():
    return json.loads((GOLDEN / "known_answers.json").read_text())
