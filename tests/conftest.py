"""Shared pytest plumbing.

* ``-m "not gpu"``: oracle vs golden fixtures, host logic, C-ABI symbol checks, gloo world-size-2
  choreography - no CUDA calls.
* ``-m gpu``: parity of the CUDA path (through the C ABI) against the oracle / fixtures on a B200.
"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (sm_100) GPU; run with -m gpu")


def pytest_collection_modifyitems(config, items):
    """GPU tests are skipped (not failed) when no CUDA device is visible, so a bare ``pytest``
    in the CPU container stays green; on the GPU box they run and must load the native library."""
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    """Loads ``tests/golden/<name>.npz``; a fixture made from seeded inputs gets them back, regenerated and checked
    against the digests it stores (``tests/_golden_inputs.py``)."""
    import _golden_inputs

    def load(name):
        z = np.load(os.path.join(GOLDEN, name + ".npz"))
        if name not in _golden_inputs.SEEDED:
            return z
        return {**{k: z[k] for k in z.files}, **_golden_inputs.regenerate(name, z)}
    return load


def rel_err(a, b):
    """||a - b|| / ||b|| per tensor (SURVEY.md section 8 c: the tolerance norm)."""
    import torch
    a = torch.as_tensor(a).double().cpu().reshape(-1)
    b = torch.as_tensor(b).double().cpu().reshape(-1)
    den = b.norm().item()
    return (a - b).norm().item() / (den if den > 0 else 1.0)


@pytest.fixture(scope="session")
def lib_built():
    """Build (or reuse) the in-tree shared library; nvcc cross-compiles without a GPU."""
    from mae_clip_b200 import _build
    return _build.build()
