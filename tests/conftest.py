"""Shared fixtures.  GPU tests are marked `gpu`; everything else runs on CPU.

The oracle (oracle/) is test infrastructure: it is imported HERE, never by the
package under backgammon-engine_b200/.
"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
PKG = os.path.join(ROOT, "backgammon-engine_b200")
GOLDEN = os.path.join(ROOT, "tests", "golden")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_sessionstart(session):
    """A fresh checkout has no built libraries (they are git-ignored): build them once, exactly as the driver's
    build check does.  This compiles the product; it never substitutes anything for it."""
    import shutil
    lib = os.path.join(PKG, "lib", "libbgx.so")
    if not os.path.exists(lib) and (shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc")):
        import __graft_entry__
        __graft_entry__.build()


@pytest.fixture(scope="session")
def orc():
    from oracle.oracle import Oracle
    return Oracle()


def load_golden(name):
    """Fixture file as a plain dict (NpzFile re-reads the archive on every [] access)."""
    with np.load(os.path.join(GOLDEN, name), allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture(scope="session")
def golden():
    return load_golden


def golden_weights(g, tag):
    return tuple(g[f"{tag}_{k}"] for k in ("W1", "b1", "w2", "b2"))
