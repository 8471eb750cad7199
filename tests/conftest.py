"""
pytest configuration.

  -m "not gpu"  : CPU suite (oracle vs the reference-generated golden fixtures, host logic,
                  C-ABI symbol table, gloo world_size-2 sharding logic).
  -m gpu        : parity tests proper -- the CUDA path, called through the C-ABI library and the
                  reference-shaped Python API, compared with the oracle on a B200.
"""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "fp8-mps-metal_b200")
for p in (ROOT, PKG, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)


def _ensure_built():
    """The native artefacts are git-ignored; build them in-tree if a fresh checkout lacks them
    (nvcc cross-compiles for sm_100a without a GPU)."""
    import glob
    need = [os.path.join(PKG, "libfp8_b200.so"), os.path.join(ROOT, "oracle", "liboracle_c.so")]
    if all(os.path.exists(n) for n in need) and glob.glob(os.path.join(PKG, "fp8_metal*.so")):
        return
    import importlib.util
    spec = importlib.util.spec_from_file_location("fp8_b200_build", os.path.join(PKG, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build_all(force=False)
    import c_oracle
    c_oracle.build()


class _RootIsNotATestPackage:
    """The repository root has an __init__.py because ComfyUI loads a clone of it as a custom node.  pytest would
    collect the root as a package and, before every test, import that __init__.py as a module named after the
    clone's directory, found through the directory above it.  Every test then errors when that directory cannot
    be listed, and otherwise the import installs the patches for the whole session.  The root is collected as a
    plain directory instead."""

    @pytest.hookimpl(tryfirst=True)
    def pytest_collect_directory(self, path, parent):
        if os.path.samefile(path, ROOT):
            return pytest.Dir.from_parent(parent, path=path)
        return None


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")
    config.pluginmanager.register(_RootIsNotATestPackage(), "fp8b-root-is-not-a-test-package")
    _ensure_built()


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    import numpy as np
    g = os.path.join(ROOT, "tests", "golden")
    import json
    with open(os.path.join(g, "kat.json")) as f:
        kat = json.load(f)
    return {
        "codec": np.load(os.path.join(g, "codec_golden.npz")),
        "host": np.load(os.path.join(g, "host_golden.npz")),
        "kat": kat,
    }


_TUNE_IDS = {"GEMM_CFG": 16, "GEMV_IMPL": 17, "DYNAMIC_PLAN": 18, "CAST_SHAPE": 19, "GEMM_STORE": 20, "GEMV_UNROLL": 21,
             "GEMV_BATCH": 22, "AMAX_CAP": 23, "GEMM_RASTER": 24, "GEMM_SPLITK": 25}


@pytest.fixture
def tune():
    """tune("GEMM_CFG", 3): force a result-identical kernel variant (fp8b_set_option FP8B_OPT_TUNE_*) for this test;
    every knob touched is reset to -1 (built-in rule) afterwards."""
    from _util import capi
    L = capi()
    touched = []

    def setter(name, value):
        assert L.fp8b_set_option(_TUNE_IDS[name], int(value)) == 0
        touched.append(name)

    yield setter
    for name in touched:
        L.fp8b_set_option(_TUNE_IDS[name], -1)
