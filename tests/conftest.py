import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run with -m gpu on the B200 box)")
    config.addinivalue_line("markers", "timeout: per-test limit (pytest-timeout; harmless without the plugin)")


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


# FA_EMULATED_GPU=1 (manual, slow, never set by the driver): run the `gpu` tests against the engine emulation
# (tests/emul/engine_emul.cpp: engine.cu on a CUDA-runtime test double, kernels on the SIMT emulation) — a way to put
# a kernel variant (FA_K1_OPT=...) through the full parity suite when no GPU is at hand.  Tests that need torch.cuda
# fail there and are to be deselected (-k "not device_pointer ...").
_EMULATED = os.environ.get("FA_EMULATED_GPU") == "1"


def _load_engine_emulation():
    import ctypes
    import netobserv_ebpf_agent_b200._lib as L
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from emul_build import EMUL, build, csrc
    so = build("engine_emul", csrc("engine.cu", "aggregate.cu", "evict.cu", "features.cu", "kmap.cu", "kmap_body.cuh",
                                   "misc_kernels.cu", "pbflow.cu", "snaps.cu", "dnscorr.cu", "common.cuh", "kernels.cuh", "flowgen.h") +
               [os.path.join(EMUL, "simt.h"), os.path.join(ROOT, "include", "flowagg.h")])
    lib = ctypes.CDLL(so)
    for name, (res, args) in L.SIGNATURES.items():
        if name.startswith("fa_sharded_"):            # csrc/sharded.cu (several GPUs, peer access) is not emulated
            continue
        f = getattr(lib, name)
        f.restype, f.argtypes = res, args
    return L, lib


@pytest.fixture(scope="session", autouse=_EMULATED)
def _emulated_engine():
    L, lib = _load_engine_emulation()
    saved, L._lib = L._lib, lib
    yield lib
    L._lib = saved


@pytest.fixture
def engine_emul():
    """The whole C ABI on the CPU (tests/emul/engine_emul.cpp) swapped in for libflowagg.so for one test.  Not wider:
    a module's `gpu` tests that run after its emulation tests must get the real library."""
    L, lib = _load_engine_emulation()
    saved, L._lib = L._lib, lib
    try:
        yield lib
    finally:
        L._lib = saved


def pytest_collection_modifyitems(config, items):
    if _have_gpu() or _EMULATED:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)
