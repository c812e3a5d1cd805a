import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# The ConnectX backend dlopen()s libibverbs once per process: point it at the in-tree mock provider before
# anything loads it (no rdma-core in the image, no /dev/infiniband in the sandbox).  `wire="auto"` never
# selects the mock, so the softhca tests are unaffected.
os.environ.setdefault("ROCNRDMA_VERBS_LIBDIR", os.path.join(ROOT, "rocnrdma_b200", "lib", "mock"))


def _private_kmod_sim():
    """The mock's peer-memory bridge gets its OWN copy of the kmod simulation: test_kmod_sim.py resets and
    reloads the shared one freely, and a dlopen of the same path would share its globals."""
    import shutil
    import tempfile
    try:
        from tools import build_kmod_sim
        src = build_kmod_sim.build()
    except Exception:
        return
    d = tempfile.mkdtemp(prefix="rn_kmod_sim_")
    dst = os.path.join(d, "libb200p2p_sim_bridge.so")
    shutil.copy(src, dst)
    os.environ.setdefault("ROCNRDMA_KMOD_SIM", dst)


_private_kmod_sim()


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with `-m gpu` under gpurun)")
    config.addinivalue_line("markers", "multigpu: needs >= 2 GPUs")


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_cuda():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture
def ctx():
    import rocnrdma_b200 as rn
    c = rn.Context(device=0)
    yield c
    c.close()


@pytest.fixture(scope="session")
def dmabuf_export_error():
    """None when the GPU driver exports device memory as a dma-buf, else the CUresult it refused with.  The device
    attribute is not enough: a paravirtualised driver (gVisor's nvproxy) reports CU_DEVICE_ATTRIBUTE_DMA_BUF_SUPPORTED
    and refuses every export."""
    import ctypes as C
    import torch
    from rocnrdma_b200 import _native as N
    lib = N.load()
    t = torch.empty(4 << 20, dtype=torch.uint8, device="cuda:0")
    lo = (t.data_ptr() + 65535) & ~65535
    lib.rn_set_device(0)
    cu = C.c_int(0)
    fd = lib.rn_dmabuf_export(lo, 1 << 20, C.byref(cu))
    if fd >= 0:
        lib.rn_dmabuf_close(fd)
        return None
    return cu.value


@pytest.fixture
def needs_dmabuf_export(dmabuf_export_error):
    if dmabuf_export_error is not None:
        pytest.skip(f"this GPU driver refuses dma-buf export of device memory (CUresult {dmabuf_export_error})")
