"""Driver-originated revocation on the box (reference: amdp2p.c:88-109 -- the GPU driver calls the bridge's
free_callback when pinned memory goes away, and the MR is invalidated).  In userspace the same event is observed
through the CUDA driver's allocation identity: free the memory under a live registration, and the next post must
complete with a protection error -- never touch the address."""
import json
import os
from pathlib import Path

import pytest
import torch

import rocnrdma_b200 as rn
from rocnrdma_b200 import ops, wire as W

pytestmark = pytest.mark.gpu
BIG = 64 << 20          # its own caching-allocator segment, so empty_cache() really returns it to the driver


def _victim():
    x = torch.empty(BIG, dtype=torch.uint8, device="cuda:0")
    x.fill_(7)
    torch.cuda.synchronize()
    return x


def test_tensor_registration_pins_its_storage(ctx):
    x = _victim()
    mr = ctx.reg_mr(x)
    del x
    torch.cuda.empty_cache()
    assert ctx.sweep_revoked() == 0 and mr.state == "PINNED"      # the MR holds the tensor: nothing was freed


@pytest.mark.parametrize("mode", ["direct", "dmabuf"])
def test_free_under_a_live_registration_revokes_it(request, ctx, mode):
    if mode == "dmabuf":
        request.getfixturevalue("needs_dmabuf_export")
    src = torch.full((4096,), 3, dtype=torch.uint8, device="cuda:0")
    ms = ctx.reg_mr(src)
    x = _victim()
    ptr = x.data_ptr()
    mr = ctx.reg_mr((ptr, BIG), mode=mode)                          # raw pointer: no reference to the tensor is kept
    qp = ctx.loopback_qp(depth=16, mem=W.MEM_HOST_PINNED)
    ctx.engine_start(ctas=4, idle_timeout_ms=3000)
    qp.post_write(ms, mr, 4096)
    assert qp.scq.wait(1)[0].status == "OK"
    ctx.engine_stop()
    record = {"mode": mode, "driver": torch.version.cuda}
    if mode == "dmabuf":
        assert mr.dmabuf_fd >= 0
        record["fd_size_before_free"] = ctx._lib.rn_dmabuf_size(mr.dmabuf_fd)
    fd = mr.dmabuf_fd
    del x
    torch.cuda.empty_cache()                                        # cudaFree of the segment while the MR (and the fd) is live
    if mode == "dmabuf":
        # what driver 580 does to the exported dma-buf when its backing allocation is freed
        record["fd_size_after_free"] = ctx._lib.rn_dmabuf_size(fd)
        record["fd_still_open"] = os.path.exists(f"/proc/self/fd/{fd}")
        idn = rn.api.C.c_uint64()
        record["driver_still_knows_pointer"] = ctx._lib.rn_buffer_id(ptr, rn.api.C.byref(idn)) == 0
    assert ctx.sweep_revoked() == 1
    assert mr.state == "REVOKED" and mr.driver_revoked
    assert ctx.sweep_revoked() == 0                                 # idempotent
    ctx.engine_start(ctas=4, idle_timeout_ms=3000)
    qp2 = qp
    qp2.post_write(ms, mr, 4096)                                    # names the revoked key
    wc = qp2.scq.wait(1)[0]
    ctx.engine_stop()
    assert wc.is_error and wc.status == "REMOTE_ACCESS_ERR"
    assert ctx.last_engine_fatal == 0                               # and nothing faulted on the GPU
    torch.cuda.synchronize()
    mr.dereg()
    assert mr.state == "FREE"
    if mode == "dmabuf":
        assert not os.path.exists(f"/proc/self/fd/{fd}") or os.readlink(f"/proc/self/fd/{fd}").find("dmabuf") < 0
        out = Path("gpurun_out")
        out.mkdir(exist_ok=True)
        (out / "dmabuf_after_free.json").write_text(json.dumps(record, indent=1))


def test_gpu_posted_write_to_freed_memory_is_refused(ctx):
    """The posting path of the kernels sweeps before launching: a GPU-built WQE that names a freed range gets an
    error CQE on the device."""
    src = torch.full((4096,), 5, dtype=torch.uint8, device="cuda:0")
    ms = ctx.reg_mr(src)
    x = _victim()
    mr = ctx.reg_mr((x.data_ptr(), BIG))
    qp = ctx.loopback_qp(depth=16)
    del x
    torch.cuda.empty_cache()
    ctx.engine_start(ctas=4, idle_timeout_ms=3000)
    r = ops.rdma_stream(qp, W.OP_RDMA_WRITE, ms, mr, 4096, iters=1, timeout_ms=2000)
    ctx.engine_stop()
    assert r.status == ["CQE_ERROR"] and mr.state == "REVOKED"
    assert qp.state == "ERR" and qp.counters()["state"] == "ERR"


def test_address_reuse_by_a_new_allocation_is_detected(ctx):
    x = _victim()
    ptr = x.data_ptr()
    mr = ctx.reg_mr((ptr, BIG))
    del x
    torch.cuda.empty_cache()
    y = torch.empty(BIG, dtype=torch.uint8, device="cuda:0")        # very likely the same VA again
    assert ctx.sweep_revoked() == 1 and mr.state == "REVOKED"       # same address or not, it is not the allocation that was registered
    del y
