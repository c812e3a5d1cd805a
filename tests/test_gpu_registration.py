"""N1 userspace registration on a real B200: dma-buf export, the harness twin, MR modes."""
import pytest
import torch

from rocnrdma_b200 import harness as H

pytestmark = pytest.mark.gpu
PAGE = 1 << 16


def _buf(n):
    # cudaMalloc-backed, 2 MiB aligned: the caching allocator's large blocks
    t = torch.zeros(max(n, 4 << 20), dtype=torch.uint8, device="cuda:0")
    assert t.data_ptr() % PAGE == 0
    return t


def test_twin_classifies_addresses_and_page_size():
    be = H.UserBackend()
    t = _buf(4 * PAGE)
    host = torch.zeros(4096, dtype=torch.uint8)
    assert be.is_gpu_address(t.data_ptr()) and be.is_gpu_address(t.data_ptr() + 12345)
    assert not be.is_gpu_address(host.data_ptr())
    assert be.get_page_size(t.data_ptr(), 2 * PAGE) == PAGE
    with pytest.raises(H.HarnessError):
        be.get_page_size(host.data_ptr(), 4096)
    be.close()


def test_twin_pin_multi_pin_and_cpu_window(needs_dmabuf_export):
    be = H.UserBackend()
    t = _buf(8 * PAGE)
    va = t.data_ptr()
    g = be.get_pages(va, 4 * PAGE)
    assert g.entries == 4 and g.page_size == PAGE and g.handle
    assert be.pin_size(g.handle) == 4 * PAGE            # the kernel agrees on what the dma-buf covers
    be.get_pages(va, 4 * PAGE)                           # same range pinned again
    be.get_pages(va, 2 * PAGE)
    assert be.live_pins == 3
    # CPU window: poke through the pin, read back on the GPU and vice versa
    be.poke(va + 100, b"b200p2p!")
    torch.cuda.synchronize()
    assert bytes(t[100:108].cpu().tolist()) == b"b200p2p!"
    t[PAGE:PAGE + 4] = torch.tensor([1, 2, 3, 4], dtype=torch.uint8, device="cuda:0")
    torch.cuda.synchronize()
    assert be.peek(va + PAGE, 4) == bytes([1, 2, 3, 4])
    with pytest.raises(H.HarnessError):
        be.peek(va + 4 * PAGE, 16)                       # outside every pin
    assert be.put_pages(va, 4 * PAGE) == 2               # one PUT releases every exact match
    assert be.put_pages(va + PAGE, PAGE) == 0
    assert be.live_pins == 1
    assert be.close() == 1                               # close-with-leaks releases the rest


def test_twin_cpu_mapping_of_the_pin_is_attempted_and_reported(needs_dmabuf_export):
    """The kernel harness maps the pinned pages into the caller (reference: tests/amdp2ptest.c:336-395).  From userspace the
    only handle on a pin is its dma-buf: mmap() of that fd is the same window where the exporter implements it.  Either it
    maps -- then peek / poke are CPU accesses through the BAR and must agree with the GPU's view -- or the attempt fails
    cleanly with the driver's errno (driver 580: ENOTSUPP, 524) and the twin says it is on the cudaMemcpy fallback."""
    be = H.UserBackend()
    t = _buf(2 * PAGE)
    va = t.data_ptr()
    g = be.get_pages(va, 2 * PAGE)
    try:
        addr, n = be.map_window(g.handle)
    except H.HarnessError as e:
        assert e.errno > 0
        assert be.window_kind(va).startswith("cudaMemcpy")
    else:
        assert addr and n == 2 * PAGE
        assert be.window_kind(va).startswith("dmabuf-mmap")
    be.poke(va + 8, b"window")
    torch.cuda.synchronize()
    assert bytes(t[8:14].cpu().tolist()) == b"window"
    assert be.close() == 1


def test_twin_rejects_misaligned_and_host_ranges():
    be = H.UserBackend()
    t = _buf(4 * PAGE)
    with pytest.raises(H.HarnessError):
        be.get_pages(t.data_ptr() + 4096, PAGE)
    with pytest.raises(H.HarnessError):
        be.get_pages(torch.zeros(PAGE * 2, dtype=torch.uint8).data_ptr() & ~(PAGE - 1), PAGE)
    be.close()


def test_reg_mr_dmabuf_mode_holds_a_pin(needs_dmabuf_export, ctx):
    import os
    t = _buf(1 << 20)
    mr = ctx.reg_mr(t, nbytes=1 << 20, mode="dmabuf")
    assert mr.dmabuf_fd >= 0 and os.fstat(mr.dmabuf_fd)
    fd = mr.dmabuf_fd
    mr.revoke()                                           # the pin goes with the memory
    with pytest.raises(OSError):
        os.fstat(fd)
    mr.dereg()
    mr2 = ctx.reg_mr(t, nbytes=1 << 20, mode="dmabuf")
    fd2 = mr2.dmabuf_fd
    mr2.dereg()
    with pytest.raises(OSError):
        os.fstat(fd2)


def test_probe_reports_this_box():
    from rocnrdma_b200 import probe
    r = probe.probe()
    assert len(r["gpus"]) >= 1 and r["gpus"][0]["caps"]["dmabuf"]
    assert r["plan"]["wire"] in ("softhca", "verbs")
