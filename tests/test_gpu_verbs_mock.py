"""GPU tier: the verbs wire on a real B200 against the mock provider -- HBM registered with the (mock) HCA the
three ways, host-posted baselines on GPU MRs, and the product path: the mlx5dv queues of a QP mapped into the GPU
and driven by the SAME sm_100a kernels that drive the software HCA (rdma_stream_kernel, pack_fp8_write_kernel,
gemm_send2_kernel), directly and through the CPU doorbell proxy.  The NIC here is a host thread that DMAs with
cuMemcpyAsync; nothing else about the path differs from a ConnectX."""
import os

import pytest
import torch

import rocnrdma_b200 as rn
from rocnrdma_b200 import _native as N, ops, wire as W

pytestmark = pytest.mark.gpu


@pytest.fixture
def vctx():
    c = rn.Context(device=0, wire="verbs", nic=0)
    assert c.nic_is_mock
    yield c
    c.close()


def _bufs(n):
    src = torch.empty(n, dtype=torch.uint8, device="cuda:0")
    dst = torch.zeros(n, dtype=torch.uint8, device="cuda:0")
    ops.fill_random(src, seed=99)
    torch.cuda.synchronize()
    return src, dst


@pytest.mark.parametrize("mode", ["peermem", "dmabuf", "auto"])
def test_host_posted_write_on_hbm_mrs(request, dmabuf_export_error, vctx, mode):
    """BASELINE config 2 shape: cudaMalloc HBM registered with the HCA, host-posted RDMA write, CPU-polled CQ.  ``auto``
    takes the dma-buf where the driver exports one and falls back to the peer-memory client where it does not."""
    if mode == "dmabuf":
        request.getfixturevalue("needs_dmabuf_export")
    n = 1 << 20
    src, dst = _bufs(n)
    ms, md = vctx.reg_mr(src, mode=mode), vctx.reg_mr(dst, mode=mode)
    assert ms.mode == ("dmabuf" if mode == "dmabuf" or (mode == "auto" and dmabuf_export_error is None) else "peermem")
    assert (ms.dmabuf_fd >= 0) == (ms.mode == "dmabuf")
    qp = vctx.loopback_qp(depth=16, mem=W.MEM_HOST_PINNED)
    assert not qp.on_gpu
    qp.post_write(ms, md, n)
    wc = qp.scq.wait(1)[0]
    assert wc.status == "OK" and wc.byte_cnt == n
    assert ops.compare(src, dst) == 0
    qp.post_read(md, ms, 4096, local_off=0, remote_off=8192)      # READ: local = dst[0:4096] <- remote = src[8192:...]
    assert qp.scq.wait(1)[0].status == "OK"
    assert torch.equal(dst[:4096], src[8192:8192 + 4096])
    ms.dereg(); md.dereg()
    assert ms.state == "FREE" and ms.dmabuf_fd == -1


def test_gpu_pointer_without_peer_memory_client_is_refused(vctx, monkeypatch):
    src, _ = _bufs(1 << 16)
    monkeypatch.setenv("ROCNRDMA_MOCK_PEERMEM", "0")
    with pytest.raises(N.NativeError, match="no peer-memory client"):
        vctx.reg_mr(src, mode="peermem")
    host = torch.empty(4096, dtype=torch.uint8)
    assert vctx.reg_mr(host, mode="peermem").state == "PINNED"     # host memory never needed one


@pytest.mark.parametrize("nbytes,iters,window", [(64, 40, 1), (4096, 100, 8), (1 << 20, 12, 4), ((1 << 20) + 3, 3, 2)])
def test_gpu_initiated_write_into_mlx5dv_queues(vctx, nbytes, iters, window):
    """K1 on the verbs wire: the kernel writes WQEs into the NIC's send queue (host memory, mapped), updates the
    doorbell record, stores to the BlueFlame register and polls the NIC's CQ -- no host in the loop."""
    src, dst = _bufs(nbytes + 64)
    ms, md = vctx.reg_mr(src), vctx.reg_mr(dst)
    qp = vctx.loopback_qp(depth=16)                 # mem=MEM_DEVICE: GPU-posted
    assert qp.on_gpu and rn.api.N.load().rn_qp_is_adopted(qp._q) == 1
    r = ops.rdma_stream(qp, W.OP_RDMA_WRITE, ms, md, nbytes, iters=iters, window=window, timeout_ms=5000)
    assert r.ok and r.done == [iters], r.status
    assert torch.equal(src[:nbytes], dst[:nbytes]) and int(dst[nbytes:].sum()) == 0
    c = qp.counters()
    assert c["nic"] == "mock" and c["n_wqe"] == iters and c["n_err"] == 0 and c["n_db_order_violations"] == 0
    assert c["sq_cons"] == iters and c["cq_overruns"] == 0
    with pytest.raises(N.NativeError, match="owned by the GPU poster"):
        qp.post_write(ms, md, 8)


def test_gpu_initiated_read_send_and_bursts(vctx):
    n = 1 << 16
    src, dst = _bufs(n)
    ms, md = vctx.reg_mr(src), vctx.reg_mr(dst)
    qp = vctx.loopback_qp(depth=64)
    r = ops.rdma_stream(qp, W.OP_RDMA_READ, md, ms, 4096, iters=8, slot_stride=4096, nslots=8, window=4, timeout_ms=5000)
    assert r.ok, r.status
    assert torch.equal(dst[:8 * 4096], src[:8 * 4096])
    # perftest-style post lists: 8 WQEs per doorbell, one CQE per 8
    dst.zero_()
    r = ops.rdma_stream(qp, W.OP_RDMA_WRITE, ms, md, 1024, iters=64, slot_stride=1024, nslots=64, window=32, burst=8, signal_every=8,
                        timeout_ms=5000)
    assert r.ok and r.done == [64], r.status
    assert torch.equal(dst, src)
    c = qp.counters()
    assert c["n_doorbells"] <= 8 + 8 + 2 and c["n_db_order_violations"] == 0, c
    # an error completion reaches the device poller and fails the QP
    bad = rn.api.MemoryRegion(vctx, md.addr, md.length, 0x5555, md.access)
    r = ops.rdma_stream(qp, W.OP_RDMA_WRITE, ms, bad, 64, iters=1, timeout_ms=3000)
    assert r.status == ["CQE_ERROR"] and qp.state == "ERR"


def test_doorbell_through_the_cpu_proxy(monkeypatch):
    """What runs when the driver refuses to map the UAR page (cudaHostRegisterIoMemory): WQE + doorbell record are
    still written by the GPU, a host thread forwards the 8-byte doorbell."""
    monkeypatch.setenv("ROCNRDMA_DB_PROXY", "1")
    c = rn.Context(device=0, wire="verbs", nic=1)
    try:
        src, dst = _bufs(1 << 16)
        ms, md = c.reg_mr(src), c.reg_mr(dst)
        qp = c.loopback_qp(depth=16)
        assert qp.db_proxy
        r = ops.rdma_stream(qp, W.OP_RDMA_WRITE, ms, md, 8192, iters=8, slot_stride=8192, nslots=8, window=4, timeout_ms=5000)
        assert r.ok, r.status
        assert torch.equal(src, dst)
        assert qp.counters()["db_proxy_forwarded"] >= 2
    finally:
        c.close()


@pytest.mark.parametrize("with_imm", [False, True])
def test_fused_pack_posts_to_the_nic(vctx, with_imm):
    """K3 on the verbs wire: every CTA that completes a record posts its own WQE into the shared mlx5 send queue."""
    chunk = 1 << 16
    x = torch.randn(1 << 20, device="cuda:0").to(torch.bfloat16)
    nb = ops.staging_bytes(x.numel(), chunk)
    stg = torch.zeros(nb, dtype=torch.uint8, device="cuda:0")
    rem = torch.zeros(nb, dtype=torch.uint8, device="cuda:0")
    smr, rmr = vctx.reg_mr(stg), vctx.reg_mr(rem)
    qp = vctx.loopback_qp(depth=64)
    if with_imm:
        scratch = torch.zeros(64, dtype=torch.uint8, device="cuda:0")
        rq = vctx.reg_mr(scratch)
        for _ in range(x.numel() // chunk):
            qp._vcheck(vctx._lib.rn_verbs_post_recv(qp._vq, rq.addr, rq.lkey, 64, None), "post_recv")   # receive posting stays a host verb
    pr = ops.pack_fp8_write(vctx, x, smr, qp=qp, dst_mr=rmr, chunk_elems=chunk, with_imm=with_imm, signal_every=4, timeout_ms=5000)
    assert pr.ok, pr.status
    assert torch.equal(rem, ops.ref_pack_fp8(x, chunk))
    if with_imm:
        y = torch.zeros_like(x)
        u = ops.unpack_fp8(vctx, rem, y, chunk_elems=chunk, qp=qp, timeout_ms=5000)      # waits on the NIC's receive CQ from the device
        assert u["status"] == "OK" and u["records_seen"] == x.numel() // chunk
        assert torch.equal(y, ops.ref_unpack_fp8(rem, x.numel(), chunk))
    assert qp.counters()["n_db_order_violations"] == 0


def test_gemm_epilogue_posts_panels_to_the_nic(vctx):
    """K4 on the verbs wire."""
    M, Nn, K = 512, 512, 256
    a = torch.randn(M, K, device="cuda:0").to(torch.bfloat16)
    b = torch.randn(Nn, K, device="cuda:0").to(torch.bfloat16)
    c = torch.zeros(M, Nn, device="cuda:0", dtype=torch.bfloat16)
    d = torch.zeros_like(c)
    cm, dm = vctx.reg_mr(c), vctx.reg_mr(d)
    qp = vctx.loopback_qp(depth=64)
    gr = ops.gemm_send(vctx, a, b, c, c_mr=cm, qp=qp, dst_mr=dm, timeout_ms=5000)
    assert gr.ok, gr.status
    ref = a.float() @ b.float().T
    assert torch.allclose(d.float(), ref, rtol=2e-2, atol=0.5)
    assert qp.counters()["n_wqe"] == M // 128 + 1


def test_host_staged_and_host_posted_baselines(vctx):
    """B1 (cudaMemcpy D2H -> host MRs -> H2D) and B2 (host-posted on HBM MRs) run as one-call streams."""
    import ctypes as C
    n, iters = 1 << 20, 8
    src, dst = _bufs(n * 2)
    ms, md = vctx.reg_mr(src), vctx.reg_mr(dst)
    ha, hb = torch.empty(n, dtype=torch.uint8).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory()
    ma, mb = vctx.reg_mr(ha), vctx.reg_mr(hb)
    qp = vctx.loopback_qp(depth=16, mem=W.MEM_HOST_PINNED)
    ns, err = C.c_uint64(), C.c_uint32()
    lib = vctx._lib
    assert lib.rn_verbs_host_stream(qp._vq, W.OP_RDMA_WRITE, ms.addr, ms.lkey, md.addr, md.rkey, n, iters, 4, n, 2, 5000,
                                    C.byref(ns), C.byref(err)) == 0, lib.rn_verbs_why()
    assert err.value == 0 and ns.value > 0 and ops.compare(src, dst) == 0
    dst.zero_()
    assert lib.rn_verbs_host_staged_stream(qp._vq, src.data_ptr(), dst.data_ptr(), ma.addr, ma.lkey, mb.addr, mb.rkey, n, iters, n, 2,
                                           5000, C.byref(ns)) == 0, lib.rn_verbs_why()
    assert ops.compare(src, dst) == 0


def test_bridged_registration_of_real_hbm_and_revocation(vctx, monkeypatch):
    """ibv_reg_mr on a cudaMalloc pointer answered by kmod/b200p2p.c (under kmod/shim): bus addresses in the MR,
    DMA through them, and the module's free callback invalidating the MR."""
    monkeypatch.setenv("ROCNRDMA_MOCK_PEERMEM", "b200p2p")
    lib = vctx._lib
    assert lib.rn_verbs_mock_bridge_status() == b"ok", lib.rn_verbs_mock_bridge_status()
    src, dst = _bufs(1 << 20)
    ms, md = vctx.reg_mr(src, mode="peermem"), vctx.reg_mr(dst, mode="peermem")
    qp = vctx.loopback_qp(depth=16)
    r = ops.rdma_stream(qp, W.OP_RDMA_WRITE, ms, md, 1 << 20, iters=1, timeout_ms=5000)
    assert r.ok and ops.compare(src, dst) == 0
    # the GPU driver revokes the pins of dst's allocation (what cudaFree does): the next access must fail cleanly
    base = dst.untyped_storage().data_ptr() & ~65535
    import ctypes as C
    ab, asz = C.c_uint64(), C.c_uint64()
    lib.rn_alloc_range(dst.data_ptr(), C.byref(ab), C.byref(asz))
    assert lib.rn_verbs_mock_gpu_free(ab.value & ~65535) >= 1
    r = ops.rdma_stream(qp, W.OP_RDMA_WRITE, ms, md, 4096, iters=1, timeout_ms=3000)
    assert r.status == ["CQE_ERROR"]
    md.dereg(); ms.dereg()
    assert base
