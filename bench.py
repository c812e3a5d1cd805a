#!/usr/bin/env python
"""Headline benchmark: GPU-initiated RDMA write GB/s on HBM buffers, each GPU driving its own HCA, next to the
host-posted and host-staged baselines measured in the same process (BASELINE.md section 3: B1 / B2 / P1).

Contract (driver): ``python bench.py --gpus N --steps K --warmup W`` (torchrun for N > 1) prints ONE JSON line from
rank 0.  One *step* = ONE launch of the sm_100a poster kernel, which builds ``msgs_per_step`` RDMA WRITE work requests
of ``--msg-bytes`` (default 256 MiB, larger than the 126 MB L2, rotating over 4 distinct buffers), rings the doorbell
for each and polls the completion queue on the device (window 8).  ``msgs_per_step`` is fixed before the timed region
from a calibration run so that the K timed steps last >= ``--min-seconds`` (default 1.2 s): long enough for the clock
record to mean something.  ``value`` is the whole-job aggregate GB/s, device-timed with CUDA events, max over ranks.

Wire (``--wire auto``): a ConnectX through libibverbs / mlx5dv when one is reachable (real /dev/infiniband + rdma-core;
then the same code measures BASELINE configs 1-3 on the NIC), else the software HCA: mlx5-format queues in HBM and a
persistent sm_100a DMA engine on ``--engine-ctas`` SMs (default 32: the engine stands in for a NIC and is deliberately
NOT given the whole GPU; ``extras.engine_128_ctas`` records what it reaches with 128).  This sandbox exposes no
/dev/infiniband, so the numbers the driver records are software-HCA numbers (``config.wire`` says so), and BASELINE.md
publishes no reference figure, hence ``vs_baseline: null``.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


_REAL_STDOUT = None


def quiet_stdout():
    """Library banners (NCCL prints its version to stdout under NCCL_DEBUG=VERSION) must not share stdout with the
    result: point fd 1 at stderr for the run and keep the original for the one JSON line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(obj):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def reference_arm():
    # `pip install --no-index ... /root/reference` fails: the reference is a Linux kernel module for
    # AMD KFD + MLNX_OFED 3.2 (no setup.py / pyproject, no userspace, needs amd_rdma.h); see DESIGN.md.
    if int(os.environ.get("RANK", "0")) != 0:      # launched like our own arm (torchrun for N > 1): one line, from rank 0
        return 0
    emit({"impl": "reference",
          "unavailable": "reference is an AMD-KFD/MLNX_OFED kernel module (amdp2p.ko): not pip-installable, "
                         "no userspace entry point, cannot build or load on a B200 box"})
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--wire", default="auto", help="auto | softhca | verbs")
    ap.add_argument("--msg-bytes", type=int, default=256 << 20)
    ap.add_argument("--engine-ctas", type=int, default=32)
    ap.add_argument("--window", type=int, default=8, help="work requests in flight per poster")
    ap.add_argument("--min-seconds", type=float, default=2.0, help="lower bound on the timed region (msgs_per_step is sized for it)")
    ap.add_argument("--msgs-per-step", type=int, default=0, help="0 = calibrate")
    ap.add_argument("--extras", type=int, default=1, help="also run baselines' siblings: ring, fused pack, small messages, GEMM, mock NIC")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step delivered (rank 0) as DIR/<name>.npy, to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return reference_arm()
    quiet_stdout()

    import torch
    import rocnrdma_b200 as rn
    from rocnrdma_b200 import _native as N, ops, wire as W
    from rocnrdma_b200.ops import pack as P
    from rocnrdma_b200.utils.clocks import ClockSampler, visible_gpu_index
    from rocnrdma_b200.utils import roofline as R

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        args.gpus = world
    warmup = max(args.warmup, 3)
    steps = args.steps
    if not torch.cuda.is_available():
        # the GPU-initiated path has no CPU fallback by design: say so in one line instead of a traceback
        if rank == 0:
            emit({"metric": "rdma_write_gbps_gpu_hbm_device_timed", "value": None, "impl": "ours",
                  "unavailable": "no CUDA device visible: the data path is sm_100a kernels only"})
        return 2
    torch.cuda.set_device(local_rank)
    from rocnrdma_b200.utils.affinity import bind_to_gpu
    cpus = bind_to_gpu(local_rank)          # pinned buffers get first-touched on the GPU's NUMA node
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier(device_ids=[local_rank])

    wire = rn.api.resolve_wire(args.wire)
    lib = N.load()
    msg = args.msg_bytes
    nslots = 4
    window = max(1, min(args.window, 16))
    dev = torch.device("cuda", local_rank)
    peaks = R.measured_peaks()
    ctx = rn.Context(device=local_rank, wire=wire)
    softhca = ctx.wire == "softhca"
    wire_desc = ("softhca: mlx5-format queues in HBM, persistent sm_100a DMA engine on %d SMs (no /dev/infiniband in this container; "
                 "the ConnectX backend is compiled in and selected automatically when a NIC is reachable)" % args.engine_ctas) if softhca else \
                ("verbs: %s through libibverbs/mlx5dv%s, GPU-posted into the NIC's own send queue" % (ctx.nic, " (MOCK provider)" if ctx.nic_is_mock else ""))

    # ---------------- everything that allocates happens before the engine starts (allocation stalls behind a resident kernel)
    src = torch.empty(msg * nslots, dtype=torch.uint8, device=dev)
    dst = torch.zeros(msg * nslots, dtype=torch.uint8, device=dev)
    ops.fill_random(src, seed=1000 + rank)
    host_in = torch.empty(msg, dtype=torch.uint8).pin_memory()       # e2e: step inputs live in pinned host memory
    host_in.random_(0, 255)
    bounce_a, bounce_b = torch.empty(msg, dtype=torch.uint8).pin_memory(), torch.empty(msg, dtype=torch.uint8).pin_memory()
    ms, md = ctx.reg_mr(src), ctx.reg_mr(dst)
    mba, mbb = ctx.reg_mr(bounce_a), ctx.reg_mr(bounce_b)
    qp = ctx.loopback_qp(depth=64)                                    # GPU-posted (product)
    hqp = ctx.loopback_qp(depth=64, mem=W.MEM_HOST_PINNED)            # host-posted (baselines B1 / B2)
    sm_qp = ctx.loopback_qp(depth=256, cq_depth=512)                  # small-message extras
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(8)]
    stream = ctx.stream
    out_a = ctx.scratch(64, 0)
    MR = rn.api.MemoryRegion
    mr_slot = [MR(ctx, ms.addr + i * msg, msg, ms.lkey, ms.access, rkey=ms.rkey) for i in range(nslots)]
    md_slot = [MR(ctx, md.addr + i * msg, msg, md.lkey, md.access, rkey=md.rkey) for i in range(nslots)]
    cmp_out = torch.zeros(1, dtype=torch.int64, device=dev)

    def device_compare(x, y):
        """Engine-safe byte compare: no allocation, work stream only (see the rule below)."""
        with torch.cuda.stream(stream):
            lib.rn_k_compare(stream.cuda_stream, x.data_ptr(), y.data_ptr(), x.numel() * x.element_size(), cmp_out.data_ptr())
            stream.synchronize()
            return int(cmp_out.item())

    gemm_bufs = {}
    if args.extras and rank == 0:
        for (M, Nn, K) in ((4096, 4096, 4096), (8192, 8192, 8192)):
            a = torch.randn(M, K, device=dev).to(torch.bfloat16); b = torch.randn(Nn, K, device=dev).to(torch.bfloat16)
            c = torch.zeros(M, Nn, device=dev, dtype=torch.bfloat16); d = torch.zeros_like(c)
            gemm_bufs[(M, Nn, K)] = (a, b, c, d, ctx.reg_mr(c), ctx.reg_mr(d))
    ring = None
    if world > 1 and softhca and args.extras:
        from rocnrdma_b200 import parallel
        rcq = ctx.create_cq(512)
        rqp = ctx.create_qp(rcq, ctx.create_cq(512), 256, 256)
        torch.cuda.synchronize()
        _, remote = parallel.connect_ring(ctx, rqp, [md])
        ring = (rqp, remote[md.key] if md.key in remote else list(remote.values())[0])
    torch.cuda.synchronize()
    barrier()

    def post(n_msgs, sync=True, w=window, q=qp, nbytes=msg, out=out_a):
        """ONE poster-kernel launch: n_msgs GPU-built WQEs over the rotating slots, device-polled completions."""
        return ops.rdma_stream(q, W.OP_RDMA_WRITE, ms, md, nbytes, iters=n_msgs, window=w, slot_stride=msg, nslots=nslots,
                               stream=stream, sync=sync, out=out, timeout_ms=10000)

    # Rule of the house while the engine kernel is resident: no default-stream work, no allocation, no device-wide
    # synchronize, no NCCL (each would wait for the persistent kernel: DESIGN.md 3.2).  Those happen between engine runs.
    def engine_on():
        ctx.engine_start(ctas=args.engine_ctas, idle_timeout_ms=20000)

    def engine_off():
        ctx.engine_stop()

    # ---------------- warm-up + calibration
    engine_on()
    r = post(8)
    assert r.ok, r.status
    r = post(16)
    assert r.ok, r.status
    engine_off()
    t = torch.tensor([r.device_ns / 16 / 1e9], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                      # every rank must do the same work per step
    per_msg_s = float(t.item())
    mps = args.msgs_per_step or max(1, int(args.min_seconds / (steps * per_msg_s) + 0.999))
    mps = min(mps, 4096)
    engine_on()
    for _ in range(warmup):
        r = post(mps)
        assert r.ok, r.status
    engine_off()
    dst.zero_()                                                       # verification below must see bytes moved by the timed region
    torch.cuda.synchronize()
    barrier()

    # ---------------- device-timed headline: exactly `steps` poster launches
    engine_on()
    r = post(min(mps, 8))                                             # the engine is resident and warm before the clock starts
    assert r.ok, r.status
    gpu_idx = visible_gpu_index(local_rank)
    sampler = ClockSampler(gpu_index=gpu_idx, period_s=0.1).start()
    t_wall0 = time.time()
    ev[0].record(stream)
    for _ in range(steps):
        post(mps, sync=False)
    ev[1].record(stream)
    ev[1].synchronize()
    dev_ms = ev[0].elapsed_time(ev[1])
    clocks = sampler.stop(skip_first_s=0.25)
    last = ops.rdma.parse_stream_out(out_a[1], 1, msg)
    assert last.ok and last.done == [mps], (last.status, last.done)
    counters = qp.counters()
    engine_off()
    # byte verification: every destination slot equals its source slot
    n_bad = sum(ops.compare(src[i * msg:(i + 1) * msg], dst[i * msg:(i + 1) * msg]) for i in range(nslots))
    if args.dump_outputs and rank == 0:                               # before the baselines below overwrite dst
        dump_outputs(args.dump_outputs, dst, msg, nslots, last, mps)

    # ---------------- baselines in the same process, same buffers, same wire
    base = {}
    n_base = max(8, min(mps, 64))
    with torch.cuda.stream(stream):                                   # (a) what the copy engines do with zero SMs
        for i in range(2):
            dst[:msg].copy_(src[:msg], non_blocking=True)
        ev[2].record()
        for i in range(n_base):
            s = i % nslots
            dst[s * msg:(s + 1) * msg].copy_(src[s * msg:(s + 1) * msg], non_blocking=True)
        ev[3].record()
    ev[3].synchronize()
    base["cudaMemcpyAsync_d2d_gbps"] = round(n_base * msg / (ev[2].elapsed_time(ev[3]) * 1e-3) / 1e9, 1)
    engine_on()
    ns, nerr = C.c_uint64(), C.c_uint32()
    try:                                                              # (b) B2: the host posts, the CPU polls (ib_write_bw on a GPU MR)
        if softhca:
            rc = lib.rn_host_stream(hqp._q, W.OP_RDMA_WRITE, ms.addr, ms.lkey, md.addr, md.rkey, msg, n_base, window, msg, nslots, 20000,
                                    C.byref(ns), C.byref(nerr))
        else:
            rc = lib.rn_verbs_host_stream(hqp._vq, W.OP_RDMA_WRITE, ms.addr, ms.lkey, md.addr, md.rkey, msg, n_base, window, msg, nslots, 20000,
                                          C.byref(ns), C.byref(nerr))
        base["host_posted_gbps"] = round(n_base * msg / ns.value, 1) if rc == 0 and nerr.value == 0 else None
    except Exception as e:
        base["host_posted_error"] = str(e)[:160]
    try:                                                              # (c) B1: D2H -> host MR -> RDMA -> host MR -> H2D per message
        n_st = 6
        if softhca:
            rc = lib.rn_host_staged_stream(hqp._q, src.data_ptr(), dst.data_ptr(), mba.addr, mba.lkey, mbb.addr, mbb.rkey, msg, n_st, msg,
                                           nslots, 20000, C.byref(ns))
        else:
            rc = lib.rn_verbs_host_staged_stream(hqp._vq, src.data_ptr(), dst.data_ptr(), mba.addr, mba.lkey, mbb.addr, mbb.rkey, msg, n_st,
                                                 msg, nslots, 20000, C.byref(ns))
        base["host_staged_gbps"] = round(n_st * msg / ns.value, 1) if rc == 0 else None
    except Exception as e:
        base["host_staged_error"] = str(e)[:160]

    # ---------------- end to end through the public API: pinned host -> H2D -> GPU-posted write -> status D2H
    with torch.cuda.stream(stream):                                   # H2D alone, for the breakdown
        src[:msg].copy_(host_in, non_blocking=True)
        ev[4].record()
        for i in range(4):
            src[(i % nslots) * msg:(i % nslots + 1) * msg].copy_(host_in, non_blocking=True)
        ev[5].record()
    ev[5].synchronize()
    h2d_gbps = 4 * msg / (ev[4].elapsed_time(ev[5]) * 1e-3) / 1e9
    e2e_steps = max(16, min(400, int(1.0 / (msg / (h2d_gbps * 1e9)) + 1)))
    with torch.cuda.stream(stream):
        for i in range(2):
            src[:msg].copy_(host_in, non_blocking=True)
            post(1)
        ev[6].record()
    # A two-deep pipeline, as a user streaming inputs would write it: message i's host -> device copy runs on the copy
    # stream while message i-1 is being written on the posting stream; every message's status words are read back on the
    # host (the write of slot s is known complete before slot s is copied over again: its status was read nslots - 1 steps ago).
    copy_stream = ctx.aux_stream
    copy_stream.wait_event(ev[6])
    outs = (out_a, ctx.scratch(64, 64))
    h2d_done = [torch.cuda.Event() for _ in range(2)]
    wr_done = [torch.cuda.Event() for _ in range(2)]
    for i in range(e2e_steps):
        s = i % nslots
        with torch.cuda.stream(copy_stream):
            src[s * msg:(s + 1) * msg].copy_(host_in, non_blocking=True)     # H2D of this message's input
            h2d_done[i & 1].record(copy_stream)
        stream.wait_event(h2d_done[i & 1])
        ops.rdma_stream(qp, W.OP_RDMA_WRITE, mr_slot[s], md_slot[s], msg, iters=1, stream=stream, sync=False, out=outs[i & 1])
        wr_done[i & 1].record(stream)
        if i >= 1:
            wr_done[(i - 1) & 1].synchronize()                               # result visible to the host: the 64 B of status / timing
            st = ops.rdma.parse_stream_out(outs[(i - 1) & 1][1], 1, msg)     # words the kernel wrote to mapped pinned memory
            assert st.ok, st.status
    wr_done[(e2e_steps - 1) & 1].synchronize()
    st = ops.rdma.parse_stream_out(outs[(e2e_steps - 1) & 1][1], 1, msg)
    assert st.ok, st.status
    with torch.cuda.stream(stream):
        ev[7].record()
    ev[7].synchronize()
    e2e_ms = ev[6].elapsed_time(ev[7])

    # ---------------- extras (never take the headline down)
    extras = {}
    ring_ns = 0.0
    if ring is not None:
        try:
            rqp, rmd = ring
            n_ring = max(16, int(0.5 / (msg / 600e9)))
            ops.rdma_stream(rqp, W.OP_RDMA_WRITE, ms, rmd, msg, iters=8, window=window, slot_stride=msg, nslots=nslots, stream=stream, timeout_ms=10000)
            rr = ops.rdma_stream(rqp, W.OP_RDMA_WRITE, ms, rmd, msg, iters=n_ring, window=window, slot_stride=msg, nslots=nslots, stream=stream,
                                 timeout_ms=10000)
            ring_ns = float(rr.device_ns) if rr.ok else 0.0
            extras["ring"] = {"ok": bool(rr.ok), "msgs": n_ring}
        except Exception as e:
            extras["ring"] = {"error": str(e)[:160]}
    if args.extras and rank == 0:
        try:   # fused bf16 -> fp8 pack + GPU-initiated write (config 3)
            n_el = min(1 << 28, (msg * nslots) // 2)
            n_el -= n_el % (1 << 22)
            chunk = 1 << 22
            nb = P.staging_bytes(n_el, chunk)
            if n_el >= (1 << 22) and 2 * nb <= msg * nslots:
                x = src[:2 * n_el].view(torch.bfloat16)
                stg = MR(ctx, md.addr, nb, md.lkey, md.access, rkey=md.rkey)
                rmt = MR(ctx, md.addr + (msg * nslots) // 2, nb, md.lkey, md.access, rkey=md.rkey)
                P.pack_fp8_write(ctx, x, stg, qp=qp, dst_mr=rmt, chunk_elems=chunk, signal_every=8)
                pr = min((P.pack_fp8_write(ctx, x, stg, qp=qp, dst_mr=rmt, chunk_elems=chunk, signal_every=8) for _ in range(3)),
                         key=lambda r: r.device_ns if r.ok else 1 << 62)      # best of 3 after one warm-up
                pack_bound = R.fused_pack_roofline_gbps(peaks)
                extras["fused_pack_fp8_write"] = {"elems": n_el, "ok": pr.ok, "device_us": round(pr.device_ns / 1e3, 1),
                                                  "source_bf16_gbps": round(pr.source_gbps, 1), "wire_fp8_gbps": round(pr.payload_gbps, 1),
                                                  "roofline_source_gbps": round(pack_bound, 1),
                                                  "frac_of_roofline": round(pr.source_gbps / pack_bound, 3),
                                                  "roofline_model": "algorithmic HBM bytes of the pack (2 B read + 1.03 B written per element) at the measured copy peak"}
        except Exception as e:
            extras["fused_pack_fp8_write"] = {"error": str(e)[:160]}
        try:   # the poster's own cost: single post / poll, and perftest-style post lists
            kw = dict(slot_stride=4096, nslots=64, stream=stream)
            ops.rdma_stream(sm_qp, W.OP_RDMA_WRITE, ms, md, 4096, iters=256, window=16, **kw)
            sm = ops.rdma_stream(sm_qp, W.OP_RDMA_WRITE, ms, md, 4096, iters=4096, window=16, **kw)
            ops.rdma_stream(sm_qp, W.OP_RDMA_WRITE, ms, md, 64, iters=32, window=1, stream=stream)
            lat = ops.rdma_stream(sm_qp, W.OP_RDMA_WRITE, ms, md, 64, iters=256, window=1, stream=stream)
            bkw = dict(window=32, burst=8, signal_every=8, stream=stream)
            ops.rdma_stream(sm_qp, W.OP_RDMA_WRITE, ms, md, 4096, iters=64, slot_stride=4096, nslots=64, **bkw)
            bm = ops.rdma_stream(sm_qp, W.OP_RDMA_WRITE, ms, md, 4096, iters=4096, slot_stride=4096, nslots=64, **bkw)
            extras["small_msg"] = {"4KiB_w16_us_per_msg": round(sm.us_per_msg, 3), "64B_latency_us": round(lat.us_per_msg, 2),
                                   "4KiB_burst8_us_per_msg": round(bm.us_per_msg, 3), "ok": bool(sm.ok and lat.ok and bm.ok)}
        except Exception as e:
            extras["small_msg"] = {"error": str(e)[:160]}
        try:   # K4 fused: panels RDMA-written from the GEMM epilogue vs GEMM-then-send, the engine holding its SMs
            gs = {}
            grid = 148 - args.engine_ctas if softhca else 0
            for (M, Nn, K), (a, b, c, d, cm, dm) in gemm_bufs.items():
                ops.gemm_send(ctx, a, b, c, c_mr=cm, qp=qp, dst_mr=dm, signal_every=4, grid=grid)
                f = min((ops.gemm_send(ctx, a, b, c, c_mr=cm, qp=qp, dst_mr=dm, signal_every=4, grid=grid) for _ in range(3)), key=lambda r: r.device_ns)
                fused_ok = bool(f.ok and device_compare(c, d) == 0)
                unf_us = 1e30
                for _ in range(3):
                    with torch.cuda.stream(stream):
                        ev[2].record()
                        ops.gemm_send(ctx, a, b, c, grid=grid, sync=False)
                        ops.rdma_stream(qp, W.OP_RDMA_WRITE, cm, dm, min(2 * M * Nn, (1 << 31) - 65536), iters=1, sync=False, stream=stream)
                        ev[3].record()
                    ev[3].synchronize()
                    unf_us = min(unf_us, ev[2].elapsed_time(ev[3]) * 1e3)
                gs[f"{M}x{Nn}x{K}"] = {"gemm_ctas": grid or 148, "fused_gemm_send_us": round(f.device_ns / 1e3, 1), "fused_tflops": round(f.tflops, 1),
                                       "gemm_then_send_us": round(unf_us, 1), "fused_speedup": round(unf_us / (f.device_ns / 1e3), 3),
                                       "fused_verified": fused_ok}
            extras["gemm_send"] = gs
        except Exception as e:
            extras["gemm_send"] = {"error": str(e)[:200]}
    if softhca:
        ctx.engine_stop()
    if args.extras and rank == 0 and gemm_bufs:
        try:   # K4 compute only, whole GPU, next to cuBLAS on the same box (library GEMM: the roofline reference only)
            sustained = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops")
            shapes = [(k, v[:3]) for k, v in gemm_bufs.items()]
            for (M, Nn, K) in ((8192, 8192, 2048), (16384, 4096, 1024)):      # the other two benchmark shapes, compute only (engine is off: allocation is safe)
                shapes.append(((M, Nn, K), (torch.randn(M, K, device=dev).to(torch.bfloat16), torch.randn(Nn, K, device=dev).to(torch.bfloat16),
                                            torch.zeros(M, Nn, device=dev, dtype=torch.bfloat16))))
            for (M, Nn, K), (a, b, c) in shapes:
                flops = 2.0 * M * Nn * K
                with torch.cuda.stream(stream):
                    for _ in range(3):
                        torch.matmul(a, b.T, out=c)
                    ev[2].record()
                    for _ in range(10):
                        torch.matmul(a, b.T, out=c)
                    ev[3].record()
                ev[3].synchronize()
                cublas = flops * 10 / (ev[2].elapsed_time(ev[3]) * 1e-3) / 1e12
                for _ in range(3):
                    ops.gemm_send(ctx, a, b, c)
                with torch.cuda.stream(stream):
                    ev[2].record()
                    for _ in range(10):
                        ops.gemm_send(ctx, a, b, c, sync=False, stream=stream)
                    ev[3].record()
                ev[3].synchronize()
                ours = flops * 10 / (ev[2].elapsed_time(ev[3]) * 1e-3) / 1e12
                singles = [ops.gemm_send(ctx, a, b, c) for _ in range(5)]
                best = max(r.tflops for r in singles)
                ref = a.float()[:256] @ b.float().T
                good = bool(torch.allclose(c[:256].float(), ref, rtol=2e-2, atol=2.0))
                row = extras.setdefault("gemm_send", {}).setdefault(f"{M}x{Nn}x{K}", {})
                row.update({"cublas_tflops": round(cublas, 1), "ours_tflops": round(ours, 1), "ours_best_single_launch_tflops": round(best, 1),
                            "vs_cublas": round(ours / cublas, 3), "frac_of_sustained_peak": round(ours / sustained, 3) if sustained else None,
                            "kernel": {1: "single CTA (128x256)", 2: "CTA pair (256x256 per pair)", 3: "wide CTA pair (512x256 per pair)"}.get(singles[0].variant, "?"),
                            "timing": "10 back-to-back launches between CUDA events, both libraries", "numerics_ok": good})
                if (M, Nn, K) not in gemm_bufs:
                    continue
                # K7: the same product with block-scaled fp8 operands (what a receiver of K3 / K4 records multiplies)
                from rocnrdma_b200.ops import gemm_mx as MX
                (aq, as_), (bq, bs) = MX.quantize_mx(a), MX.quantize_mx(b)
                oa, ob = MX.MxOperand.from_tensors(aq, as_), MX.MxOperand.from_tensors(bq, bs)
                for _ in range(2):
                    ops.gemm_mxfp8(ctx, oa, ob, c)
                with torch.cuda.stream(stream):
                    ev[2].record()
                    for _ in range(10):
                        ops.gemm_mxfp8(ctx, oa, ob, c, sync=False, stream=stream)
                    ev[3].record()
                ev[3].synchronize()
                mx = flops * 10 / (ev[2].elapsed_time(ev[3]) * 1e-3) / 1e12
                refq = MX.dequantize_mx(aq[:128], as_[:128]) @ MX.dequantize_mx(bq, bs).T
                row.update({"mxfp8_block_scaled_tflops": round(mx, 1),
                            "mxfp8_numerics_ok": bool((c[:128].float() - refq).abs().max().item() <= 2e-2 * refq.abs().max().item() + 1e-3)})
                del aq, as_, bq, bs
        except Exception as e:
            extras.setdefault("gemm_send", {})["compute_only_error"] = str(e)[:200]
    if softhca:
        if args.extras:
            try:   # the emulator at its copy-peak configuration, for continuity with round 1 (not the default: see module docstring)
                ctx.engine_start(ctas=128, idle_timeout_ms=15000)
                post(8)
                r128 = post(64)
                ctx.engine_stop()
                extras["engine_128_ctas"] = {"gbps": round(r128.gbps, 1), "ok": r128.ok,
                                             "frac_of_measured_copy_peak": round(r128.gbps / R.copy_roofline_gbps(peaks), 3)}
            except Exception as e:
                extras["engine_128_ctas"] = {"error": str(e)[:160]}
    torch.cuda.synchronize()
    if args.extras and world > 1 and softhca:
        # BASELINE config 4 at N >= 2: GEMM on GPU0, every finished panel lands in GPU1's HBM over NVLink, consumer kernel
        # on GPU1 polls the receive CQ.  One process drives both GPUs (two HCA contexts, QP to QP), so rank 0 runs it while
        # the other ranks wait on the host (a NCCL barrier would put a spinning kernel of another process on GPU1).
        store = torch.distributed.distributed_c10d._get_default_store()
        if rank == 0:
            try:
                from rocnrdma_b200.models import sendrecv_gemm as SG
                res = {}
                for shape, mode in (((8192, 8192, 2048), "engine"), ((4096, 4096, 4096), "direct")):
                    r4 = SG.run(*shape, mode=mode, gpus=(local_rank, local_rank + 1), reps=3)
                    res["x".join(str(v) for v in shape)] = {
                        "mode": r4.mode, "ok": bool(r4.ok and r4.verified), "fused_gemm_send_recv_us": round(r4.fused_us, 1),
                        "gemm_then_write_us": round(r4.unfused_us, 1), "fused_speedup": round(r4.unfused_us / r4.fused_us, 3),
                        "tflops_incl_delivery": round(r4.tflops, 1), "wire_gbps": round(r4.wire_gbps, 1), "panels": r4.panels,
                        "engine_ctas": r4.engine_ctas,
                        "limiter": ("NVLink store burstiness: all GEMM CTAs reach their epilogue together (~450 GB/s of SM-issued stores)"
                                    if r4.mode == "direct" else "the 32 SMs the engine takes from the GEMM")}
                # the same wire fused into BOTH GEMMs: GPU0's epilogue sends fp8 panel records, GPU1's block-scaled GEMM starts tiles on arrival
                ch = SG.run_chain(8192, 8192, 2048, 8192, gpus=(local_rank, local_rank + 1), reps=3)
                res["chain_8192x8192x2048_then_x8192"] = {
                    "ok": bool(ch["verified"]), "fused_us": round(ch["fused_us"], 1) if ch["fused_us"] else None,
                    "sequential_us": round(ch["sequential_us"], 1) if ch["sequential_us"] else None,
                    "fused_speedup": round(ch["speedup"], 3) if ch["speedup"] else None, "wire_bytes": ch["wire_bytes"],
                    "timing": "host wall clock, launch to completion on both GPUs (no common device clock), best of 3",
                    "what": ch["what"], "limiter": "GEMM 2 cannot finish before GEMM 1's last panel arrives; GEMM 1 runs on 116 SMs next to the engine"}
                extras["config4_gemm_send_recv_nvlink"] = res
            except Exception as e:
                extras["config4_gemm_send_recv_nvlink"] = {"error": str(e)[:200]}
            finally:
                store.set("rn_cfg4_done", "1")
        else:
            store.wait(["rn_cfg4_done"])
    if args.extras and rank == 0 and softhca:
        try:   # the ConnectX code path, executed: same kernels, verbs wire, the in-tree mock provider as the NIC
            extras["verbs_wire_mock_nic"] = mock_nic_extra(rn, ops, W, N, C, local_rank, src, dst)
        except Exception as e:
            extras["verbs_wire_mock_nic"] = {"error": str(e)[:200]}
    barrier()

    # ---------------- max over ranks
    t = torch.tensor([dev_ms, e2e_ms, ring_ns, float(n_bad)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_ms_max, ring_ns_max, n_bad_max = t.tolist()
    ok = counters["n_err"] == 0 and counters["n_db_order_violations"] == 0 and n_bad_max == 0
    if rank == 0:
        total_bytes = msg * mps * steps * world
        value = total_bytes / (dev_ms_max * 1e-3) / 1e9
        e2e_value = msg * e2e_steps * world / (e2e_ms_max * 1e-3) / 1e9
        per_gpu = value / world
        if "ring" in extras and ring_ns_max > 0:
            per = msg * extras["ring"]["msgs"] / ring_ns_max
            extras["ring"].update({"per_gpu_gbps": round(per, 1), "aggregate_gbps": round(per * world, 1), "roofline_per_gpu_gbps": R.NVLINK_PEER_GBS,
                                   "frac_of_nvlink_roofline": round(per / R.NVLINK_PEER_GBS, 3),
                                   "what": "rank r GPU-posts RDMA writes into rank r+1's HBM (QPs connected through CUDA IPC; the engine moves the bytes over NVLink)",
                                   "limiter": "the posting GPU's engine CTAs issuing NVLink stores (32 SMs)"})
        for k in ("host_posted_gbps", "host_staged_gbps", "cudaMemcpyAsync_d2d_gbps"):
            if base.get(k):
                base["vs_" + k.replace("_gbps", "")] = round(per_gpu / base[k], 2)
        out = {
            "metric": "rdma_write_gbps_gpu_hbm_device_timed",
            "value": round(value, 2), "unit": "GB/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": round(dev_ms_max / steps, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bytes (payload-agnostic; fused extras are bf16 / bf16->fp8)", "data": "synthetic",
            "impl": "ours",
            "config": {"model": "gpu_initiated_rdma_write_loopback", "msg_bytes": msg, "msgs_per_step": mps, "global_batch": world * mps,
                       "seq_len": msg, "parallelism": f"{world}x(GPU+own HCA), loopback per GPU (BASELINE config 5 shape)",
                       "wire": wire_desc, "engine_ctas": args.engine_ctas if softhca else None, "window": window,
                       "step": f"one poster-kernel launch = {mps} GPU-built RDMA WRITE WQEs of {msg >> 20} MiB (doorbell per WQE, device-polled CQ, window {window})",
                       "poster": "sm_100a kernel: WQE + doorbell record + doorbell register + device CQ poll, queue state in registers",
                       "l2_policy": f"inputs larger than L2: {msg >> 20} MiB messages rotating over {nslots} buffers",
                       "timing": "CUDA events on the posting stream around exactly `steps` launches, max over ranks",
                       "timed_region_s": round(dev_ms_max / 1e3, 3), "wall_s": round(time.time() - t_wall0, 1)},
            "roofline": {"bound_gbps_per_gpu": round(R.copy_roofline_gbps(peaks), 1),
                         "frac_of_measured_copy_peak": round(per_gpu / R.copy_roofline_gbps(peaks), 3),
                         "peaks_source": peaks.get("_source"),
                         "limiter": "softhca: the DMA engine's SM count (~38 GB/s per engine CTA; 32 of 148 SMs by choice)" if softhca else "NIC line rate / PCIe Gen5 x16"},
            "baselines": base,
            "e2e": {"value": round(e2e_value, 2), "unit": "GB/s", "h2d_bytes_per_step": msg, "d2h_bytes_per_step": 64, "steps": e2e_steps,
                    "step": "one message: H2D of its input from pinned host memory, one GPU-posted RDMA WRITE, status words read back on the host; two messages in flight (copy of i overlaps the write of i-1)",
                    "h2d_only_gbps": round(h2d_gbps, 1), "cpu_affinity": f"{len(cpus)} cpus local to the GPU" if cpus else "unbound",
                    "limiter": "host -> device copy over PCIe Gen5 x16",
                    "path": "pinned host -> cudaMemcpyAsync H2D -> GPU-posted RDMA write -> status words in mapped pinned memory"},
            "gpu_launches": steps,
            "gpu_launches_note": f"one rdma_stream_kernel launch per step ({mps} WQEs each); the DMA engine is one persistent kernel launched before the timed region",
            "clocks": {"sm_mhz": clocks.get("sm_mhz"), "sm_max_mhz": clocks.get("sm_max_mhz"), "reasons": clocks.get("reasons", []),
                       "samples": clocks.get("samples", 0), "gpu_index": gpu_idx},
            "verified": bool(ok), "verification": {"mismatching_16B_words": int(n_bad_max), "bytes_compared_per_gpu": msg * nslots,
                                                   "error_cqes": counters["n_err"], "doorbell_order_violations": counters["n_db_order_violations"]},
            "extras": extras,
        }
        emit(out)
    if dist is not None:
        dist.destroy_process_group()
    ctx.close()
    return 0


def dump_outputs(path, dst, msg, nslots, last, mps):
    """What the last timed step delivered, as float arrays under ``path``: a fixed, seeded sample of 4 Mi destination bytes
    (16 MB), the exact byte sum of every destination slot, and the step's completion status.  The source bytes are
    seeded, so with the same arguments two builds must write the same files.  The message count per step follows the
    calibration unless ``--msgs-per-step`` fixes it, so the status records the completed fraction, not the count."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    n = msg * nslots
    idx = torch.randint(0, n, (min(n, 1 << 22),), generator=torch.Generator().manual_seed(0)).sort().values
    np.save(os.path.join(path, "dst_bytes_sample.npy"), dst[idx.to(dst.device)].float().cpu().numpy())
    sums = [float(dst[s * msg:(s + 1) * msg].sum(dtype=torch.int64)) for s in range(nslots)]
    np.save(os.path.join(path, "dst_slot_byte_sums.npy"), np.array(sums, dtype=np.float64))
    np.save(os.path.join(path, "last_step_status.npy"), np.array([float(last.ok), sum(last.done) / mps], dtype=np.float64))


def mock_nic_extra(rn, ops, W, N, C, device, src, dst):
    """P1 / B2 / B1 through the verbs wire with the mock provider as the NIC (host thread, DMA by cuMemcpyAsync): the
    exact code path a ConnectX takes -- ibv_reg_mr / ibv_reg_dmabuf_mr on HBM, mlx5dv queues mapped into the GPU,
    rdma_stream_kernel posting into them.  Bandwidth here is the mock's, reported only to show the path runs."""
    import torch
    lib = N.load()
    if lib.rn_verbs_available() <= 0 or not lib.rn_verbs_is_mock():
        # the provider is dlopen()ed once per process; a run that already resolved the system libraries cannot switch
        return {"skipped": "mock provider not selected in this process (set ROCNRDMA_VERBS_LIBDIR=rocnrdma_b200/lib/mock)",
                "why": lib.rn_verbs_why().decode(errors="replace")}
    c = rn.Context(device=device, wire="verbs", nic=device)
    try:
        m = 64 << 20
        ms, md = c.reg_mr(src[:4 * m], mode="auto"), c.reg_mr(dst[:4 * m], mode="auto")
        gq = c.loopback_qp(depth=32)
        hq = c.loopback_qp(depth=32, mem=W.MEM_HOST_PINNED)
        dst[:4 * m].zero_()
        torch.cuda.synchronize()
        ops.rdma_stream(gq, W.OP_RDMA_WRITE, ms, md, m, iters=4, window=4, slot_stride=m, nslots=4, timeout_ms=10000)
        r = ops.rdma_stream(gq, W.OP_RDMA_WRITE, ms, md, m, iters=32, window=4, slot_stride=m, nslots=4, timeout_ms=10000)
        good = ops.compare(src[:4 * m], dst[:4 * m]) == 0
        ns, ne = C.c_uint64(), C.c_uint32()
        rc = lib.rn_verbs_host_stream(hq._vq, W.OP_RDMA_WRITE, ms.addr, ms.lkey, md.addr, md.rkey, m, 32, 4, m, 4, 10000, C.byref(ns), C.byref(ne))
        sm = ops.rdma_stream(gq, W.OP_RDMA_WRITE, ms, md, 4096, iters=512, window=16, slot_stride=4096, nslots=64, timeout_ms=10000)
        cnt = gq.counters()
        return {"nic": c.nic, "registration": ms.mode, "gpu_posted_64MiB_gbps": round(r.gbps, 1), "gpu_posted_ok": bool(r.ok and good),
                "host_posted_64MiB_gbps": round(32 * m / ns.value, 1) if rc == 0 and ne.value == 0 else None,
                "gpu_posted_4KiB_us_per_msg": round(sm.us_per_msg, 2), "doorbell_via_cpu_proxy": gq.db_proxy,
                "nic_counters": {k: cnt[k] for k in ("n_wqe", "n_err", "n_db_order_violations", "n_doorbells")},
                "note": "mock NIC = host thread + cuMemcpyAsync; numbers are the mock's, the code path is the ConnectX one"}
    finally:
        c.close()


if __name__ == "__main__":
    # the mock provider is only ever used for the clearly-labelled extra; a real rdma-core on the box wins
    if not os.environ.get("ROCNRDMA_VERBS_LIBDIR") and not os.path.exists("/dev/infiniband"):
        os.environ["ROCNRDMA_VERBS_LIBDIR"] = os.path.join(os.path.dirname(os.path.abspath(__file__)), "rocnrdma_b200", "lib", "mock")
    sys.exit(main())
