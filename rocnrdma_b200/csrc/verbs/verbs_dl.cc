// N2 / N3 real-NIC backend: a ConnectX driven through libibverbs + mlx5dv -- the wire the software
// HCA stands in for.  Compiled in EVERY build against the self-written ABI declarations in
// verbs/abi/verbs_abi.h; the libraries themselves are only ever dlopen()ed, so nothing links against
// rdma-core.  ROCNRDMA_VERBS_LIBDIR selects where libibverbs.so.1 / libmlx5.so.1 come from: unset = the
// system's (a box with MLNX_OFED / rdma-core and /dev/infiniband), or lib/mock for the in-tree mock
// provider (csrc/mockverbs), which is how this file runs in CI on a box without a NIC.
//
// What it provides (flat C ABI, rn_verbs_*):
//   * device enumeration / open / PD / port + GID query;
//   * memory registration in the three ways GPU memory reaches an HCA: ibv_reg_mr on the pointer (host
//     memory, or HBM through a peer-memory client -- nvidia-peermem or kmod/b200p2p.ko: the reference's
//     whole purpose, README.md:5-6, amdp2p.c:363-371) and ibv_reg_dmabuf_mr on an exported dma-buf fd;
//   * CQ / RC QP creation, RESET -> INIT -> RTR -> RTS towards a (lid | gid, qpn) -- loopback, port to
//     port, or a remote host -- host-posted WRITE / WRITE_IMM / READ / SEND / SEND_IMM, receive posting,
//     CQ polling: the "IB verbs" the reference tells its users to use (README.md:67) and the baselines
//     B0 / B1 / B2 of BASELINE.md (host-DRAM loopback, host-staged, host-posted on a GPU MR);
//   * mlx5dv_init_obj() + cudaHostRegister(): the raw SQ / RQ / CQ / doorbell-record memory and the
//     BlueFlame doorbell register of a QP mapped into the GPU's address space, so the device-side poster
//     (hca/post.cuh) writes WQEs, rings the doorbell and polls the CQ itself (IBGDA; K1 / K2).  When the
//     driver refuses to map the UAR page (cudaHostRegisterIoMemory needs PeerMappingOverride on some
//     platforms) a CPU proxy thread forwards the 8-byte doorbell value from a pinned mailbox to the
//     register: the GPU still builds the WQE and the doorbell record, the host only pokes the BAR.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <errno.h>
#include <sched.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

#include <atomic>
#include <map>
#include <mutex>
#include <thread>
#include <vector>

#include "abi/verbs_abi.h"

using namespace rnabi;

#define RN_API extern "C" __attribute__((visibility("default")))

namespace {

thread_local char g_why[384] = "";
int why(int rc, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_why, sizeof g_why, fmt, ap);
  va_end(ap);
  return rc;
}
uint64_t now_ns() {
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return (uint64_t)ts.tv_sec * 1000000000ull + (uint64_t)ts.tv_nsec;
}
bool uverbs_nodes_present() { return access("/dev/infiniband", R_OK | X_OK) == 0; }

struct Api {
  void* verbs = nullptr;
  void* mlx5 = nullptr;
  bool ok = false, is_mock = false, tried = false;
  char libdir[256] = "";
  ibv_device** (*get_device_list)(int*) = nullptr;
  void (*free_device_list)(ibv_device**) = nullptr;
  const char* (*get_device_name)(ibv_device*) = nullptr;
  ibv_context* (*open_device)(ibv_device*) = nullptr;
  int (*close_device)(ibv_context*) = nullptr;
  ibv_pd* (*alloc_pd)(ibv_context*) = nullptr;
  int (*dealloc_pd)(ibv_pd*) = nullptr;
  ibv_mr* (*reg_mr)(ibv_pd*, void*, size_t, int) = nullptr;
  ibv_mr* (*reg_dmabuf_mr)(ibv_pd*, uint64_t, size_t, uint64_t, int, int) = nullptr;
  int (*dereg_mr)(ibv_mr*) = nullptr;
  ibv_cq* (*create_cq)(ibv_context*, int, void*, ibv_comp_channel*, int) = nullptr;
  int (*destroy_cq)(ibv_cq*) = nullptr;
  ibv_qp* (*create_qp)(ibv_pd*, ibv_qp_init_attr*) = nullptr;
  int (*destroy_qp)(ibv_qp*) = nullptr;
  int (*modify_qp)(ibv_qp*, ibv_qp_attr*, int) = nullptr;
  int (*query_port)(ibv_context*, uint8_t, ibv_port_attr*) = nullptr;
  int (*query_gid)(ibv_context*, uint8_t, int, ibv_gid*) = nullptr;
  int (*dv_init_obj)(mlx5dv_obj*, uint64_t) = nullptr;
  // mock control plane (null on a real library)
  int (*mock_qp_stats)(ibv_qp*, void*) = nullptr;
  int (*mock_declare_gpu_range)(uint64_t, uint64_t) = nullptr;
  int (*mock_gpu_free)(uint64_t) = nullptr;
  void (*mock_set_rnr_timeout_ms)(uint64_t) = nullptr;
  const char* (*mock_bridge_status)() = nullptr;
};
std::mutex g_api_mu;
Api& api() {
  static Api a;
  std::lock_guard<std::mutex> g(g_api_mu);
  if (a.tried) return a;
  a.tried = true;
  const char* dir = getenv("ROCNRDMA_VERBS_LIBDIR");
  char pv[512], pm[512];
  if (dir && *dir) {
    snprintf(a.libdir, sizeof a.libdir, "%s", dir);
    snprintf(pv, sizeof pv, "%s/libibverbs.so.1", dir);
    snprintf(pm, sizeof pm, "%s/libmlx5.so.1", dir);
  } else {
    snprintf(pv, sizeof pv, "libibverbs.so.1");
    snprintf(pm, sizeof pm, "libmlx5.so.1");
  }
  a.verbs = dlopen(pv, RTLD_NOW | RTLD_GLOBAL);
  if (!a.verbs) { why(0, "%s: %s", pv, dlerror()); return a; }
  a.mlx5 = dlopen(pm, RTLD_NOW | RTLD_GLOBAL);
#define SYM(field, name) a.field = (decltype(a.field))dlsym(a.verbs, name)
  SYM(get_device_list, "ibv_get_device_list"); SYM(free_device_list, "ibv_free_device_list");
  SYM(get_device_name, "ibv_get_device_name"); SYM(open_device, "ibv_open_device"); SYM(close_device, "ibv_close_device");
  SYM(alloc_pd, "ibv_alloc_pd"); SYM(dealloc_pd, "ibv_dealloc_pd"); SYM(reg_mr, "ibv_reg_mr");
  SYM(reg_dmabuf_mr, "ibv_reg_dmabuf_mr"); SYM(dereg_mr, "ibv_dereg_mr"); SYM(create_cq, "ibv_create_cq");
  SYM(destroy_cq, "ibv_destroy_cq"); SYM(create_qp, "ibv_create_qp"); SYM(destroy_qp, "ibv_destroy_qp");
  SYM(modify_qp, "ibv_modify_qp"); SYM(query_port, "ibv_query_port"); SYM(query_gid, "ibv_query_gid");
  SYM(mock_qp_stats, "mock_qp_stats"); SYM(mock_declare_gpu_range, "mock_declare_gpu_range"); SYM(mock_gpu_free, "mock_gpu_free");
  SYM(mock_set_rnr_timeout_ms, "mock_set_rnr_timeout_ms"); SYM(mock_bridge_status, "mock_bridge_status");
#undef SYM
  a.is_mock = dlsym(a.verbs, "mock_verbs_is_mock") != nullptr;
  if (a.mlx5) a.dv_init_obj = (decltype(a.dv_init_obj))dlsym(a.mlx5, "mlx5dv_init_obj");
  a.ok = a.get_device_list && a.free_device_list && a.get_device_name && a.open_device && a.close_device && a.alloc_pd &&
         a.dealloc_pd && a.reg_mr && a.dereg_mr && a.create_cq && a.destroy_cq && a.create_qp && a.destroy_qp && a.modify_qp &&
         a.query_port && a.query_gid;
  if (!a.ok) why(0, "%s is missing expected symbols", pv);
  return a;
}

struct Dev {
  ibv_context* ctx = nullptr;
  ibv_pd* pd = nullptr;
  uint8_t port = 1;
  int gid_index = 0;
  ibv_port_attr pattr;
  ibv_gid gid;
  char name[64];
};
struct CqH { Dev* dev; ibv_cq* cq; int depth; };
struct QpH {
  Dev* dev;
  CqH *scq, *rcq;
  ibv_qp* qp;
  uint32_t sq_depth, rq_depth;
  uint64_t next_wr_id = 1;
  bool raw_owned = false;     // queues handed to the GPU: host posting would fight over the producer index
  int proxy_slot = -1;
  std::vector<uint64_t> host_regs;   // pages of g_host_regs this QP holds (rn_verbs_map_qp_to_gpu)
};

// Host ranges this library cudaHostRegister()ed to map a QP's queues into the GPU, keyed by first page, with the
// number of QPs using each (CQs and UAR pages can be shared by QPs).  The memory belongs to the provider, which
// frees it when the QP / CQ is destroyed: the registration must go first, or it stays on freed heap pages and a
// later queue allocated across them fails to map (cudaHostRegister reports "already registered" for a range whose
// first page has no device pointer).
std::mutex g_host_regs_mu;
std::map<uint64_t, int> g_host_regs;

void host_regs_release(std::vector<uint64_t>& pages) {
  std::lock_guard<std::mutex> g(g_host_regs_mu);
  for (uint64_t p : pages) {
    auto it = g_host_regs.find(p);
    if (it == g_host_regs.end() || --it->second > 0) continue;
    g_host_regs.erase(it);
    cudaHostUnregister((void*)p);
    cudaGetLastError();
  }
  pages.clear();
}

struct MrH { Dev* dev; ibv_mr* mr; int mode; };

// ---------------------------------------------------------------- CPU doorbell proxy
struct ProxySlot {
  std::atomic<bool> live{false};
  volatile unsigned long long* mailbox = nullptr;   // pinned, mapped: the GPU stores the doorbell value here
  volatile unsigned long long* reg = nullptr;       // the HCA's BlueFlame register (MMIO)
  unsigned long long seen = 0;
  std::atomic<uint64_t> forwarded{0};
};
constexpr int kMaxProxy = 256;
ProxySlot g_proxy[kMaxProxy];
unsigned long long* g_mailboxes = nullptr;           // one page-aligned pinned block of kMaxProxy * 64 bytes
std::thread g_proxy_thr;
std::atomic<bool> g_proxy_run{false}, g_proxy_stop{false};
std::mutex g_proxy_mu;

void proxy_main() {
  uint64_t idle_since = 0;
  while (!g_proxy_stop.load(std::memory_order_relaxed)) {
    bool busy = false;
    for (int i = 0; i < kMaxProxy; ++i) {
      ProxySlot& s = g_proxy[i];
      if (!s.live.load(std::memory_order_acquire)) continue;
      const unsigned long long v = __atomic_load_n((unsigned long long*)s.mailbox, __ATOMIC_ACQUIRE);
      if (v == s.seen) continue;
      s.seen = v;
      // WQE bytes and the doorbell record were made visible by the GPU's system-scope release before the
      // mailbox store; the store below is the MMIO write a host ibv_post_send would have done.
      __atomic_thread_fence(__ATOMIC_SEQ_CST);
      *s.reg = v;
      s.forwarded.fetch_add(1, std::memory_order_relaxed);
      busy = true;
    }
    if (busy) { idle_since = 0; continue; }
    const uint64_t t = now_ns();
    if (!idle_since) idle_since = t;
    if (t - idle_since > 5000000ull) { struct timespec ts = {0, 20000}; nanosleep(&ts, nullptr); }
    else sched_yield();
  }
}
// Mailbox memory: pinned + mapped when CUDA can (so the GPU reaches it), plain page-aligned memory otherwise
// (CPU-only tests drive the mailbox from the host).
int proxy_attach(volatile unsigned long long* reg, unsigned long long** mailbox_host) {
  std::lock_guard<std::mutex> g(g_proxy_mu);
  if (!g_mailboxes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, kMaxProxy * 64, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
      cudaGetLastError();
      if (posix_memalign(&p, 4096, kMaxProxy * 64)) return -12;
    }
    memset(p, 0, kMaxProxy * 64);
    g_mailboxes = (unsigned long long*)p;
  }
  int slot = -1;
  for (int i = 0; i < kMaxProxy; ++i) if (!g_proxy[i].live.load()) { slot = i; break; }
  if (slot < 0) return -12;
  ProxySlot& s = g_proxy[slot];
  s.mailbox = g_mailboxes + (size_t)slot * 8;
  *s.mailbox = 0;
  s.reg = reg; s.seen = 0; s.forwarded = 0;
  s.live.store(true, std::memory_order_release);
  bool expect = false;
  if (g_proxy_run.compare_exchange_strong(expect, true)) {
    g_proxy_stop = false;
    g_proxy_thr = std::thread(proxy_main);
    atexit([] { g_proxy_stop = true; if (g_proxy_thr.joinable()) g_proxy_thr.join(); });
  }
  *mailbox_host = (unsigned long long*)s.mailbox;
  return slot;
}
void proxy_detach(int slot) {
  if (slot >= 0 && slot < kMaxProxy) g_proxy[slot].live.store(false, std::memory_order_release);
}

}  // namespace

// ------------------------------------------------------------------ discovery
RN_API int rn_verbs_compiled() { return 1; }
RN_API const char* rn_verbs_why() { return g_why; }
RN_API int rn_verbs_is_mock() { return api().ok && api().is_mock ? 1 : 0; }
RN_API const char* rn_verbs_libdir() { return api().libdir; }
// Number of usable RDMA devices (0 = none; rn_verbs_why() says why).
RN_API int rn_verbs_available() {
  Api& a = api();
  if (!a.ok) { if (!g_why[0]) why(0, "libibverbs not loadable"); return 0; }
  if (!a.is_mock && !uverbs_nodes_present()) { why(0, "/dev/infiniband is not exposed to this container"); return 0; }
  int n = 0;
  ibv_device** l = a.get_device_list(&n);
  if (l) a.free_device_list(l);
  if (n <= 0) { why(0, "no RDMA devices"); return 0; }
  return n;
}
RN_API int rn_verbs_device_name(int i, char* out, int cap) {
  Api& a = api();
  int n = 0;
  ibv_device** l = a.ok ? a.get_device_list(&n) : nullptr;
  if (!l || i < 0 || i >= n) { if (l) a.free_device_list(l); return -19; }
  snprintf(out, cap, "%s", a.get_device_name(l[i]));
  a.free_device_list(l);
  return 0;
}

// ------------------------------------------------------------------ device
// name: exact device name, or "" / NULL with index >= 0 for "the index-th device" (GPU i <-> NIC i affinity).
RN_API void* rn_verbs_open(const char* name, int index, int port, int gid_index) {
  Api& a = api();
  if (!a.ok) return nullptr;
  int n = 0;
  ibv_device** l = a.get_device_list(&n);
  Dev* d = nullptr;
  for (int i = 0; l && i < n; ++i) {
    if (name && *name) { if (strcmp(a.get_device_name(l[i]), name)) continue; }
    else if (index >= 0 && i != index % n) continue;
    ibv_context* c = a.open_device(l[i]);
    if (!c) continue;
    d = new Dev();
    d->ctx = c; d->port = (uint8_t)(port > 0 ? port : 1); d->gid_index = gid_index;
    snprintf(d->name, sizeof d->name, "%s", a.get_device_name(l[i]));
    memset(&d->pattr, 0, sizeof d->pattr);
    d->pd = a.alloc_pd(c);
    if (!d->pd || a.query_port(c, d->port, &d->pattr)) {
      if (d->pd) a.dealloc_pd(d->pd);
      a.close_device(c);
      delete d; d = nullptr;
      continue;
    }
    memset(&d->gid, 0, sizeof d->gid);
    a.query_gid(c, d->port, gid_index, &d->gid);
    break;
  }
  if (l) a.free_device_list(l);
  if (!d) why(0, "cannot open RDMA device %s (index %d)", name && *name ? name : "(any)", index);
  return d;
}
RN_API int rn_verbs_close(void* dev) {
  Dev* d = (Dev*)dev;
  if (!d) return 0;
  api().dealloc_pd(d->pd);
  api().close_device(d->ctx);
  delete d;
  return 0;
}
RN_API const char* rn_verbs_dev_name(void* dev) { return ((Dev*)dev)->name; }
RN_API int rn_verbs_port_active(void* dev) { return ((Dev*)dev)->pattr.state == IBV_PORT_ACTIVE; }
RN_API int rn_verbs_link_layer(void* dev) { return ((Dev*)dev)->pattr.link_layer; }
RN_API int rn_verbs_local_addr(void* dev, uint16_t* lid, uint8_t* gid16) {
  Dev* d = (Dev*)dev;
  *lid = d->pattr.lid;
  memcpy(gid16, d->gid.raw, 16);
  return 0;
}

// ------------------------------------------------------------------ memory registration
// mode 0: ibv_reg_mr on the pointer (host memory, or GPU HBM through a peer-memory client)
// mode 1: ibv_reg_dmabuf_mr on an exported dma-buf fd (fd covers [ptr - fd_offset, ...); iova = ptr)
RN_API void* rn_verbs_reg_mr(void* dev, uint64_t ptr, uint64_t len, int mode, int dmabuf_fd, uint64_t fd_offset, uint32_t access,
                             uint32_t* lkey, uint32_t* rkey) {
  Dev* d = (Dev*)dev;
  int acc = 0;
  if (access & 1) acc |= IBV_ACCESS_LOCAL_WRITE;
  if (access & 2) acc |= IBV_ACCESS_REMOTE_WRITE | IBV_ACCESS_LOCAL_WRITE;   // IB: remote write requires local write
  if (access & 4) acc |= IBV_ACCESS_REMOTE_READ;
  ibv_mr* mr = nullptr;
  errno = 0;
  if (mode == 1) {
    if (!api().reg_dmabuf_mr) { why(0, "this libibverbs has no ibv_reg_dmabuf_mr (rdma-core < 34)"); return nullptr; }
    mr = api().reg_dmabuf_mr(d->pd, fd_offset, len, ptr, dmabuf_fd, acc);
  } else {
    mr = api().reg_mr(d->pd, (void*)ptr, len, acc);
  }
  if (!mr) {
    const int e = errno;
    why(0, "%s on [0x%llx, +%llu) failed: errno %d (%s)%s", mode == 1 ? "ibv_reg_dmabuf_mr" : "ibv_reg_mr", (unsigned long long)ptr,
        (unsigned long long)len, e, strerror(e),
        e == EFAULT && mode == 0 ? " -- for GPU memory this means no peer-memory client (nvidia-peermem / b200p2p) claimed the range" : "");
    return nullptr;
  }
  *lkey = mr->lkey; *rkey = mr->rkey;
  MrH* h = new MrH{d, mr, mode};
  return h;
}
RN_API int rn_verbs_dereg_mr(void* mr) {
  MrH* h = (MrH*)mr;
  int rc = api().dereg_mr(h->mr);
  delete h;
  return rc ? -rc : 0;
}

// ------------------------------------------------------------------ queues
RN_API void* rn_verbs_create_cq(void* dev, int depth) {
  Dev* d = (Dev*)dev;
  ibv_cq* cq = api().create_cq(d->ctx, depth, nullptr, nullptr, 0);
  if (!cq) { why(0, "ibv_create_cq(%d) failed: errno %d", depth, errno); return nullptr; }
  return new CqH{d, cq, depth};
}
RN_API int rn_verbs_destroy_cq(void* cq) {
  CqH* c = (CqH*)cq;
  int rc = api().destroy_cq(c->cq);
  if (rc) return -rc;
  delete c;
  return 0;
}
RN_API void* rn_verbs_create_qp(void* dev, void* scq, void* rcq, uint32_t sq_depth, uint32_t rq_depth) {
  Dev* d = (Dev*)dev;
  ibv_qp_init_attr ia;
  memset(&ia, 0, sizeof ia);
  ia.send_cq = ((CqH*)scq)->cq; ia.recv_cq = ((CqH*)(rcq ? rcq : scq))->cq;
  ia.qp_type = IBV_QPT_RC;
  ia.cap.max_send_wr = sq_depth; ia.cap.max_recv_wr = rq_depth; ia.cap.max_send_sge = 1; ia.cap.max_recv_sge = 1;
  ibv_qp* qp = api().create_qp(d->pd, &ia);
  if (!qp) { why(0, "ibv_create_qp failed: errno %d", errno); return nullptr; }
  QpH* q = new QpH();
  q->dev = d; q->scq = (CqH*)scq; q->rcq = (CqH*)(rcq ? rcq : scq); q->qp = qp;
  q->sq_depth = ia.cap.max_send_wr; q->rq_depth = ia.cap.max_recv_wr;
  return q;
}
RN_API int rn_verbs_destroy_qp(void* qp) {
  QpH* q = (QpH*)qp;
  proxy_detach(q->proxy_slot);
  host_regs_release(q->host_regs);
  int rc = api().destroy_qp(q->qp);
  delete q;
  return rc ? -rc : 0;
}
RN_API uint32_t rn_verbs_qpn(void* qp) { return ((QpH*)qp)->qp->qp_num; }
RN_API uint32_t rn_verbs_qp_state(void* qp) { return (uint32_t)((QpH*)qp)->qp->state; }

// RESET -> INIT -> RTR -> RTS towards (remote_qpn, remote_lid / gid); loopback when it names ourselves.
RN_API int rn_verbs_connect(void* qp, uint32_t remote_qpn, uint16_t remote_lid, const uint8_t* remote_gid16) {
  QpH* q = (QpH*)qp;
  Dev* d = q->dev;
  ibv_qp_attr a;
  memset(&a, 0, sizeof a);
  a.qp_state = IBV_QPS_INIT; a.pkey_index = 0; a.port_num = d->port;
  a.qp_access_flags = IBV_ACCESS_REMOTE_WRITE | IBV_ACCESS_REMOTE_READ | IBV_ACCESS_LOCAL_WRITE;
  int rc = api().modify_qp(q->qp, &a, IBV_QP_STATE | IBV_QP_PKEY_INDEX | IBV_QP_PORT | IBV_QP_ACCESS_FLAGS);
  if (rc) return why(-rc, "modify_qp(INIT) failed: %d", rc);
  memset(&a, 0, sizeof a);
  a.qp_state = IBV_QPS_RTR; a.path_mtu = IBV_MTU_4096; a.dest_qp_num = remote_qpn; a.rq_psn = 0;
  a.max_dest_rd_atomic = 16; a.min_rnr_timer = 12;
  a.ah_attr.dlid = remote_lid; a.ah_attr.port_num = d->port;
  if (d->pattr.link_layer == IBV_LINK_LAYER_ETHERNET || (remote_gid16 && !remote_lid)) {
    a.ah_attr.is_global = 1; a.ah_attr.grh.hop_limit = 1; a.ah_attr.grh.sgid_index = (uint8_t)d->gid_index;
    memcpy(a.ah_attr.grh.dgid.raw, remote_gid16 ? remote_gid16 : d->gid.raw, 16);
  }
  rc = api().modify_qp(q->qp, &a, IBV_QP_STATE | IBV_QP_AV | IBV_QP_PATH_MTU | IBV_QP_DEST_QPN | IBV_QP_RQ_PSN |
                                    IBV_QP_MAX_DEST_RD_ATOMIC | IBV_QP_MIN_RNR_TIMER);
  if (rc) return why(-rc, "modify_qp(RTR) towards lid %u qpn 0x%x failed: %d", remote_lid, remote_qpn, rc);
  memset(&a, 0, sizeof a);
  a.qp_state = IBV_QPS_RTS; a.timeout = 14; a.retry_cnt = 7; a.rnr_retry = 7; a.sq_psn = 0; a.max_rd_atomic = 16;
  rc = api().modify_qp(q->qp, &a, IBV_QP_STATE | IBV_QP_TIMEOUT | IBV_QP_RETRY_CNT | IBV_QP_RNR_RETRY | IBV_QP_SQ_PSN | IBV_QP_MAX_QP_RD_ATOMIC);
  return rc ? why(-rc, "modify_qp(RTS) failed: %d", rc) : 0;
}
// state: 0 RESET, 6 ERR (the two transitions that need no attributes)
RN_API int rn_verbs_set_state(void* qp, uint32_t state) {
  QpH* q = (QpH*)qp;
  ibv_qp_attr a;
  memset(&a, 0, sizeof a);
  a.qp_state = (ibv_qp_state)state;
  int rc = api().modify_qp(q->qp, &a, IBV_QP_STATE);
  return rc ? why(-rc, "modify_qp(state %u) failed: %d", state, rc) : 0;
}

// ------------------------------------------------------------------ host-posted verbs (baselines B0 / B2)
// opcode is the mlx5 WQE opcode the rest of the project uses (wire.OP_*).
RN_API int rn_verbs_post_send(void* qp, uint32_t opcode, uint64_t laddr, uint32_t lkey, uint64_t raddr, uint32_t rkey, uint32_t len,
                              int signaled, uint32_t imm, uint64_t* wr_id_out) {
  QpH* q = (QpH*)qp;
  if (q->raw_owned) return why(-16, "this QP's queues are owned by the GPU poster; host posting would corrupt the producer index");
  ibv_sge sge = {laddr, len, lkey};
  ibv_send_wr wr, *bad = nullptr;
  memset(&wr, 0, sizeof wr);
  wr.wr_id = q->next_wr_id++;
  wr.sg_list = &sge; wr.num_sge = 1;
  switch (opcode) {
    case 0x08: wr.opcode = IBV_WR_RDMA_WRITE; break;
    case 0x09: wr.opcode = IBV_WR_RDMA_WRITE_WITH_IMM; break;
    case 0x0a: wr.opcode = IBV_WR_SEND; break;
    case 0x0b: wr.opcode = IBV_WR_SEND_WITH_IMM; break;
    case 0x10: wr.opcode = IBV_WR_RDMA_READ; break;
    default: return why(-22, "unsupported opcode 0x%x for a host post", opcode);
  }
  wr.send_flags = signaled ? IBV_SEND_SIGNALED : 0;
  wr.imm_data = __builtin_bswap32(imm);            // host value -> network order
  wr.wr.rdma.remote_addr = raddr; wr.wr.rdma.rkey = rkey;
  int rc = ibv_post_send(q->qp, &wr, &bad);
  if (rc) return why(-rc, "ibv_post_send failed: %d (%s)", rc, strerror(rc));
  if (wr_id_out) *wr_id_out = wr.wr_id;
  return 0;
}
RN_API int rn_verbs_post_recv(void* qp, uint64_t addr, uint32_t lkey, uint32_t len, uint64_t* wr_id_out) {
  QpH* q = (QpH*)qp;
  ibv_sge sge = {addr, len, lkey};
  ibv_recv_wr wr, *bad = nullptr;
  memset(&wr, 0, sizeof wr);
  wr.wr_id = q->next_wr_id++;
  wr.sg_list = &sge; wr.num_sge = 1;
  int rc = ibv_post_recv(q->qp, &wr, &bad);
  if (rc) return why(-rc, "ibv_post_recv failed: %d (%s)", rc, strerror(rc));
  if (wr_id_out) *wr_id_out = wr.wr_id;
  return 0;
}
struct RnVWc { uint64_t wr_id; uint32_t status, opcode, byte_len, imm, qp_num, vendor_err, with_imm, pad; };
RN_API int rn_verbs_poll(void* cq, int max, RnVWc* out) {
  CqH* c = (CqH*)cq;
  ibv_wc wc[32];
  if (max > 32) max = 32;
  int n = ibv_poll_cq(c->cq, max, wc);
  for (int i = 0; i < n; ++i) {
    out[i].wr_id = wc[i].wr_id; out[i].status = wc[i].status; out[i].opcode = wc[i].opcode; out[i].byte_len = wc[i].byte_len;
    out[i].with_imm = (wc[i].wc_flags & IBV_WC_WITH_IMM) ? 1 : 0;
    out[i].imm = out[i].with_imm ? __builtin_bswap32(wc[i].imm_data) : 0;
    out[i].qp_num = wc[i].qp_num; out[i].vendor_err = wc[i].vendor_err; out[i].pad = 0;
  }
  return n;
}

// B0 / B2: window-limited stream of `iters` host-posted work requests (ib_write_bw / ib_read_bw), CQ polled by
// the CPU.  laddr / raddr rotate over `nslots` slots of `slot_stride` bytes.  Host-timed (steady clock): the
// baseline is a host program.
RN_API int rn_verbs_host_stream(void* qp, uint32_t opcode, uint64_t laddr, uint32_t lkey, uint64_t raddr, uint32_t rkey, uint32_t bytes,
                                uint32_t iters, uint32_t window, uint64_t slot_stride, uint32_t nslots, uint64_t timeout_ms,
                                uint64_t* ns_out, uint32_t* errors_out) {
  QpH* q = (QpH*)qp;
  if (!window || window > q->sq_depth) window = q->sq_depth;
  if (!nslots) nslots = 1;
  uint32_t posted = 0, done = 0, errors = 0;
  RnVWc wc[32];
  const uint64_t t0 = now_ns(), deadline = t0 + (timeout_ms ? timeout_ms : 5000) * 1000000ull;
  while (done < iters) {
    while (posted < iters && posted - done < window) {
      const uint64_t off = (uint64_t)(posted % nslots) * slot_stride;
      int rc = rn_verbs_post_send(qp, opcode, laddr + off, lkey, raddr + off, rkey, bytes, 1, 0, nullptr);
      if (rc) return rc;
      ++posted;
    }
    int n = rn_verbs_poll(q->scq, 32, wc);
    if (n < 0) return why(-5, "ibv_poll_cq failed");
    for (int i = 0; i < n; ++i) errors += wc[i].status != 0;
    done += (uint32_t)n;
    if (!n && now_ns() > deadline) return why(-110, "host_stream: timed out with %u/%u completions", done, iters);
  }
  *ns_out = now_ns() - t0;
  if (errors_out) *errors_out = errors;
  return 0;
}
// B1: host-staged.  Per message: cudaMemcpy D2H into a registered bounce buffer, host-posted RDMA write between
// two host MRs, cudaMemcpy H2D out of the destination bounce buffer -- the path GPUDirect exists to avoid.
RN_API int rn_verbs_host_staged_stream(void* qp, uint64_t dev_src, uint64_t dev_dst, uint64_t host_a, uint32_t lkey_a, uint64_t host_b,
                                       uint32_t rkey_b, uint32_t bytes, uint32_t iters, uint64_t slot_stride, uint32_t nslots,
                                       uint64_t timeout_ms, uint64_t* ns_out) {
  QpH* q = (QpH*)qp;
  if (!nslots) nslots = 1;
  cudaStream_t st = nullptr;
  if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) return why(-5, "host_staged: no CUDA stream");
  RnVWc wc;
  int rc = 0;
  const uint64_t t0 = now_ns();
  for (uint32_t i = 0; i < iters && !rc; ++i) {
    const uint64_t off = (uint64_t)(i % nslots) * slot_stride;
    if (cudaMemcpyAsync((void*)host_a, (const void*)(dev_src + off), bytes, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) { rc = why(-5, "host_staged: D2H failed"); break; }
    rc = rn_verbs_post_send(qp, 0x08, host_a, lkey_a, host_b, rkey_b, bytes, 1, 0, nullptr);
    if (rc) break;
    const uint64_t deadline = now_ns() + (timeout_ms ? timeout_ms : 5000) * 1000000ull;
    int n = 0;
    while ((n = rn_verbs_poll(q->scq, 1, &wc)) == 0)
      if (now_ns() > deadline) { rc = why(-110, "host_staged: completion timed out"); break; }
    if (rc) break;
    if (n < 0 || wc.status) { rc = why(-5, "host_staged: error completion (status %u)", wc.status); break; }
    if (cudaMemcpyAsync((void*)(dev_dst + off), (const void*)host_b, bytes, cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) { rc = why(-5, "host_staged: H2D failed"); break; }
  }
  *ns_out = now_ns() - t0;
  cudaStreamDestroy(st);
  return rc;
}

// ------------------------------------------------------------------ raw queues (mlx5dv) and the GPU mapping
struct RnRawQp {
  uint64_t sq_buf; uint32_t sq_wqe_cnt, sq_stride;
  uint64_t rq_buf; uint32_t rq_wqe_cnt, rq_stride;
  uint64_t dbrec; uint64_t bf_reg; uint32_t bf_size, qpn;
  uint64_t cq_buf; uint32_t cq_cqe_cnt, cq_cqe_size; uint64_t cq_dbrec; uint32_t cqn, pad0;
  uint64_t rcq_buf; uint32_t rcq_cqe_cnt, rcq_cqe_size; uint64_t rcq_dbrec; uint32_t rcqn, pad1;
};
RN_API int rn_verbs_raw_qp(void* qp, RnRawQp* out) {
  QpH* q = (QpH*)qp;
  if (!api().dv_init_obj) return why(-38, "libmlx5 (mlx5dv_init_obj) not available: direct verbs need an mlx5 device");
  mlx5dv_qp dq; mlx5dv_cq dc, drc; mlx5dv_obj obj;
  memset(&dq, 0, sizeof dq); memset(&dc, 0, sizeof dc); memset(&drc, 0, sizeof drc); memset(&obj, 0, sizeof obj);
  obj.qp.in = q->qp; obj.qp.out = &dq; obj.cq.in = q->scq->cq; obj.cq.out = &dc;
  int rc = api().dv_init_obj(&obj, MLX5DV_OBJ_QP | MLX5DV_OBJ_CQ);
  if (rc) return why(-rc, "mlx5dv_init_obj(QP|CQ) failed: %d", rc);
  if (q->rcq != q->scq) {
    memset(&obj, 0, sizeof obj);
    obj.cq.in = q->rcq->cq; obj.cq.out = &drc;
    rc = api().dv_init_obj(&obj, MLX5DV_OBJ_CQ);
    if (rc) return why(-rc, "mlx5dv_init_obj(recv CQ) failed: %d", rc);
  } else {
    drc = dc;
  }
  memset(out, 0, sizeof *out);
  out->sq_buf = (uint64_t)dq.sq.buf; out->sq_wqe_cnt = dq.sq.wqe_cnt; out->sq_stride = dq.sq.stride;
  out->rq_buf = (uint64_t)dq.rq.buf; out->rq_wqe_cnt = dq.rq.wqe_cnt; out->rq_stride = dq.rq.stride;
  out->dbrec = (uint64_t)dq.dbrec; out->bf_reg = (uint64_t)dq.bf.reg; out->bf_size = dq.bf.size; out->qpn = q->qp->qp_num;
  out->cq_buf = (uint64_t)dc.buf; out->cq_cqe_cnt = dc.cqe_cnt; out->cq_cqe_size = dc.cqe_size; out->cq_dbrec = (uint64_t)dc.dbrec; out->cqn = dc.cqn;
  out->rcq_buf = (uint64_t)drc.buf; out->rcq_cqe_cnt = drc.cqe_cnt; out->rcq_cqe_size = drc.cqe_size; out->rcq_dbrec = (uint64_t)drc.dbrec; out->rcqn = drc.cqn;
  return 0;
}

// Attach the CPU doorbell proxy to this QP (also the fallback of rn_verbs_map_qp_to_gpu): returns the host
// address of the 8-byte mailbox; whatever is stored there is forwarded to the BlueFlame register.
RN_API int rn_verbs_db_proxy_attach(void* qp, uint64_t* mailbox_host) {
  QpH* q = (QpH*)qp;
  RnRawQp raw;
  int rc = rn_verbs_raw_qp(qp, &raw);
  if (rc) return rc;
  unsigned long long* mb = nullptr;
  int slot = proxy_attach((volatile unsigned long long*)raw.bf_reg, &mb);
  if (slot < 0) return why(slot, "doorbell proxy: no free slot / no memory");
  q->proxy_slot = slot;
  q->raw_owned = true;
  *mailbox_host = (uint64_t)mb;
  return 0;
}
RN_API uint64_t rn_verbs_db_proxy_forwarded(void* qp) {
  QpH* q = (QpH*)qp;
  return q->proxy_slot >= 0 ? g_proxy[q->proxy_slot].forwarded.load() : 0;
}

// N3 on hardware: make the NIC's queues visible to the GPU so hca/post.cuh can drive it.
//   * SQ / RQ buffers, doorbell records and CQ buffers are host memory owned by rdma-core:
//     cudaHostRegister(Mapped) gives the GPU a device pointer to the same bytes (the NIC keeps reading them
//     where it always did);
//   * the BlueFlame register is a PCIe BAR page of the HCA: cudaHostRegisterIoMemory maps it so an SM's
//     8-byte store IS the MMIO doorbell write.  If the driver refuses (no PeerMappingOverride / IoMemory
//     support) -- or ROCNRDMA_DB_PROXY=1 asks for it -- the doorbell goes through the CPU proxy instead.
// flags out: bit 0 = doorbell through the CPU proxy.
struct RnGpuQp {
  uint64_t sq_dev, rq_dev, dbrec_dev, bf_dev, cq_dev, cq_dbrec_dev, rcq_dev, rcq_dbrec_dev;
  uint32_t sq_wqe_cnt, rq_wqe_cnt, cq_cqe_cnt, rcq_cqe_cnt, qpn, cqn, rcqn, flags;
};
RN_API int rn_verbs_map_qp_to_gpu(void* qp, RnGpuQp* out) {
  QpH* q = (QpH*)qp;
  RnRawQp raw;
  int rc = rn_verbs_raw_qp(qp, &raw);
  if (rc) return rc;
  if (raw.sq_stride != 64 || raw.cq_cqe_size != 64 || raw.rcq_cqe_size != 64)
    return why(-22, "unexpected WQE/CQE stride %u/%u/%u (the device poster speaks 64-byte WQEBBs and CQE64)", raw.sq_stride, raw.cq_cqe_size, raw.rcq_cqe_size);
  if (raw.rq_stride != 16) return why(-22, "unexpected receive stride %u (one 16-byte data segment per receive WQE expected)", raw.rq_stride);
  auto pow2 = [](uint32_t v) { return v && !(v & (v - 1)); };
  if (!pow2(raw.sq_wqe_cnt) || !pow2(raw.rq_wqe_cnt) || !pow2(raw.cq_cqe_cnt) || !pow2(raw.rcq_cqe_cnt))
    return why(-22, "queue sizes must be powers of two (sq %u rq %u cq %u rcq %u)", raw.sq_wqe_cnt, raw.rq_wqe_cnt, raw.cq_cqe_cnt, raw.rcq_cqe_cnt);
  auto map = [&](uint64_t host, size_t bytes, unsigned flags, uint64_t* dev, bool quiet) -> int {
    const uint64_t page = host & ~4095ull;
    const size_t len = ((host + bytes + 4095) & ~4095ull) - page;
    cudaError_t e;
    {
      std::lock_guard<std::mutex> g(g_host_regs_mu);
      e = cudaHostRegister((void*)page, len, flags);
      if (e == cudaSuccess || (e == cudaErrorHostMemoryAlreadyRegistered && g_host_regs.count(page))) {
        ++g_host_regs[page];
        q->host_regs.push_back(page);
      }
    }
    if (e != cudaSuccess && e != cudaErrorHostMemoryAlreadyRegistered) {
      cudaGetLastError();
      if (!quiet) why(-5, "cudaHostRegister(0x%llx, %zu, 0x%x): %s", (unsigned long long)page, len, flags, cudaGetErrorString(e));
      return -5;
    }
    cudaGetLastError();
    void* d = nullptr;
    if (cudaHostGetDevicePointer(&d, (void*)page, 0) != cudaSuccess) { cudaGetLastError(); if (!quiet) why(-5, "cudaHostGetDevicePointer failed"); return -5; }
    *dev = (uint64_t)d + (host - page);
    return 0;
  };
  const unsigned M = cudaHostRegisterMapped | cudaHostRegisterPortable;
  memset(out, 0, sizeof *out);
  if ((rc = map(raw.sq_buf, (size_t)raw.sq_wqe_cnt * 64, M, &out->sq_dev, false))) return rc;
  if ((rc = map(raw.rq_buf, (size_t)raw.rq_wqe_cnt * 16, M, &out->rq_dev, false))) return rc;
  if ((rc = map(raw.dbrec, 8, M, &out->dbrec_dev, false))) return rc;
  if ((rc = map(raw.cq_buf, (size_t)raw.cq_cqe_cnt * 64, M, &out->cq_dev, false))) return rc;
  if ((rc = map(raw.cq_dbrec, 8, M, &out->cq_dbrec_dev, false))) return rc;
  if ((rc = map(raw.rcq_buf, (size_t)raw.rcq_cqe_cnt * 64, M, &out->rcq_dev, false))) return rc;
  if ((rc = map(raw.rcq_dbrec, 8, M, &out->rcq_dbrec_dev, false))) return rc;
  const char* force = getenv("ROCNRDMA_DB_PROXY");
  bool proxy = force && atoi(force) == 1;
  if (!proxy) {
    // the UAR page: IoMemory for a real BAR; the mock's "UAR" is ordinary memory, for which the plain mapping is right
    rc = map(raw.bf_reg, raw.bf_size ? raw.bf_size : 256, cudaHostRegisterIoMemory | M, &out->bf_dev, true);
    if (rc) rc = map(raw.bf_reg, raw.bf_size ? raw.bf_size : 256, M, &out->bf_dev, true);
    if (rc) proxy = true;
  }
  if (proxy) {
    uint64_t mb = 0;
    if ((rc = rn_verbs_db_proxy_attach(qp, &mb))) return rc;
    void* d = nullptr;
    if (cudaHostGetDevicePointer(&d, (void*)mb, 0) != cudaSuccess) { cudaGetLastError(); return why(-5, "doorbell mailbox is not GPU-mapped"); }
    out->bf_dev = (uint64_t)d;
    out->flags |= 1u;
  }
  out->sq_wqe_cnt = raw.sq_wqe_cnt; out->rq_wqe_cnt = raw.rq_wqe_cnt; out->cq_cqe_cnt = raw.cq_cqe_cnt; out->rcq_cqe_cnt = raw.rcq_cqe_cnt;
  out->qpn = raw.qpn; out->cqn = raw.cqn; out->rcqn = raw.rcqn;
  q->raw_owned = true;
  return 0;
}

// ------------------------------------------------------------------ mock control plane pass-through (tests)
struct RnMockQpStats { uint64_t n_wqe, n_cqe, n_err, n_bytes, n_rnr, n_db_no_progress, n_doorbells, hw_sq_cons, sq_cq_overruns; };
RN_API int rn_verbs_mock_qp_stats(void* qp, RnMockQpStats* out) {
  if (!api().mock_qp_stats) return -38;
  return api().mock_qp_stats(((QpH*)qp)->qp, out);
}
RN_API int rn_verbs_mock_declare_gpu_range(uint64_t va, uint64_t len) { return api().mock_declare_gpu_range ? api().mock_declare_gpu_range(va, len) : -38; }
RN_API int rn_verbs_mock_gpu_free(uint64_t va) { return api().mock_gpu_free ? api().mock_gpu_free(va) : -38; }
RN_API int rn_verbs_mock_set_rnr_timeout_ms(uint64_t ms) { if (!api().mock_set_rnr_timeout_ms) return -38; api().mock_set_rnr_timeout_ms(ms); return 0; }
RN_API const char* rn_verbs_mock_bridge_status() { return api().mock_bridge_status ? api().mock_bridge_status() : "not a mock provider"; }
