// Cross-check of csrc/wire/mlx5_wire.h against an INDEPENDENT statement of the mlx5 work-queue layout: the
// DOCA GPUNetIO definitions NVIDIA ships inside the NCCL wheel (doca_gpunetio_verbs_def.h: written by other people,
// for their own GPU-initiated mlx5 posting).  tests/test_wire_format.py compares the native encoder with a Python
// mirror written by the same hand as the encoder; this file is the outside reference the verdict asked for: if a field
// offset, a segment size, an opcode or a flag of ours disagreed with theirs, it would not compile.
// Built with -fsyntax-only by tests/test_wire_crosscheck.py (header: the copy in tests/golden).
#include <stddef.h>
#include <stdint.h>

#include DOCA_VERBS_DEF_H          // -DDOCA_VERBS_DEF_H='"<...>/doca_gpunetio_verbs_def.h"'
#include "wire/mlx5_wire.h"

using namespace rn;
#define SAME_OFFSET(ours, ofield, theirs, tfield) \
  static_assert(offsetof(ours, ofield) == offsetof(theirs, tfield), #ours "::" #ofield " vs " #theirs "::" #tfield)

// ---- segments
static_assert(sizeof(CtrlSeg) == sizeof(doca_gpunetio_ib_mlx5_wqe_ctrl_seg), "ctrl segment size");
SAME_OFFSET(CtrlSeg, opmod_idx_opcode, doca_gpunetio_ib_mlx5_wqe_ctrl_seg, opmod_idx_opcode);
SAME_OFFSET(CtrlSeg, qpn_ds, doca_gpunetio_ib_mlx5_wqe_ctrl_seg, qpn_ds);
SAME_OFFSET(CtrlSeg, signature, doca_gpunetio_ib_mlx5_wqe_ctrl_seg, signature);
SAME_OFFSET(CtrlSeg, fm_ce_se, doca_gpunetio_ib_mlx5_wqe_ctrl_seg, fm_ce_se);
SAME_OFFSET(CtrlSeg, imm, doca_gpunetio_ib_mlx5_wqe_ctrl_seg, imm);
static_assert(sizeof(RaddrSeg) == sizeof(doca_gpunetio_ib_mlx5_wqe_raddr_seg), "raddr segment size");
SAME_OFFSET(RaddrSeg, raddr, doca_gpunetio_ib_mlx5_wqe_raddr_seg, raddr);
SAME_OFFSET(RaddrSeg, rkey, doca_gpunetio_ib_mlx5_wqe_raddr_seg, rkey);
static_assert(sizeof(DataSeg) == sizeof(doca_gpunetio_ib_mlx5_wqe_data_seg), "data segment size");
SAME_OFFSET(DataSeg, byte_count, doca_gpunetio_ib_mlx5_wqe_data_seg, byte_count);
SAME_OFFSET(DataSeg, lkey, doca_gpunetio_ib_mlx5_wqe_data_seg, lkey);
SAME_OFFSET(DataSeg, addr, doca_gpunetio_ib_mlx5_wqe_data_seg, addr);
static_assert(sizeof(AtomicSeg) == sizeof(doca_gpunetio_ib_mlx5_wqe_atomic_seg), "atomic segment size");
SAME_OFFSET(AtomicSeg, swap_add, doca_gpunetio_ib_mlx5_wqe_atomic_seg, swap_add);
SAME_OFFSET(AtomicSeg, compare, doca_gpunetio_ib_mlx5_wqe_atomic_seg, compare);
static_assert(WQEBB == (1u << DOCA_GPUNETIO_IB_MLX5_WQE_SQ_SHIFT), "WQE basic block");
static_assert(DOCA_GPUNETIO_VERBS_WQE_IDX_SHIFT == 8, "wqe index sits at bits [23:8] of opmod_idx_opcode (ctrl_word0)");
static_assert(DOCA_GPUNETIO_VERBS_WQE_PI_MASK == 0xffff, "16-bit producer index in the doorbell record");

// ---- completion queue entry
static_assert(sizeof(Cqe64) == sizeof(doca_gpunetio_ib_mlx5_cqe64) && sizeof(Cqe64) == DOCA_GPUNETIO_VERBS_CQE_SIZE, "CQE64 size");
SAME_OFFSET(Cqe64, wqe_id, doca_gpunetio_ib_mlx5_cqe64, wqe_id);
SAME_OFFSET(Cqe64, slid, doca_gpunetio_ib_mlx5_cqe64, slid);
SAME_OFFSET(Cqe64, flags_rqpn, doca_gpunetio_ib_mlx5_cqe64, flags_rqpn);
SAME_OFFSET(Cqe64, srqn, doca_gpunetio_ib_mlx5_cqe64, srqn_uidx);
SAME_OFFSET(Cqe64, imm_inval_pkey, doca_gpunetio_ib_mlx5_cqe64, imm_inval_pkey);
SAME_OFFSET(Cqe64, byte_cnt, doca_gpunetio_ib_mlx5_cqe64, byte_cnt);
SAME_OFFSET(Cqe64, timestamp_h, doca_gpunetio_ib_mlx5_cqe64, timestamp);
SAME_OFFSET(Cqe64, sop_drop_qpn, doca_gpunetio_ib_mlx5_cqe64, sop_drop_qpn);
SAME_OFFSET(Cqe64, wqe_counter, doca_gpunetio_ib_mlx5_cqe64, wqe_counter);
SAME_OFFSET(Cqe64, signature, doca_gpunetio_ib_mlx5_cqe64, signature);
SAME_OFFSET(Cqe64, op_own, doca_gpunetio_ib_mlx5_cqe64, op_own);
static_assert(sizeof(ErrCqe) == sizeof(doca_gpunetio_ib_mlx5_err_cqe_ex), "error CQE size");
SAME_OFFSET(ErrCqe, srqn, doca_gpunetio_ib_mlx5_err_cqe_ex, srqn);
SAME_OFFSET(ErrCqe, vendor_err_synd, doca_gpunetio_ib_mlx5_err_cqe_ex, vendor_err_synd);
SAME_OFFSET(ErrCqe, syndrome, doca_gpunetio_ib_mlx5_err_cqe_ex, syndrome);
SAME_OFFSET(ErrCqe, s_wqe_opcode_qpn, doca_gpunetio_ib_mlx5_err_cqe_ex, s_wqe_opcode_qpn);
SAME_OFFSET(ErrCqe, wqe_counter, doca_gpunetio_ib_mlx5_err_cqe_ex, wqe_counter);
SAME_OFFSET(ErrCqe, op_own, doca_gpunetio_ib_mlx5_err_cqe_ex, op_own);
static_assert(DOCA_GPUNETIO_VERBS_MLX5_CQE_OPCODE_SHIFT == 4 && DOCA_GPUNETIO_IB_MLX5_CQE_OWNER_MASK == 1, "op_own = opcode[7:4] | owner[0]");
static_assert(DOCA_GPUNETIO_VERBS_CQE_CI_MASK == 0xffffff, "24-bit consumer index in the CQ doorbell record");

// ---- opcodes, flags, doorbell-record slots
static_assert(OP_NOP == DOCA_GPUNETIO_IB_MLX5_OPCODE_NOP && OP_SEND_INVAL == DOCA_GPUNETIO_IB_MLX5_OPCODE_SEND_INVAL, "opcodes");
static_assert(OP_RDMA_WRITE == DOCA_GPUNETIO_IB_MLX5_OPCODE_RDMA_WRITE && OP_RDMA_WRITE_IMM == DOCA_GPUNETIO_IB_MLX5_OPCODE_RDMA_WRITE_IMM, "opcodes");
static_assert(OP_SEND == DOCA_GPUNETIO_IB_MLX5_OPCODE_SEND && OP_SEND_IMM == DOCA_GPUNETIO_IB_MLX5_OPCODE_SEND_IMM, "opcodes");
static_assert(OP_RDMA_READ == DOCA_GPUNETIO_IB_MLX5_OPCODE_RDMA_READ && OP_ATOMIC_CS == DOCA_GPUNETIO_IB_MLX5_OPCODE_ATOMIC_CS &&
              OP_ATOMIC_FA == DOCA_GPUNETIO_IB_MLX5_OPCODE_ATOMIC_FA, "opcodes");
static_assert(CTRL_CQ_UPDATE == DOCA_GPUNETIO_IB_MLX5_WQE_CTRL_CQ_UPDATE && CTRL_SOLICITED == DOCA_GPUNETIO_IB_MLX5_WQE_CTRL_SOLICITED, "ctrl flags");
static_assert(CTRL_FENCE == DOCA_GPUNETIO_IB_MLX5_WQE_CTRL_FENCE && CTRL_INITIATOR_SMALL_FENCE == DOCA_GPUNETIO_IB_MLX5_WQE_CTRL_INITIATOR_SMALL_FENCE, "fence flags");
static_assert(CQE_REQ == DOCA_GPUNETIO_IB_MLX5_CQE_REQ && CQE_RESP_WR_IMM == DOCA_GPUNETIO_IB_MLX5_CQE_RESP_WR_IMM &&
              CQE_RESP_SEND == DOCA_GPUNETIO_IB_MLX5_CQE_RESP_SEND && CQE_RESP_SEND_IMM == DOCA_GPUNETIO_IB_MLX5_CQE_RESP_SEND_IMM &&
              CQE_RESP_SEND_INV == DOCA_GPUNETIO_IB_MLX5_CQE_RESP_SEND_INV && CQE_RESIZE_CQ == DOCA_GPUNETIO_IB_MLX5_CQE_RESIZE_CQ, "CQE opcodes");
static_assert(CQE_REQ_ERR == DOCA_GPUNETIO_IB_MLX5_CQE_REQ_ERR && CQE_RESP_ERR == DOCA_GPUNETIO_IB_MLX5_CQE_RESP_ERR &&
              CQE_INVALID == DOCA_GPUNETIO_IB_MLX5_CQE_INVALID, "CQE error / invalid opcodes");
static_assert(DBR_RCV == DOCA_GPUNETIO_IB_MLX5_RCV_DBR && DBR_SND == DOCA_GPUNETIO_IB_MLX5_SND_DBR, "doorbell record slots");
static_assert((0x80000000u) == DOCA_GPUNETIO_IB_MLX5_INLINE_SEG, "inline flag is bit 31 of byte_count (we mask it off: bytes & 0x7fffffff)");

int main() { return 0; }
