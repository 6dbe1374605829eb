/* include/rs_sched_nccl_ue_upt.h -- the multi-GPU end-of-run reduce of the per-UE throughput over active time (UPT)
 * histograms (rs_enable_ue_upt_hist), from C/C++.  A companion of include/rs_sched_nccl.h, rs_sched_nccl_buffers.h,
 * rs_sched_nccl_hol_hist.h and rs_sched_nccl_ue_rate.h: the same library (radiosaber_b200/librs_nccl.so), the same
 * communicators, the same rules (import torch before loading it in a process that also uses PyTorch).  It has a
 * header of its own so that the other four keep exactly the entry points they had. */
#ifndef RS_SCHED_NCCL_UE_UPT_H_
#define RS_SCHED_NCCL_UE_UPT_H_

#include "rs_sched_nccl_ue_rate.h"

#ifdef __cplusplus
extern "C" {
#endif

/* rs_reduce_ue_rate_hist for the UPT histograms: rs_ue_upt_hist_device() of this rank's cells, then ncclReduce(sum,
 * root) of the uint64 [P][S][n_bins] block on the handle's stream; on the root the counts over all ranks' cells are
 * copied to hist_out (HOST uint64 [P][S][n_bins]; ignored on the other ranks).  Integers, so the result is the same
 * bits whatever the reduction order.  Every rank of the communicator must call it, with the same n_bins; synchronous;
 * a handle without UPT fails (rs_nccl_last_error names rs_ue_upt_hist_device). */
int rs_reduce_ue_upt_hist(rs_handle* h, void* nccl_comm, int32_t root, uint64_t* hist_out);

#ifdef __cplusplus
}
#endif
#endif /* RS_SCHED_NCCL_UE_UPT_H_ */
