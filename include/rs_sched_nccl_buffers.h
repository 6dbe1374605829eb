/* include/rs_sched_nccl_buffers.h -- the multi-GPU end-of-run reduce of the per-slice BUFFER totals of buffered
 * handles (rs_enable_buffers), from C/C++.  A companion of include/rs_sched_nccl.h: the same library
 * (radiosaber_b200/librs_nccl.so), the same communicators, the same rules (import torch before loading it in a process
 * that also uses PyTorch).  It has a header of its own so that rs_sched_nccl.h keeps exactly the entry points it had. */
#ifndef RS_SCHED_NCCL_BUFFERS_H_
#define RS_SCHED_NCCL_BUFFERS_H_

#include "rs_sched_nccl.h"

#ifdef __cplusplus
extern "C" {
#endif

/* rs_reduce_stats for the buffers: rs_buffer_stats_device() of this rank's cells, then ncclReduce(sum, root) of the
 * uint64 [P][3][S] block (queued bytes, dropped bytes, records held) on the handle's stream; on the root the totals
 * over all ranks' cells are copied to stats_out (HOST uint64 [P][3][S]; ignored on the other ranks).  Integers, so the
 * result is the same bits whatever the reduction order.  Every rank of the communicator must call it; synchronous;
 * a handle without buffers fails (rs_nccl_last_error names rs_buffer_stats_device). */
int rs_reduce_buffer_stats(rs_handle* h, void* nccl_comm, int32_t root, uint64_t* stats_out);

#ifdef __cplusplus
}
#endif
#endif /* RS_SCHED_NCCL_BUFFERS_H_ */
