/* include/rs_sched_nccl.h -- the multi-GPU end-of-run reduce of the per-slice statistics, from C/C++.
 *
 * Lives in its own small library (radiosaber_b200/librs_nccl.so = this header's entry points, linked against
 * libnccl.so.2 and librs_sched.so) so that librs_sched.so itself carries no NCCL dependency.  In a process that also
 * uses PyTorch, import torch BEFORE loading this library: both then share torch's bundled NCCL (the loader resolves
 * libnccl.so.2 to the copy already in the process); the other way round torch finds the system's older NCCL and fails.
 *
 * What this replaces.  The reference runs ONE cell per process (nbCells = 1,
 * src/scenarios/single-cell-with-interference.h:74), one process per seed
 * (NSDI23-radiosaber-experiments/exp-customization/run_backlogged.sh:5-12), and sums the per-slice bytes of all
 * runs afterwards in NSDI23-radiosaber-experiments/exp-customization/plot_throughput.py:26-56.  Here the cells of a
 * batch are block-partitioned over the GPUs of one box (no traffic between GPUs inside a TTI) and ONE ncclReduce
 * over NVLink sums the per-slice totals at the end of the run (SURVEY.md section 8(e)).  The totals are integers, so
 * the result is the same bits whatever the reduction order.
 */
#ifndef RS_SCHED_NCCL_H_
#define RS_SCHED_NCCL_H_

#include "rs_sched.h"

#ifdef __cplusplus
extern "C" {
#endif

#define RS_NCCL_ID_BYTES 128   /* sizeof(ncclUniqueId) */

/* Message of the last failing call of THIS library on this thread. */
const char* rs_nccl_last_error(void);

/* One communicator per GPU of this process (ncclCommInitAll): comms[i] drives devices[i].  For the one-thread-per-GPU
 * host (radiosaber_b200/host/rs_batch_main.cpp --gpus N). */
int rs_comm_init_all(int32_t n, const int32_t* devices, void** comms);
/* One process per GPU: rank 0 makes the id, every rank receives it out of band (e.g. through the launcher's
 * store) and joins with its own rank and device. */
int rs_comm_unique_id(void* id_out /* RS_NCCL_ID_BYTES */);
int rs_comm_init_rank(int32_t n_ranks, int32_t rank, const void* id /* RS_NCCL_ID_BYTES */, int32_t device, void** comm);
void rs_comm_destroy(void* comm);

/* rs_stats_device() of this rank's cells, then ncclReduce(sum, root) of the uint64 [P][4][S] block on the handle's
 * stream; on the root the totals over all ranks' cells are copied to stats_out (HOST uint64 [P][4][S]; ignored on the
 * other ranks).  nccl_comm is an ncclComm_t passed as void*.  Every rank of the communicator must call it;
 * synchronous. */
int rs_reduce_stats(rs_handle* h, void* nccl_comm, int32_t root, uint64_t* stats_out);

#ifdef __cplusplus
}
#endif
#endif /* RS_SCHED_NCCL_H_ */
