/* rs_nccl.cpp -- include/rs_sched_nccl.h: the end-of-run NCCL reduce of the per-slice totals (SURVEY 8e),
 * include/rs_sched_nccl_buffers.h: the same for the per-slice buffer totals, include/rs_sched_nccl_hol_hist.h: the
 * same for the head-of-line delay histograms, include/rs_sched_nccl_ue_rate.h: the same for the per-UE throughput
 * histograms, and include/rs_sched_nccl_ue_upt.h: the same for the throughput over active time (UPT) histograms.
 * Uses only the public ABI of librs_sched.so plus NCCL and the CUDA runtime. */
#include "../../include/rs_sched_nccl_ue_upt.h"

#include <cuda_runtime.h>
#include <nccl.h>

#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

static_assert(sizeof(ncclUniqueId) == RS_NCCL_ID_BYTES, "ncclUniqueId size");

namespace {
thread_local std::string g_nccl_err;
int nfail(const char* what, const char* why) {
  g_nccl_err = std::string(what) + ": " + why;
  return RS_ERR_CUDA;
}
#define NC(call)                                                            \
  do {                                                                      \
    ncclResult_t r_ = (call);                                               \
    if (r_ != ncclSuccess) return nfail(#call, ncclGetErrorString(r_));     \
  } while (0)
#define CUR(call)                                                           \
  do {                                                                      \
    cudaError_t e_ = (call);                                                \
    if (e_ != cudaSuccess) return nfail(#call, cudaGetErrorString(e_));     \
  } while (0)

/* fill(h, d) writes this rank's uint64 [P][rows][S] totals to device memory; one ncclReduce(sum) on the handle's stream
 * adds them up on the root, which copies them to stats_out. */
int reduce_totals(rs_handle* h, void* nccl_comm, int32_t root, uint64_t* stats_out, int rows,
                  int (*fill)(rs_handle*, uint64_t*), const char* name, const char* fill_name) {
  if (!h || !nccl_comm) return nfail(name, "bad argument");
  ncclComm_t comm = (ncclComm_t)nccl_comm;
  int32_t S = 0, dev = 0;
  if (rs_dims(h, nullptr, &S, nullptr, nullptr, &dev) != RS_OK || S < 1) return nfail("rs_dims", rs_last_error());
  const size_t n = (size_t)rows * S * rs_n_profiles(h);
  int rank = -1;
  NC(ncclCommUserRank(comm, &rank));
  CUR(cudaSetDevice(dev));
  cudaStream_t st = (cudaStream_t)rs_get_stream(h);
  uint64_t* d = nullptr;
  CUR(cudaMalloc((void**)&d, sizeof(uint64_t) * n));
  int rc = fill(h, d);
  if (rc != RS_OK) { cudaFree(d); return nfail(fill_name, rs_last_error()); }
  ncclResult_t r = ncclReduce(d, d, n, ncclUint64, ncclSum, root, comm, st);
  cudaError_t e = cudaSuccess;
  if (r == ncclSuccess && rank == root && stats_out)
    e = cudaMemcpyAsync(stats_out, d, sizeof(uint64_t) * n, cudaMemcpyDeviceToHost, st);
  if (r == ncclSuccess && e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(d);
  if (r != ncclSuccess) return nfail("ncclReduce", ncclGetErrorString(r));
  if (e != cudaSuccess) return nfail(name, cudaGetErrorString(e));
  return RS_OK;
}
}  // namespace

extern "C" {

const char* rs_nccl_last_error(void) { return g_nccl_err.c_str(); }

int rs_comm_init_all(int32_t n, const int32_t* devices, void** comms) {
  if (n < 1 || !devices || !comms) return nfail("rs_comm_init_all", "bad argument");
  std::vector<ncclComm_t> c((size_t)n);
  std::vector<int> dev(devices, devices + n);
  NC(ncclCommInitAll(c.data(), n, dev.data()));
  for (int i = 0; i < n; ++i) comms[i] = (void*)c[(size_t)i];
  return RS_OK;
}

int rs_comm_unique_id(void* id_out) {
  if (!id_out) return nfail("rs_comm_unique_id", "bad argument");
  ncclUniqueId id;
  NC(ncclGetUniqueId(&id));
  memcpy(id_out, &id, sizeof id);
  return RS_OK;
}

int rs_comm_init_rank(int32_t n_ranks, int32_t rank, const void* id_in, int32_t device, void** comm) {
  if (n_ranks < 1 || rank < 0 || rank >= n_ranks || !id_in || !comm) return nfail("rs_comm_init_rank", "bad argument");
  ncclUniqueId id;
  memcpy(&id, id_in, sizeof id);
  CUR(cudaSetDevice(device));
  ncclComm_t c;
  NC(ncclCommInitRank(&c, n_ranks, id, rank));
  *comm = (void*)c;
  return RS_OK;
}

void rs_comm_destroy(void* comm) {
  if (comm) ncclCommDestroy((ncclComm_t)comm);
}

int rs_reduce_stats(rs_handle* h, void* nccl_comm, int32_t root, uint64_t* stats_out) {
  return reduce_totals(h, nccl_comm, root, stats_out, 4, rs_stats_device, "rs_reduce_stats", "rs_stats_device");
}

int rs_reduce_buffer_stats(rs_handle* h, void* nccl_comm, int32_t root, uint64_t* stats_out) {
  return reduce_totals(h, nccl_comm, root, stats_out, 3, rs_buffer_stats_device, "rs_reduce_buffer_stats",
                       "rs_buffer_stats_device");
}

int rs_reduce_hol_hist(rs_handle* h, void* nccl_comm, int32_t root, uint64_t* hist_out) {
  const int32_t bins = rs_hol_hist_bins(h);   /* [P][2][S][bins]: 2 x bins rows per slice */
  if (h && bins == 0) return nfail("rs_hol_hist_device", "the handle has no delay histogram (rs_enable_hol_hist)");
  return reduce_totals(h, nccl_comm, root, hist_out, 2 * bins, rs_hol_hist_device, "rs_reduce_hol_hist",
                       "rs_hol_hist_device");
}

int rs_reduce_ue_rate_hist(rs_handle* h, void* nccl_comm, int32_t root, uint64_t* hist_out) {
  const int32_t bins = rs_ue_rate_hist_bins(h);   /* [P][S][bins]: bins rows per slice */
  if (h && bins == 0)
    return nfail("rs_ue_rate_hist_device", "the handle has no throughput histogram (rs_enable_ue_rate_hist)");
  return reduce_totals(h, nccl_comm, root, hist_out, bins, rs_ue_rate_hist_device, "rs_reduce_ue_rate_hist",
                       "rs_ue_rate_hist_device");
}

int rs_reduce_ue_upt_hist(rs_handle* h, void* nccl_comm, int32_t root, uint64_t* hist_out) {
  const int32_t bins = rs_ue_upt_hist_bins(h);   /* [P][S][bins]: bins rows per slice */
  if (h && bins == 0)
    return nfail("rs_ue_upt_hist_device", "the handle has no UPT histogram (rs_enable_ue_upt_hist)");
  return reduce_totals(h, nccl_comm, root, hist_out, bins, rs_ue_upt_hist_device, "rs_reduce_ue_upt_hist",
                       "rs_ue_upt_hist_device");
}

}  /* extern "C" */
