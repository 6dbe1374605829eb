/* rs_sched.cu -- host side of the C ABI declared in include/rs_sched.h.
 *
 * Owns the device state of a batch of cells, builds the lookup tables the kernels use (with the
 * host's glibc, so that every libm value is the one the reference's x86-64 build computes) and
 * launches the sm_100a kernels of rs_device.cuh.  No CPU implementation of the scheduling path
 * lives here: without a CUDA device every compute entry point fails with RS_ERR_CUDA.
 */
#include "../../include/rs_sched.h"
#include "rs_kernels.h"
/* the device code twice: rs:: = 128 threads per cell, eight cells per SM (the headline shape);
 * rsw:: = 512 threads per cell, two per SM, for cells with hundreds of UEs */
#define RS_NS rs
#ifndef RS_NARROW_THREADS
#define RS_NARROW_THREADS 128   /* experiments: -DRS_NARROW_THREADS=256 -DRS_NARROW_MIN_BLOCKS=4 */
#endif
#define RS_THREADS RS_NARROW_THREADS
#ifndef RS_NARROW_MIN_BLOCKS
#define RS_NARROW_MIN_BLOCKS 8   /* cells per SM the 128-thread kernels are compiled for (register cap 65536 / 128 / this) */
#endif
#define RS_MIN_BLOCKS RS_NARROW_MIN_BLOCKS
#include "rs_device.cuh"
#undef RS_NS
#undef RS_THREADS
#undef RS_MIN_BLOCKS
#ifndef RS_WIDE_THREADS
#define RS_WIDE_THREADS 512
#define RS_WIDE_MIN_BLOCKS 2
#endif
#define RS_NS rsw
#define RS_THREADS RS_WIDE_THREADS
#define RS_MIN_BLOCKS RS_WIDE_MIN_BLOCKS
#define RS_CORE_ONLY
#include "rs_device.cuh"
#undef RS_NS
#undef RS_THREADS
#undef RS_MIN_BLOCKS
#undef RS_CORE_ONLY

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) return fail(RS_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_));      \
  } while (0)

/* ---- AMC tables: standard LTE data (3GPP TS 36.213), same values as AMCModule.cpp:36-231 ------- */
const double kSinrForCqi[15] = {-4.63, -2.6, -0.12, 2.26, 4.73, 7.53, 8.67, 11.32,
                                14.24, 15.21, 18.63, 21.32, 23.47, 28.49, 34.6};
const int kMcsToItbs[29] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 10, 11, 12, 13, 14, 15, 15, 16,
                            17, 18, 19, 20, 21, 22, 23, 24, 25, 26};
const int kTbs[110 * 27] = {
#include "../../include/rs_tbs_36213.inc"
};
inline int mcs_from_cqi(int cqi) { return 2 * (cqi - 1); }          /* MapCQIToMCS */
inline int tbs_row(int row, int itbs, const int32_t* row_m1) {
  return row < 0 ? row_m1[itbs] : kTbs[row * 27 + itbs];
}
/* AMCModule::GetTBSizeFromMCS(mcs, nbRBs), AMCModule.cpp:305-317 incl. the row -1 read (SURVEY H2) */
int tbs_n(int mcs, int nb_rbs, const int32_t* row_m1) {
  const int itbs = kMcsToItbs[mcs];
  if (nb_rbs <= 110) return tbs_row(nb_rbs - 1, itbs, row_m1);
  return 5 * tbs_row(nb_rbs / 5 - 1, itbs, row_m1) + tbs_row(nb_rbs % 5 - 1, itbs, row_m1);
}
/* AMCModule::GetEfficiencyFromCQI, AMCModule.cpp:319-327 */
double eff_from_cqi(int cqi) {
  const int bits = kTbs[kMcsToItbs[mcs_from_cqi(cqi)]];
  volatile double eff = (bits / 0.001) / 180000.;
  return eff;
}
/* The stock -O0 build reads McsToItbs[5..28],0,0,0 for TransportBlockSizeTable[-1] (oracle/_ref probe). */
void default_row_m1(int32_t* out) {
  for (int i = 0; i < 27; ++i) out[i] = (i + 5 < 29) ? kMcsToItbs[i + 5] : 0;
}

/* 10*log10(-log(mean)) as GetEesmEffectiveSinr computes it (eesm-effective-sinr.h:42-44, beta = 1) */
double eesm_tail(double mean) {
  volatile double beta = 1;
  volatile double eff = -beta * log(mean);
  return 10 * log10(eff);
}

bool build_const_tables(rs::ConstTables* t, std::string* why) {
  memset(t, 0, sizeof *t);
  for (int c = 1; c <= 15; ++c) {
    volatile double s = pow(10, kSinrForCqi[c - 1] / 10);
    volatile double beta = 1;
    t->tval[c] = exp(-s / beta);
    t->eff[c] = eff_from_cqi(c);
  }
  t->tval[0] = t->tval[1];
  for (int k = 1; k <= 14; ++k) {
    const double thr = kSinrForCqi[k];
    auto pred = [&](uint64_t bits) {
      double m;
      memcpy(&m, &bits, 8);
      return thr <= eesm_tail(m);
    };
    uint64_t lo = 0, hi;             /* pred(lo) true (mean 0 -> +inf dB), pred(hi) false (mean 1 -> -inf dB) */
    const double one = 1.0;
    memcpy(&hi, &one, 8);
    if (!pred(lo) || pred(hi)) { *why = "EESM threshold bracket"; return false; }
    while (hi - lo > 1) {
      const uint64_t mid = lo + (hi - lo) / 2;
      if (pred(mid)) lo = mid; else hi = mid;
    }
    /* glibc's log/log10 must be monotone around the cut for the single comparison to be exact */
    for (uint64_t d = 1; d <= 512; ++d) {
      if (lo >= d && !pred(lo - d)) { *why = "EESM tail not monotone below a cut"; return false; }
      if (pred(lo + d)) { *why = "EESM tail not monotone above a cut"; return false; }
    }
    memcpy(&t->cut[k], &lo, 8);
  }
  for (int k = 2; k <= 14; ++k)
    if (!(t->cut[k] <= t->cut[k - 1])) { *why = "EESM cuts not ordered"; return false; }
  return true;
}

/* What libstdc++'s __introsort_loop does to a range of `len` EQUAL keys is independent of the data:
 * __move_median_to_first picks `mid` (every comparison is false, stl_algo.h:1893-1899),
 * __unguarded_partition stops on every element from both sides, i.e. swaps pair k of
 * (first+1+k, last-1-k) while the former is left of the latter and returns first+1+(len-1)/2, and
 * the two halves recurse the same way until they are <= 16 long.  tab[eq_offset(len)+i] = index,
 * in the range as it is AFTER the first median swap, of the entry that ends at position i. */
void build_eq_table(int nmax, std::vector<unsigned short>* tab) {
  tab->assign(nmax >= 17 ? rs::eq_offset(nmax + 1) : 1, 0);
  std::vector<unsigned short> a(nmax > 0 ? nmax : 1);
  std::vector<std::pair<int, int>> stack;
  for (int len = 17; len <= nmax; ++len) {
    for (int i = 0; i < len; ++i) a[i] = (unsigned short)i;
    stack.clear();
    stack.emplace_back(0, len);
    while (!stack.empty()) {
      int f = stack.back().first, l = stack.back().second;
      stack.pop_back();
      while (l - f > 16) {
        std::swap(a[f], a[f + (l - f) / 2]);
        for (int k = 0; f + 1 + k < l - 1 - k; ++k) std::swap(a[f + 1 + k], a[l - 1 - k]);
        const int cut = f + 1 + (l - f - 1) / 2;
        stack.emplace_back(cut, l);
        l = cut;
      }
    }
    unsigned short* out = tab->data() + rs::eq_offset(len);
    const int mid = len / 2;
    for (int i = 0; i < len; ++i) {
      const int x = a[i];
      out[i] = (unsigned short)(x == 0 ? mid : (x == mid ? 0 : x));
    }
  }
}
/* VogelApproximate's gaps (transport.cpp:378-451): e1 - e2 over the AMC efficiencies of CQI 0..15 (0 = a slice without a
 * listed user) with e2 = -1 when a line has no second element.  tab[k1 * 17 + k2 + 1] = dense rank of that double among
 * all 272 (equal doubles, equal ranks); tab[272 + r + 1] = rank of the largest gap <= (double)(int)gap_r, -1 if none:
 * "candidate gap > (int) running maximum" is then a comparison of ranks.  Index 272 (running maximum "none") holds the
 * threshold of max_diff's initial -1. */
void build_vogel_tab(std::vector<short>* tab) {
  double eff[17];
  eff[0] = -1.0;   /* k2 = -1 */
  eff[1] = 0.0;    /* CQI 0 */
  for (int c = 1; c <= 15; ++c) eff[c + 1] = eff_from_cqi(c);
  std::vector<double> gaps;
  for (int k1 = 0; k1 < 16; ++k1)
    for (int k2 = -1; k2 < 16; ++k2) { volatile double g = eff[k1 + 1] - eff[k2 + 1]; const double gv = g; gaps.push_back(gv); }
  std::vector<double> uniq(gaps);
  std::sort(uniq.begin(), uniq.end());
  uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
  tab->assign(rs::kVogelTab, 0);
  for (size_t i = 0; i < gaps.size(); ++i)
    (*tab)[i] = (short)(std::lower_bound(uniq.begin(), uniq.end(), gaps[i]) - uniq.begin());
  auto thr_of = [&](double running_max) {   /* rank of the largest gap <= (double)(int)running_max */
    const double t = (double)(int)running_max;
    return (short)((std::upper_bound(uniq.begin(), uniq.end(), t) - uniq.begin()) - 1);
  };
  (*tab)[272] = thr_of(-1.0);
  for (size_t r = 0; r < uniq.size(); ++r) (*tab)[272 + 1 + r] = thr_of(uniq[r]);
}
constexpr int kEqMax = 2048;
#ifndef RS_WIDE_MIN_UES
#define RS_WIDE_MIN_UES 480   /* cells with at least this many UEs run 512 threads wide (tools/sweep_bench.py) */
#endif
#ifndef RS_STAGE_MIN_FIT
#define RS_STAGE_MIN_FIT 8   /* narrow cells: staging the CQI must leave room for this many cells per SM (or all the batch offers) */
#endif

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  cudaError_t alloc(size_t count) {
    if (count <= n && p) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
    cudaError_t e = cudaMalloc((void**)&p, std::max<size_t>(count, 1) * sizeof(T));
    if (e == cudaSuccess) n = count;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};

}  // namespace

struct rs_handle {
  int device = 0;
  rs::DevCfg d{};
  int B = 0, cqi_cols = 0;           /* cqi_cols = G or R */
  rs::Layout layout{};
  cudaStream_t own_stream = nullptr, stream = nullptr;
  cudaStream_t copy_in = nullptr, copy_out = nullptr;
  /* Big batches run as up to four part-batches on as many streams: each part's launches are chained on its own stream,
   * so the partial last wave of one part's launch is filled by CTAs of another part's launch instead of leaving SMs
   * idle until the grid drains (4096 cells = 3.46 waves of 1184 resident cells: +5-10 %, profiles/README.md). */
  static constexpr int kMaxParts = 4;
  cudaStream_t xs[kMaxParts - 1] = {};    /* streams of parts 1.. (part 0 runs on `stream`) */
  cudaEvent_t join_evs[kMaxParts - 1] = {};
  cudaEvent_t fork_ev = nullptr, join_ev = nullptr;
  int parts = 1;
  int64_t launches = 0;
  int P = 1;                         /* slice profiles (rs_create_profiles) */
  DevBuf<int> cell_profile;          /* [B], allocated when P > 1 */
  int32_t row_m1[27];
  /* static tables */
  DevBuf<int> ue_to_slice, slice_ptr, slice_ues, chunk_slice, tbs_n;
  DevBuf<double> weight, epow;
  DevBuf<unsigned char> psi;
  DevBuf<unsigned short> eq_tab;
  /* state */
  DevBuf<double> avg, offset, ewma;
  DevBuf<int> tx;
  DevBuf<unsigned long long> cum_bytes, cum_rbs;
  /* trace-driven CQI (rs_set_traces) */
  DevBuf<uint8_t> trace_tab;
  DevBuf<int> ue_trace_off;
  int n_traces = 0, trace_rows = 0;
  bool stage_ok = false;   /* the layout has room for a TTI of CQI (staged in shared memory) */
  bool wide = false;       /* 512 threads per cell (rsw::) instead of 128 */
  int fixed = -1;          /* >= 0: the FixedShape instantiation this handle's backlogged launches use (fixed_kernel) */
  /* queue state for the next run call (rs_set_queues), consumed by it */
  const int32_t* q_next = nullptr;
  const double* hol_next = nullptr;
  DevBuf<unsigned char> holmul;
  /* per-bearer FIFOs (rs_enable_buffers): buf_k records per bearer, 0 = off */
  int buf_k = 0;
  DevBuf<rs::BufMeta> buf_meta;
  DevBuf<double> buf_time;
  DevBuf<int> buf_bytes;
  std::vector<unsigned char> buf_backlogged;   /* [B][U][nb], what rs_reset_state restores */
  double last_now = -HUGE_VAL;                 /* `now` of the last TTI run on the buffers */
  bool traffic_set = false;                    /* rs_set_traffic for the next run call, consumed by it */
  rs_traffic traffic{};
  DevBuf<int> shown_q;                         /* rs_run_device without queue_out / hol_out: what the TTIs show */
  DevBuf<double> shown_hol;
  DevBuf<int> synth_spec;                      /* rs_synth_arrivals' [P][S][2] */
  DevBuf<unsigned char> buf_scratch;           /* rs_get_buffers */
  DevBuf<int> tbs1;
  DevBuf<short> vogel_tab;
  DevBuf<unsigned long long> stats;
  /* staging for rs_step / rs_run_host*: a ring of slots that stays in flight across calls.  Chunk n of the
   * handle's lifetime uses slot n % kSlots; a slot is refilled once the kernel that read it is done (k_done) and
   * its kernel starts once the previous results have left it (out_done) -- all stream-side waits, the host never
   * blocks while enqueueing. */
  static constexpr int kSlots = 3;
  struct Slot {
    DevBuf<uint8_t> cqi, active, mcs, final_cqi;
    DevBuf<int> rand2, tbs_bits, slice_target, slice_quota, nvs_slice;
    DevBuf<short> rbg_to_ue, alloc_ue, alloc_rbg;
    DevBuf<int> alloc_n, queue, arrivals;
    DevBuf<double> hol;
    cudaEvent_t in_done = nullptr, k_done = nullptr, out_done = nullptr;
    cudaEvent_t k_done_x[3] = {};   /* kernel-done events of parts 1.. */
    bool k_rec = false, out_rec = false;   /* the events have been recorded at least once */
  } slot[kSlots];
  uint64_t chunk_seq = 0;
  /* CQI slabs shared by consecutive chunks (rs_run_host with a refresh > 1): two buffers, the kernels of the slab
   * before last must be done before it is overwritten */
  struct Slab {
    DevBuf<uint8_t> cqi;
    cudaEvent_t used = nullptr, used_x[3] = {};   /* recorded after the last kernel (of each part) that read the slab */
    bool used_rec = false;
    int index = -1;               /* slab of the CURRENT call resident here */
  } slab[2];
  /* completion of whole rs_run_host* calls: ticket n -> call_done[n % kTickets] (recorded on copy_out) */
  static constexpr int kTickets = 16;
  cudaEvent_t call_done[kTickets] = {};
  int64_t calls = 0;
  /* rs_step_cell: one pinned and one device mailbox (inputs | state | outputs) */
  unsigned char* mb_host = nullptr;
  DevBuf<unsigned char> mb_dev;
  size_t mb_bytes = 0;
};

namespace {

static_assert(sizeof(rs::DevCfg) == sizeof(rsw::DevCfg) && sizeof(rs::RunArgs) == sizeof(rsw::RunArgs) &&
                  sizeof(rs::ConstTables) == sizeof(rsw::ConstTables),
              "the two instantiations of rs_device.cuh share their parameter structs");

/* one kernel per (scheduler id, CQI source, backlogged / queue-aware, CTA width); the instantiations live in five
 * translation units of their own (rs_kernels.cu) */
const void* tti_kernel_any(int algo, bool trace, bool queue, bool wide) {
  const bool first = algo == 9 || algo == 8 || algo == 10 || algo == 1;
  if (wide) return first ? rs_kernel_tu3(algo, trace, queue) : rs_kernel_tu4(algo, trace, queue);
  return first ? rs_kernel_tu1(algo, trace, queue) : rs_kernel_tu2(algo, trace, queue);
}
/* The headline cell -- 20 slices x 5 UEs, 64 RBGs of 8 RBs, one CQI value per RBG (u8 or 4-bit), backlogged, ids 9,
 8, 10, 101 and 103 (the transport ids: same layout) and the NVS ids 7 and 11 -- has FixedShape instantiations of the TTI kernel (rs_device.cuh): same code, dimensions and shared-memory
 * layout known at compile time.  A handle uses one only if its configuration and its host-computed layout match the
 * instantiation exactly; RS_NO_FIXED_SHAPE=1 in the environment keeps every handle on the general kernel. */
using FixedU8 = rs::FixedShape<20, 5, 64, 8, 0>;
using FixedNib = rs::FixedShape<20, 5, 64, 8, 2>;
template <class SH>
bool shape_matches(const rs_handle* h, const std::vector<int>& u2s) {
  const rs::DevCfg& d = h->d;
  if (h->wide || d.nb != 1 || d.S != SH::S || d.U != SH::U || d.G != SH::G || d.rbg != SH::RBG || d.cqi_per_rb != SH::LAY ||
      d.n_chunks != SH::chunks(d.algo) || d.m_cap != SH::mcap(d.algo) || d.sort_n != SH::kSortN || d.sort_depth != SH::kSortDepth ||
      !h->stage_ok || d.direct)
    return false;
  for (size_t i = 0; i < u2s.size(); ++i)   /* every profile ([P][U]): weights and parameters may differ */
    if (u2s[i] != (int)(i % (size_t)d.U) / SH::UPS) return false;
  const rs::Layout want = SH::layout(h->d.algo);
  return memcmp(&want, &h->layout, sizeof want) == 0;
}
bool has_fixed_kernel(int algo) { return algo == 9 || algo == 8 || algo == 10 || algo == 101 || algo == 103 || algo == 7 || algo == 11; }
const void* fixed_kernel(int algo, int which, bool trace) {
  return (algo == 7 || algo == 11) ? rs_kernel_tu6(algo, which, trace) : rs_kernel_tu5(algo, which, trace);
}

/* part < 0: the whole batch on the handle's stream; part p of h->parts: cells [p B / P, (p + 1) B / P) on stream / xs[p-1] */
int launch_ttis(rs_handle* h, const rs::RunArgs& a0, bool trace, const rs::DevCfg* cfg = nullptr, int part = -1) {
  rs::RunArgs a = a0;
  int n = h->B;
  cudaStream_t st = h->stream;
  if (part >= 0) {
    const long long lo = (long long)h->B * part / h->parts, hi = (long long)h->B * (part + 1) / h->parts;
    a.cell_off = (int)lo;
    n = (int)(hi - lo);
    if (part > 0) st = h->xs[part - 1];
    if (n <= 0) return RS_OK;
  }
  const dim3 grid(n), block(h->wide ? rsw::kThreads : rs::kThreads);
  const size_t sm = (size_t)h->layout.total;
  /* by address: the rsw:: kernels take rsw::DevCfg / rsw::RunArgs, the same bytes as the rs:: structs */
  const void* fn = (h->fixed >= 0 && !a.queue) ? fixed_kernel(h->d.algo, h->fixed, trace)
                                               : tti_kernel_any(h->d.algo, trace, a.queue != nullptr, h->wide);
  void* args[2] = {(void*)(cfg ? cfg : &h->d), (void*)&a};
  CU(cudaLaunchKernel(fn, grid, block, args, sm, st));
  CU(cudaGetLastError());
  h->launches++;
  return RS_OK;
}

/* cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the kernel function (per device), not to a handle:
 * every instantiation is opened up to the device's opt-in maximum once, so handles of different cell sizes
 * can be alive together and launch in any order. */
int set_smem_attr(rs_handle* h) {
  int max_optin = 0;
  CU(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
  for (int t = 0; t < 4; ++t)
    CU(cudaFuncSetAttribute(tti_kernel_any(h->d.algo, (t & 1) != 0, (t & 2) != 0, h->wide),
                            cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin));
  if (h->fixed >= 0)
    for (int t = 0; t < 2; ++t)
      CU(cudaFuncSetAttribute(fixed_kernel(h->d.algo, h->fixed, t != 0), cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin));
  return RS_OK;
}

/* dt and trace rows of one launch ride in the kernel parameters.  trace_row -1 = no report received yet: the
 * extra all-10 row behind every trace (ENodeB.cpp:207-217). */
void fill_scalars(const rs_handle* h, rs::RunArgs* a, const double* dt, const int32_t* trace_row, int T) {
  for (int t = 0; t < T; ++t) {
    a->dt[t] = dt[t];
    a->trace_row[t] = trace_row ? (trace_row[t] < 0 ? h->trace_rows : trace_row[t]) : 0;
  }
}
int check_trace_rows(const rs_handle* h, const int32_t* trace_row, int n) {
  for (int t = 0; t < n; ++t)
    if (trace_row[t] < -1 || trace_row[t] >= h->trace_rows)
      return fail(RS_ERR_ARG, "trace_row[%d] = %d outside -1..%d", t, trace_row[t], h->trace_rows - 1);
  return RS_OK;
}

template <typename T>
int upload(DevBuf<T>& b, const std::vector<T>& v) {
  CU(b.alloc(v.size()));
  if (!v.empty()) CU(cudaMemcpy(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return RS_OK;
}

int alloc_slot(rs_handle* h, rs_handle::Slot& s, int T, const rs_outputs* out, bool want_active, bool want_cqi,
               bool want_queue, bool want_hol, bool want_arrivals) {
  const size_t B = h->B, U = h->d.U, S = h->d.S, G = h->d.G, C = h->cqi_cols;
  if (want_cqi) CU(s.cqi.alloc((size_t)T * B * U * C));
  CU(s.rand2.alloc((size_t)T * B * std::max(h->d.rand_stride, 1)));
  if (want_active) CU(s.active.alloc((size_t)T * B * U));
  if (want_queue) CU(s.queue.alloc((size_t)T * B * U * h->d.nb));
  if (want_hol) CU(s.hol.alloc((size_t)T * B * U * h->d.nb));
  if (want_arrivals) CU(s.arrivals.alloc((size_t)T * B * U * h->d.nb));
  if (out) {
    if (out->rbg_to_ue) CU(s.rbg_to_ue.alloc((size_t)T * B * G));
    if (out->tbs_bits) CU(s.tbs_bits.alloc((size_t)T * B * U));
    if (out->mcs) CU(s.mcs.alloc((size_t)T * B * U));
    if (out->final_cqi) CU(s.final_cqi.alloc((size_t)T * B * U));
    if (out->slice_target) CU(s.slice_target.alloc((size_t)T * B * S));
    if (out->slice_quota) CU(s.slice_quota.alloc((size_t)T * B * S));
    if (out->nvs_slice) CU(s.nvs_slice.alloc((size_t)T * B));
    if (h->d.algo == 10) {
      if (out->alloc_n) CU(s.alloc_n.alloc((size_t)T * B));
      if (out->alloc_ue) CU(s.alloc_ue.alloc((size_t)T * B * h->d.grant_len));
      if (out->alloc_rbg) CU(s.alloc_rbg.alloc((size_t)T * B * h->d.grant_len));
    }
  }
  if (!s.in_done) {
    CU(cudaEventCreateWithFlags(&s.in_done, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&s.k_done, cudaEventDisableTiming));
    for (auto& e : s.k_done_x) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&s.out_done, cudaEventDisableTiming));
  }
  return RS_OK;
}

/* DownlinkTransportScheduler with one of its inter-slice algorithms (the constructor's second argument):
 * 8 GreedyByRow (0), 9 MaximizeCell (2), 10 UpperBound (4); SubOpt (1) and VogelApproximate (3) have no id in the
 * SingleCellWithI scenario (ENodeB.cpp:363-379) and go by 100 + that argument */
bool is_transport(int a) { return a == 8 || a == 9 || a == 10 || a == 101 || a == 103; }

/* the rs_config fields every profile of a handle shares; tbs_row_m1 by value (NULL = the stock row) */
int check_shared_fields(const rs_config* c, int P) {
  int32_t row0[27], row[27];
  if (c[0].tbs_row_m1) memcpy(row0, c[0].tbs_row_m1, sizeof row0); else default_row_m1(row0);
  for (int p = 1; p < P; ++p) {
    const rs_config& a = c[0];
    const rs_config& x = c[p];
    if (x.tbs_row_m1) memcpy(row, x.tbs_row_m1, sizeof row); else default_row_m1(row);
    const char* f = x.algo != a.algo ? "algo" : x.n_slices != a.n_slices ? "n_slices" : x.n_ues != a.n_ues ? "n_ues"
                  : x.n_rbs != a.n_rbs ? "n_rbs" : x.rbg_size != a.rbg_size ? "rbg_size"
                  : x.cqi_per_rb != a.cqi_per_rb ? "cqi_per_rb" : x.data_to_transmit != a.data_to_transmit ? "data_to_transmit"
                  : x.n_bearers != a.n_bearers ? "n_bearers" : memcmp(row, row0, sizeof row) ? "tbs_row_m1" : nullptr;
    if (f) return fail(RS_ERR_ARG, "rs_create_profiles: profile %d: %s differs from profile 0 (profiles share it)", p, f);
  }
  return RS_OK;
}

/* Every FIFO empty, the backlogged bearers flagged (n = -1), counters 0 and no `now` seen yet.  The caller has waited
 * for the handle's work. */
int buf_empty(rs_handle* h) {
  h->last_now = -HUGE_VAL;
  if (h->buf_k == 0) return RS_OK;
  std::vector<rs::BufMeta> m(h->buf_backlogged.size());
  for (size_t i = 0; i < m.size(); ++i) m[i] = rs::BufMeta{0, 0, 0, h->buf_backlogged[i] ? -1 : 0};
  CU(cudaMemcpy(h->buf_meta.p, m.data(), m.size() * sizeof(rs::BufMeta), cudaMemcpyHostToDevice));
  return RS_OK;
}

/* A buffered handle's traffic for a call of n TTIs (rs_set_traffic), consumed by the call; the times are checked here,
 * before anything is enqueued. */
int take_traffic(rs_handle* h, int n, rs_traffic* tr) {
  const bool set = h->traffic_set;
  *tr = h->traffic;
  h->traffic_set = false;
  if (h->buf_k == 0) return RS_OK;
  if (!set) return fail(RS_ERR_ARG, "buffered handle: every run call needs rs_set_traffic");
  if (n > 0 && (!tr->arrivals || !tr->now || !tr->arrival_time))
    return fail(RS_ERR_ARG, "rs_set_traffic: arrivals, now and arrival_time are required");
  double prev = h->last_now;
  for (int t = 0; t < n; ++t) {
    if (!(tr->now[t] >= prev))
      return fail(RS_ERR_ARG, "rs_set_traffic: now[%d] = %.17g is before the previous TTI's %.17g", t, tr->now[t], prev);
    if (!(tr->arrival_time[t] <= tr->now[t]))
      return fail(RS_ERR_ARG, "rs_set_traffic: arrival_time[%d] = %.17g is after now[%d] = %.17g", t, tr->arrival_time[t], t,
                  tr->now[t]);
    prev = tr->now[t];
  }
  return RS_OK;
}
/* the FIFOs and the times of TTIs [t0, t0 + T) of a buffered call (the caller points a->arrivals at the launch's rows) */
void fill_buffers(const rs_handle* h, rs::RunArgs* a, const rs_traffic& tr, int t0, int T) {
  a->buf_k = h->buf_k;
  a->buf_meta = h->buf_meta.p;
  a->buf_time = h->buf_time.p;
  a->buf_bytes = h->buf_bytes.p;
  for (int t = 0; t < T; ++t) {
    a->now[t] = tr.now[t0 + t];
    a->arr_time[t] = tr.arrival_time[t0 + t];
  }
}

bool wants(const rs_handle* h, int which) { /* outputs that exist for this scheduler id */
  const int a = h->d.algo;
  if (which == 0) return is_transport(a);   /* slice_target / slice_quota */
  return a == 7 || a == 11;                  /* nvs_slice */
}

}  // namespace

extern "C" {

const char* rs_last_error(void) { return g_err.c_str(); }
int32_t rs_abi_version(void) { return 3; }

void rs_destroy(rs_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (auto st : h->xs) if (st) cudaStreamSynchronize(st);
  if (h->copy_in) cudaStreamSynchronize(h->copy_in);
  if (h->copy_out) cudaStreamSynchronize(h->copy_out);
  h->ue_to_slice.release(); h->slice_ptr.release(); h->slice_ues.release(); h->chunk_slice.release();
  h->tbs_n.release(); h->weight.release(); h->epow.release(); h->psi.release(); h->eq_tab.release();
  h->avg.release(); h->offset.release(); h->ewma.release(); h->tx.release();
  h->cum_bytes.release(); h->cum_rbs.release(); h->stats.release(); h->cell_profile.release();
  for (auto& s : h->slot) {
    s.cqi.release(); s.active.release(); s.mcs.release(); s.final_cqi.release(); s.rand2.release();
    s.tbs_bits.release(); s.slice_target.release(); s.slice_quota.release(); s.nvs_slice.release();
    s.rbg_to_ue.release(); s.alloc_ue.release(); s.alloc_rbg.release(); s.alloc_n.release();
    s.queue.release(); s.hol.release(); s.arrivals.release();
    if (s.in_done) cudaEventDestroy(s.in_done);
    if (s.k_done) cudaEventDestroy(s.k_done);
    for (auto e : s.k_done_x) if (e) cudaEventDestroy(e);
    if (s.out_done) cudaEventDestroy(s.out_done);
  }
  for (auto& sl : h->slab) { sl.cqi.release(); if (sl.used) cudaEventDestroy(sl.used); for (auto e : sl.used_x) if (e) cudaEventDestroy(e); }
  if (h->fork_ev) cudaEventDestroy(h->fork_ev);
  if (h->join_ev) cudaEventDestroy(h->join_ev);
  for (auto e : h->join_evs) if (e) cudaEventDestroy(e);
  for (auto st : h->xs) if (st) cudaStreamDestroy(st);
  for (auto& e : h->call_done) if (e) cudaEventDestroy(e);
  if (h->mb_host) cudaFreeHost(h->mb_host);
  h->mb_dev.release();
  h->trace_tab.release(); h->ue_trace_off.release();
  h->holmul.release(); h->tbs1.release(); h->vogel_tab.release();
  h->buf_meta.release(); h->buf_time.release(); h->buf_bytes.release(); h->shown_q.release(); h->shown_hol.release();
  h->synth_spec.release(); h->buf_scratch.release();
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  if (h->copy_in) cudaStreamDestroy(h->copy_in);
  if (h->copy_out) cudaStreamDestroy(h->copy_out);
  delete h;
}

int rs_create(const rs_config* cfg, int32_t n_cells, int32_t device, rs_handle** out) {
  return rs_create_profiles(cfg, 1, nullptr, n_cells, device, out);
}

int rs_create_profiles(const rs_config* cfgs, int32_t n_profiles, const int32_t* cell_profile, int32_t n_cells,
                       int32_t device, rs_handle** out) {
  if (!cfgs || !out || n_cells <= 0) return fail(RS_ERR_ARG, "rs_create: bad argument");
  *out = nullptr;
  const int P = n_profiles;
  if (P < 1 || P > n_cells) return fail(RS_ERR_ARG, "rs_create_profiles: n_profiles %d outside 1..n_cells (%d)", P, n_cells);
  if (!cell_profile && P > 1) return fail(RS_ERR_ARG, "rs_create_profiles: cell_profile is NULL with %d profiles", P);
  if (cell_profile)
    for (int b = 0; b < n_cells; ++b)
      if (cell_profile[b] < 0 || cell_profile[b] >= P)
        return fail(RS_ERR_ARG, "rs_create_profiles: cell_profile[%d] = %d outside 0..%d", b, cell_profile[b], P - 1);
  const rs_config* cfg = cfgs;   /* profile 0: every field but weight / params / ue_to_slice holds for all */
  { const int rc = check_shared_fields(cfgs, P); if (rc != RS_OK) return rc; }
  /* "profile p: " in front of the messages of per-profile checks when there is more than one */
  auto pfx = [P](int p) { return P > 1 ? std::string("profile ") + std::to_string(p) + ": " : std::string(); };
  const int algo = cfg->algo, S = cfg->n_slices, U = cfg->n_ues;
  if (algo != 1 && algo != 7 && algo != 11 && !is_transport(algo))
    return fail(RS_ERR_UNSUPPORTED, "scheduler id %d: only 1 (PF), 7 (NVS), 8 (Sequential), 9 (RadioSaber), 10 (UpperBound), "
                "11 (NVS non-greedy), 101 (SubOpt), 103 (VogelApproximate)", algo);
  if (S < 1 || S > RS_MAX_SLICES) return fail(RS_ERR_UNSUPPORTED, "n_slices %d outside 1..%d", S, RS_MAX_SLICES);
  if (U < 1 || U > 32767) return fail(RS_ERR_UNSUPPORTED, "n_ues %d outside 1..32767 (rbg_to_ue / alloc_ue are int16)", U);
  if (cfg->rbg_size < 1 || cfg->n_rbs < cfg->rbg_size || cfg->n_rbs % cfg->rbg_size != 0)
    return fail(RS_ERR_UNSUPPORTED, "n_rbs %d must be a positive multiple of rbg_size %d", cfg->n_rbs, cfg->rbg_size);
  const int G = cfg->n_rbs / cfg->rbg_size;
  if (G > RS_MAX_RBGS) return fail(RS_ERR_UNSUPPORTED, "%d RBGs > %d", G, RS_MAX_RBGS);
  for (int p = 0; p < P; ++p)
    if (!cfgs[p].ue_to_slice || (algo != 1 && (!cfgs[p].weight || !cfgs[p].params)))
      return fail(RS_ERR_ARG, "rs_create: %sweight/params/ue_to_slice missing", pfx(p).c_str());
  const int nb = cfg->n_bearers == 2 ? 2 : 1;
  if (cfg->n_bearers < 0 || cfg->n_bearers > 2) return fail(RS_ERR_ARG, "n_bearers %d outside 0..2 (MAX_BEARERS = 2)", cfg->n_bearers);
  if (nb == 2 && algo == 1)
    return fail(RS_ERR_UNSUPPORTED, "two bearers per UE: id 1 schedules flows, not users -- give it one user per bearer");
  if (cfg->data_to_transmit < 0 || cfg->data_to_transmit > 268435455)
    return fail(RS_ERR_ARG, "data_to_transmit %d outside 0..2^28-1 (data*8 is an int in the reference)", cfg->data_to_transmit);
  for (int p = 0; p < P; ++p)
    for (int u = 0; u < U; ++u)
      if (cfgs[p].ue_to_slice[u] < 0 || cfgs[p].ue_to_slice[u] >= S)
        return fail(RS_ERR_ARG, "%sue_to_slice[%d] out of range", pfx(p).c_str(), u);

  rs_handle* h = new (std::nothrow) rs_handle;
  if (!h) return fail(RS_ERR_ARG, "out of memory");
  h->device = device;
  h->B = n_cells;
  h->P = P;
  if (cfg->tbs_row_m1) memcpy(h->row_m1, cfg->tbs_row_m1, sizeof h->row_m1);
  else default_row_m1(h->row_m1);

  rs::DevCfg& d = h->d;
  d.algo = algo; d.S = S; d.U = U; d.G = G; d.R = cfg->n_rbs; d.rbg = cfg->rbg_size;
  d.grant_len = 2 * G;   /* id 10's reported grant list; rs_set_grant_list_len */
  if (cfg->cqi_per_rb < 0 || cfg->cqi_per_rb > 2) { delete h; return fail(RS_ERR_ARG, "cqi_per_rb must be 0, 1 or 2"); }
  if (cfg->cqi_per_rb == 2 && (G % 8) != 0) { delete h; return fail(RS_ERR_UNSUPPORTED, "4-bit CQI layout needs a multiple of 8 RBGs"); }
  d.cqi_per_rb = cfg->cqi_per_rb;
  d.data = cfg->data_to_transmit;
  d.nb = nb;
  d.n_cells = n_cells;
  d.sort_n = G * S;
  { int lg = 0; for (int m = d.sort_n; m > 1; m >>= 1) lg++; d.sort_depth = 2 * lg; }
  h->cqi_cols = d.cqi_per_rb == 1 ? d.R : (d.cqi_per_rb == 2 ? G / 2 : G);
  d.cqi_row = h->cqi_cols;

#define BAIL(code_)            \
  do {                         \
    int rc_ = (code_);         \
    if (rc_ != RS_OK) {        \
      std::string keep = g_err;\
      rs_destroy(h);           \
      g_err = keep;            \
      return rc_;              \
    }                          \
  } while (0)

  /* ---- tables: one row per profile ([P][S], [P][S][16], [P][U], ...) ---- */
  std::vector<double> epow;
  std::vector<unsigned char> psi((size_t)P * S, 0);
  std::vector<double> weight((size_t)P * S, 0.0);
  int max_tbs = 0;
  std::vector<int> tbsn((size_t)(G + 1) * 16, 0);
  for (int k = 1; k <= G; ++k)
    for (int c = 1; c <= 15; ++c) {
      tbsn[(size_t)k * 16 + c] = tbs_n(mcs_from_cqi(c), k * d.rbg, h->row_m1);
      max_tbs = std::max(max_tbs, tbsn[(size_t)k * 16 + c]);
    }
  if (algo == 1 || algo == 11) {
    epow.assign(16, 0.0);   /* one row for every profile: it depends on no slice parameter */
    for (int c = 1; c <= 15; ++c) { volatile double m = eff_from_cqi(c) * 180000.; epow[c] = m; }  /* dl-pf:137 */
    /* dlps.cpp:264-269: a flow leaves the candidate set once TBS >= data*8; with an infinite buffer never */
    if (algo == 11) {
      for (int p = 0; p < P; ++p)
        for (int s = 0; s < S; ++s) weight[(size_t)p * S + s] = cfgs[p].weight[s];
    } else if ((long long)d.data * 8 <= (long long)max_tbs)
      BAIL(fail(RS_ERR_UNSUPPORTED, "id 1 with data_to_transmit*8 <= %d bits (flow-satisfied cut-off) is not covered", max_tbs));
  } else {
    epow.assign((size_t)P * S * 16, 0.0);
    for (int p = 0; p < P; ++p)
      for (int s = 0; s < S; ++s) {
        const int32_t* pr = cfgs[p].params + 4 * s;
        const size_t ps = (size_t)p * S + s;
        weight[ps] = cfgs[p].weight[s];
        if (pr[3] != 0 && pr[3] != 1)
          BAIL(fail(RS_ERR_UNSUPPORTED, "%sslice %d: psi=%d; pow(avg, psi) is bit-exact on the device only for psi in {0,1}",
                    pfx(p).c_str(), s, pr[3]));
        psi[ps] = (unsigned char)pr[3];
        for (int c = 1; c <= 15; ++c) {
          volatile double e = eff_from_cqi(c);
          volatile double se = e * 180000 / 1000;                       /* transport.cpp:686 */
          double v = pow(se, pr[2]);                                     /* transport.cpp:692 */
          if (pr[0] != 0 && d.data == 0) v = 0.0;                        /* transport.cpp:694-697 */
          epow[ps * 16 + c] = v;
        }
      }
    if (algo == 7) {
      /* nvs.cpp:299-300: allocated RBs < m_requiredRBs = data*8 / TBS1(mcs(wideband CQI)) >= data*8/712 */
      d.nvs_guard = (d.data > 0 && (long long)d.data * 8 / 712 < (long long)d.R) ? 1 : 0;
      if (d.nvs_guard)
        BAIL(fail(RS_ERR_UNSUPPORTED, "id 7 with data_to_transmit=%d: the required-RBs guard can bind; not covered", d.data));
    }
  }
  /* head-of-line delay in the metric: transport.cpp:702-706 (alpha and beta set), nvs.cpp:384-386 (alpha set) */
  std::vector<unsigned char> holmul((size_t)P * S, 0);
  if (algo != 1 && algo != 11)
    for (int p = 0; p < P; ++p)
      for (int s = 0; s < S; ++s) {
        const int32_t* pr = cfgs[p].params + 4 * s;
        unsigned char& hm = holmul[(size_t)p * S + s];
        hm = (pr[0] != 0 && (algo == 7 || pr[1] != 0)) ? 1 : 0;
        /* alpha without beta (transport ids): the delay is not in the metric, but a NEGATIVE hol_delay of rs_set_queues
         * marks a user whose prioritised bearer is empty (two bearers per UE, transport.cpp:696-698): metric 0 */
        if (pr[0] != 0 && algo != 7 && pr[1] == 0) hm = 2;
      }
  std::vector<int> tbs1(16, 1);
  for (int c = 1; c <= 15; ++c) tbs1[c] = tbs_n(mcs_from_cqi(c), 1, h->row_m1);
  tbs1[0] = tbs1[1];
  /* CSR of UEs by slice (ascending UE id inside a slice == the reference's user order), per profile */
  const int SL = (algo == 1) ? 1 : S;
  std::vector<int> ptr((size_t)P * (SL + 1), 0), ues((size_t)P * U), u2s((size_t)P * U);
  int max_slice = 0;
  for (int p = 0; p < P; ++p) {
    int* pp = ptr.data() + (size_t)p * (SL + 1);
    int* pu = ues.data() + (size_t)p * U;
    const int32_t* m = cfgs[p].ue_to_slice;
    std::copy(m, m + U, u2s.begin() + (size_t)p * U);
    for (int u = 0; u < U; ++u) pp[(algo == 1 ? 0 : m[u]) + 1]++;
    for (int s = 0; s < SL; ++s) pp[s + 1] += pp[s];
    std::vector<int> fill(pp, pp + SL);
    for (int u = 0; u < U; ++u) pu[fill[algo == 1 ? 0 : m[u]]++] = u;
    for (int s = 0; s < SL; ++s) max_slice = std::max(max_slice, pp[s + 1] - pp[s]);
  }
  /* metric-table chunks: consecutive slices whose UEs fit the table (one cap, from the largest slice of any profile);
   * a profile with fewer chunks than the most ends in empty ones (S, S), which give the chunk loop no items */
  std::vector<std::vector<int>> pchunks(P);
  int m_cap = 0;
  for (int p = 0; p < P; ++p) {
    const int* pp = ptr.data() + (size_t)p * (SL + 1);
    std::vector<int>& chunks = pchunks[p];
    if (is_transport(algo)) {
      const int cap = rs::metric_table_cap(max_slice, U, S * G);   /* small table: it lives in the sort's slot arrays */
      chunks.push_back(0);
      int cur = 0;
      for (int s = 0; s < S; ++s) {
        const int ns = pp[s + 1] - pp[s];
        if (cur + ns > cap) { chunks.push_back(s); cur = 0; }
        cur += ns;
        m_cap = std::max(m_cap, cur);
      }
      chunks.push_back(S);
    } else if (algo == 7 || algo == 11) {
      m_cap = max_slice;
      chunks = {0, S};
    } else {
      m_cap = (U + 15) / 16;   /* id 1 keeps one running EESM sum per flow there when queues are finite */
      chunks = {0, 1};
    }
  }
  size_t n_chunk_bounds = 0;
  for (const auto& ch : pchunks) n_chunk_bounds = std::max(n_chunk_bounds, ch.size());
  std::vector<int> chunks;
  for (auto& ch : pchunks) {
    ch.resize(n_chunk_bounds, ch.back());
    chunks.insert(chunks.end(), ch.begin(), ch.end());
  }
  d.n_chunks = (int)n_chunk_bounds - 1;
  /* Big slices (a chunk of the metric table would give the CTA fewer (slice, RBG quad) items than it has threads,
   * and there are several chunks): divide the metrics on the fly over all slices at once; the table area only has
   * to hold Epow's S rows.  RS_NO_DIRECT=1 keeps the table (A/B and the equality test). */
  d.direct = 0;
  if (is_transport(algo) && d.n_chunks > 1 && d.cqi_per_rb != 1 && G % 4 == 0 && !getenv("RS_NO_DIRECT")) {
    const int threads = (U >= RS_WIDE_MIN_UES) ? rsw::kThreads : rs::kThreads;
    const int per_chunk = std::max(1, (S + d.n_chunks - 1) / d.n_chunks) * std::max(1, G / 4);
    if ((per_chunk < threads && max_slice >= 8) || getenv("RS_FORCE_DIRECT")) { d.direct = 1; m_cap = std::max(S, 1); }
  }
  d.m_cap = m_cap;
  /* Stage a TTI's CQI in shared memory (cp.async) when the layout is one value per RBG, rows are 16-byte
   * multiples and the staged cell does not cost occupancy the batch could use: eight cells per SM for
   * big batches, fewer when there are not that many cells per SM to begin with. */
  /* hundreds of UEs per cell: the per-UE phases (EWMA, metric table, per-slice argmax, link adaptation)
   * dominate and few cells fit an SM anyway, so give the cell 512 threads */
  h->wide = U >= RS_WIDE_MIN_UES;
  d.ng_ues = (algo == 11 || algo == 7) ? max_slice : 0;   /* id 7: required / held RBs per user of the served slice */
  /* rand() draws a TTI consumes per cell: transport.cpp:490,511 (ids 8/9); nvs.cpp:437-446 draws
   * 300 x users of the served slice (id 11; the stride is sized for the largest slice) */
  d.rand_stride = (algo == 11) ? 300 * max_slice : (is_transport(algo) ? 2 : 0);
  /* id 10 sorts G entries at a time next to the parked grants; ids 101/103 keep their scratch in the slot arrays */
  /* id 10: left slot array = the grants' RBGs [S*G]; right = five warps x 3G sort buffers; 1024 entries also make the
   * range lists (5 x 16 stack entries) and the counters (5 x 32) of those warps fit whatever G is */
  const int min_sort_n = (algo == 10) ? std::max(16 * G, 1024)
                         : ((algo == 101 || algo == 103) ? (rs::inter_scratch_bytes(G, S) + 3) / 4 : 0);   /* posl + posr = 4 n bytes */
  { int lg = 0; for (int m = G; m > 1; m >>= 1) lg++; d.sort_depth_g = 2 * lg; }
  h->layout = h->wide ? reinterpret_cast<const rs::Layout&>(static_cast<const rsw::Layout&>(rsw::make_layout(S, U, G, m_cap, 0, d.ng_ues, min_sort_n, nb, rs::den_shares_cnt(algo))))
                      : rs::make_layout(S, U, G, m_cap, 0, d.ng_ues, min_sort_n, nb, rs::den_shares_cnt(algo));
  h->stage_ok = false;
  if (d.cqi_per_rb != 1 && d.cqi_row % 16 == 0) {
    const rsw::Layout staged_w = rsw::make_layout(S, U, G, m_cap, U * d.cqi_row, d.ng_ues, min_sort_n, nb, rs::den_shares_cnt(algo));
    const rs::Layout staged = h->wide ? reinterpret_cast<const rs::Layout&>(staged_w)
                                      : rs::make_layout(S, U, G, m_cap, U * d.cqi_row, d.ng_ues, min_sort_n, nb, rs::den_shares_cnt(algo));
    const int kSmemPerSm = 227 * 1024, kSms = 148;
    /* Staging pays as long as it does not cost residency: cells an SM can hold = min(register limit of the
     * instantiation, shared memory, what the batch offers).  Measured (profiles/r02_configs3_sweep.jsonl): 20 x 20 UEs
     * 4 staged cells per SM 6.3 M vs 8 unstaged 7.9 M cell-TTIs/s; 50 x 40 UEs 1 staged 0.97 M vs 2 unstaged 1.32 M;
     * same residency either way (20 x 40, 40 x 20, 50 x 10: two 512-thread cells per SM) staged wins by 10-23 %.
     * Narrow cells may give up residency down to RS_STAGE_MIN_FIT cells per SM. */
    const int reg_limit = h->wide ? RS_WIDE_MIN_BLOCKS : 8;
    const int offered = std::max(1, (n_cells + kSms - 1) / kSms);
    const int fit_staged = std::min({reg_limit, kSmemPerSm / (staged.total + 1024), offered});
    const int fit_plain = std::min({reg_limit, kSmemPerSm / (h->layout.total + 1024), offered});
    int min_fit = h->wide ? fit_plain : std::min(fit_plain, RS_STAGE_MIN_FIT);
    if (const char* e = getenv("RS_STAGE_MIN_FIT")) min_fit = std::min(fit_plain, std::max(1, atoi(e)));
    if (fit_staged >= 1 && fit_staged >= min_fit && !getenv("RS_NO_STAGE")) { h->layout = staged; h->stage_ok = true; }
  }
  d.lay = h->layout;

  /* ---- device ---- */
  {
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) BAIL(fail(RS_ERR_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e)));
    int max_optin = 0;
    e = cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e != cudaSuccess) BAIL(fail(RS_ERR_CUDA, "cudaDeviceGetAttribute: %s", cudaGetErrorString(e)));
    if (h->layout.total > max_optin)
      BAIL(fail(RS_ERR_UNSUPPORTED, "cell needs %d B of shared memory, device allows %d", h->layout.total, max_optin));
  }
  if (has_fixed_kernel(algo) && !getenv("RS_NO_FIXED_SHAPE")) {
    if (shape_matches<FixedU8>(h, u2s)) h->fixed = 0;
    else if (shape_matches<FixedNib>(h, u2s)) h->fixed = 1;
  }
  rs::ConstTables ct;
  { std::string why;
    if (!build_const_tables(&ct, &why)) BAIL(fail(RS_ERR_UNSUPPORTED, "host libm: %s", why.c_str())); }
  { cudaError_t e = rs_tables_tu1(&ct);   /* every unit that holds kernels has its own copy of the constant tables */
    if (e == cudaSuccess) e = rs_tables_tu2(&ct);
    if (e == cudaSuccess) e = rs_tables_tu3(&ct);
    if (e == cudaSuccess) e = rs_tables_tu4(&ct);
    if (e == cudaSuccess) e = rs_tables_tu5(&ct);
    if (e == cudaSuccess) e = rs_tables_tu6(&ct);
    if (e != cudaSuccess) BAIL(fail(RS_ERR_CUDA, "cudaMemcpyToSymbol: %s", cudaGetErrorString(e))); }
  BAIL(set_smem_attr(h));
  { cudaError_t e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->copy_in, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->copy_out, cudaStreamNonBlocking);
    for (auto& st : h->xs) if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
    for (auto& ev : h->join_evs) if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->fork_ev, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->join_ev, cudaEventDisableTiming);
    if (e != cudaSuccess) BAIL(fail(RS_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e))); }
  h->stream = h->own_stream;
  /* two half-batches once each half still fills the GPU (RS_NO_SPLIT=1: one launch per step of TTIs, as in round 1) */
  /* two part-batches once each still fills the GPU's resident cells; RS_PARTS = 1..4 for experiments */
  { const int resident = std::max(1, std::min(h->wide ? RS_WIDE_MIN_BLOCKS : 8, (227 * 1024) / (h->layout.total + 1024)));
    h->parts = n_cells >= 2 * 148 * resident ? 2 : 1;   /* measured: 1 part 17.9 M, 2 parts 20.3 M, 3 and 4 parts 20.3 M */
    if (const char* e = getenv("RS_PARTS")) h->parts = std::max(1, std::min({rs_handle::kMaxParts, atoi(e), n_cells}));   /* experiments */
    if (getenv("RS_NO_SPLIT")) h->parts = 1; }
  BAIL(upload(h->ue_to_slice, u2s));
  BAIL(upload(h->slice_ptr, ptr));
  BAIL(upload(h->slice_ues, ues));
  BAIL(upload(h->chunk_slice, chunks));
  BAIL(upload(h->tbs_n, tbsn));
  BAIL(upload(h->weight, weight));
  BAIL(upload(h->epow, epow));
  BAIL(upload(h->psi, psi));
  BAIL(upload(h->holmul, holmul));
  BAIL(upload(h->tbs1, tbs1));
  if (P > 1) {   /* one profile: cell_profile stays null and every cell reads row 0 */
    BAIL(upload(h->cell_profile, std::vector<int>(cell_profile, cell_profile + n_cells)));
    d.cell_profile = h->cell_profile.p;
  }
  d.holmul = h->holmul.p;
  d.tbs1 = h->tbs1.p;
  if (algo == 103) {
    std::vector<short> vt;
    build_vogel_tab(&vt);
    BAIL(upload(h->vogel_tab, vt));
    d.vogel_tab = h->vogel_tab.p;
  }
  if ((algo == 9 && d.sort_n > 16) || (algo == 10 && G > 16)) {
    std::vector<unsigned short> eq;
    d.eq_max = std::min(algo == 10 ? G : d.sort_n, kEqMax);
    build_eq_table(d.eq_max, &eq);
    BAIL(upload(h->eq_tab, eq));
    d.eq_tab = h->eq_tab.p;
  }
  d.ue_to_slice = h->ue_to_slice.p; d.slice_ptr = h->slice_ptr.p; d.slice_ues = h->slice_ues.p;
  d.chunk_slice = h->chunk_slice.p; d.tbs_n = h->tbs_n.p; d.weight = h->weight.p; d.epow = h->epow.p;
  d.psi = h->psi.p;
  const size_t BU = (size_t)n_cells * U * nb, BS = (size_t)n_cells * S;   /* per-bearer state */
  { cudaError_t e = h->avg.alloc(BU);
    if (e == cudaSuccess) e = h->tx.alloc(BU);
    if (e == cudaSuccess) e = h->cum_bytes.alloc(BU);
    if (e == cudaSuccess) e = h->cum_rbs.alloc(BU);
    if (e == cudaSuccess) e = h->offset.alloc(BS);
    if (e == cudaSuccess) e = h->ewma.alloc(BS);
    if (e == cudaSuccess) e = h->stats.alloc((size_t)4 * S * P);
    if (e != cudaSuccess) BAIL(fail(RS_ERR_CUDA, "cudaMalloc(state): %s", cudaGetErrorString(e))); }
  d.avg = h->avg.p; d.tx = h->tx.p; d.cum_bytes = h->cum_bytes.p; d.cum_rbs = h->cum_rbs.p;
  d.offset = h->offset.p; d.ewma = h->ewma.p;
  BAIL(rs_reset_state(h));
#undef BAIL
  *out = h;
  return RS_OK;
}

int rs_set_stream(rs_handle* h, void* cuda_stream) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
  return RS_OK;
}

int rs_sync(rs_handle* h) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->copy_in));
  CU(cudaStreamSynchronize(h->stream));
  for (auto st : h->xs) CU(cudaStreamSynchronize(st));
  CU(cudaStreamSynchronize(h->copy_out));
  return RS_OK;
}

void* rs_get_stream(rs_handle* h) { return h ? (void*)h->stream : nullptr; }

int rs_host_alloc(size_t bytes, int32_t write_combined, void** out) {
  if (!out || bytes == 0) return fail(RS_ERR_ARG, "rs_host_alloc: bad argument");
  *out = nullptr;
  CU(cudaHostAlloc(out, bytes, cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0)));
  return RS_OK;
}
void rs_host_free(void* p) { if (p) cudaFreeHost(p); }

int rs_reset_state(rs_handle* h) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  const size_t BU = (size_t)h->B * h->d.U * h->d.nb, BS = (size_t)h->B * h->d.S;
  std::vector<double> avg(BU, 100000.0);   /* m_averageTransmissionRate, radio-bearer.cpp:54 */
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaMemcpy(h->avg.p, avg.data(), BU * 8, cudaMemcpyHostToDevice));
  CU(cudaMemset(h->tx.p, 0, BU * 4));
  CU(cudaMemset(h->cum_bytes.p, 0, BU * 8));
  CU(cudaMemset(h->cum_rbs.p, 0, BU * 8));
  CU(cudaMemset(h->offset.p, 0, BS * 8));
  CU(cudaMemset(h->ewma.p, 0, BS * 8));
  return buf_empty(h);
}

int rs_set_state(rs_handle* h, const double* avg_rate, const int32_t* tx_bytes, const uint64_t* cum_bytes,
                 const uint64_t* cum_rbs, const double* slice_offset, const double* nvs_ewma) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  const size_t BU = (size_t)h->B * h->d.U * h->d.nb, BS = (size_t)h->B * h->d.S;
  if (avg_rate) CU(cudaMemcpy(h->avg.p, avg_rate, BU * 8, cudaMemcpyHostToDevice));
  if (tx_bytes) CU(cudaMemcpy(h->tx.p, tx_bytes, BU * 4, cudaMemcpyHostToDevice));
  if (cum_bytes) CU(cudaMemcpy(h->cum_bytes.p, cum_bytes, BU * 8, cudaMemcpyHostToDevice));
  if (cum_rbs) CU(cudaMemcpy(h->cum_rbs.p, cum_rbs, BU * 8, cudaMemcpyHostToDevice));
  if (slice_offset) CU(cudaMemcpy(h->offset.p, slice_offset, BS * 8, cudaMemcpyHostToDevice));
  if (nvs_ewma) CU(cudaMemcpy(h->ewma.p, nvs_ewma, BS * 8, cudaMemcpyHostToDevice));
  return RS_OK;
}

int rs_set_cell_profiles(rs_handle* h, const int32_t* cell_profile) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  if (!cell_profile && h->P > 1) return fail(RS_ERR_ARG, "rs_set_cell_profiles: cell_profile is NULL with %d profiles", h->P);
  if (cell_profile)
    for (int b = 0; b < h->B; ++b)
      if (cell_profile[b] < 0 || cell_profile[b] >= h->P)
        return fail(RS_ERR_ARG, "rs_set_cell_profiles: cell_profile[%d] = %d outside 0..%d", b, cell_profile[b], h->P - 1);
  if (h->P == 1) return RS_OK;   /* every cell is in profile 0 already */
  const int rc = rs_sync(h);     /* the launches in flight (rs_run_*_async included) read the old assignment */
  if (rc != RS_OK) return rc;
  CU(cudaMemcpy(h->cell_profile.p, cell_profile, sizeof(int32_t) * h->B, cudaMemcpyHostToDevice));
  return RS_OK;
}

int rs_set_grant_list_len(rs_handle* h, int32_t n) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  if (h->d.algo != 10) return fail(RS_ERR_ARG, "rs_set_grant_list_len: the grant list is id 10's output");
  const int G = h->d.G, S = h->d.S;
  if (n < 2 * G || n > std::max(S * G, 2 * G))
    return fail(RS_ERR_ARG, "rs_set_grant_list_len: %d outside 2G..max(S*G, 2G) = %d..%d", n, 2 * G, std::max(S * G, 2 * G));
  const int rc = rs_sync(h);     /* the launches in flight (rs_run_*_async included) write lists of the old length */
  if (rc != RS_OK) return rc;
  h->d.grant_len = n;
  return RS_OK;
}
int32_t rs_grant_list_len(const rs_handle* h) { return (h && h->d.algo == 10) ? h->d.grant_len : 0; }

int rs_get_state(rs_handle* h, double* avg_rate, int32_t* tx_bytes, uint64_t* cum_bytes, uint64_t* cum_rbs,
                 double* slice_offset, double* nvs_ewma) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  const size_t BU = (size_t)h->B * h->d.U * h->d.nb, BS = (size_t)h->B * h->d.S;
  if (avg_rate) CU(cudaMemcpy(avg_rate, h->avg.p, BU * 8, cudaMemcpyDeviceToHost));
  if (tx_bytes) CU(cudaMemcpy(tx_bytes, h->tx.p, BU * 4, cudaMemcpyDeviceToHost));
  if (cum_bytes) CU(cudaMemcpy(cum_bytes, h->cum_bytes.p, BU * 8, cudaMemcpyDeviceToHost));
  if (cum_rbs) CU(cudaMemcpy(cum_rbs, h->cum_rbs.p, BU * 8, cudaMemcpyDeviceToHost));
  if (slice_offset) CU(cudaMemcpy(slice_offset, h->offset.p, BS * 8, cudaMemcpyDeviceToHost));
  if (nvs_ewma) CU(cudaMemcpy(nvs_ewma, h->ewma.p, BS * 8, cudaMemcpyDeviceToHost));
  return RS_OK;
}

}  /* extern "C" */

namespace {
/* Every stream of the handle idle.  Error exits of the pipelined calls go through here so that no copy is still
 * reading or writing the caller's buffers when a "failed" call returns. */
void drain(rs_handle* h) {
  cudaStreamSynchronize(h->copy_in);
  cudaStreamSynchronize(h->stream);
  for (auto st : h->xs) cudaStreamSynchronize(st);
  cudaStreamSynchronize(h->copy_out);
}
#define CU_DRAIN(call)                                                                             \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      drain(h);                                                                                    \
      return fail(RS_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_));                           \
    }                                                                                              \
  } while (0)

void point_outputs(const rs_handle* h, rs::RunArgs* a, const rs_outputs* o, size_t t0) {
  if (!o) return;
  const size_t B = h->B, U = h->d.U, S = h->d.S, G = h->d.G;
  a->rbg_to_ue = o->rbg_to_ue ? o->rbg_to_ue + t0 * B * G : nullptr;
  a->tbs_bits = o->tbs_bits ? o->tbs_bits + t0 * B * U : nullptr;
  a->mcs = o->mcs ? o->mcs + t0 * B * U : nullptr;
  a->final_cqi = o->final_cqi ? o->final_cqi + t0 * B * U : nullptr;
  if (wants(h, 0)) {
    a->slice_target = o->slice_target ? o->slice_target + t0 * B * S : nullptr;
    a->slice_quota = o->slice_quota ? o->slice_quota + t0 * B * S : nullptr;
  }
  if (wants(h, 1)) a->nvs_slice = o->nvs_slice ? o->nvs_slice + t0 * B : nullptr;
  if (h->d.algo == 10) {
    a->alloc_n = o->alloc_n ? o->alloc_n + t0 * B : nullptr;
    a->alloc_ue = o->alloc_ue ? o->alloc_ue + t0 * B * h->d.grant_len : nullptr;
    a->alloc_rbg = o->alloc_rbg ? o->alloc_rbg + t0 * B * h->d.grant_len : nullptr;
  }
}

/* trace_row == NULL: CQI slabs in device memory; else trace-driven (d_cqi unused) */
int run_device_impl(rs_handle* h, int32_t n_ttis, const uint8_t* d_cqi, int64_t cqi_tti_stride, int32_t cqi_refresh,
                    const int32_t* trace_row, const int32_t* d_rand2, const uint8_t* d_active,
                    int64_t active_tti_stride, const double* dt, const rs_outputs* d_out, int32_t ttis_per_launch) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  /* rs_set_queues: consumed by this call whether it succeeds or not */
  const int32_t* d_queue = h->q_next;
  const double* d_hol = h->hol_next;
  h->q_next = nullptr;
  h->hol_next = nullptr;
  rs_traffic tr;
  if (const int rc = take_traffic(h, n_ttis, &tr); rc != RS_OK) return rc;
  const bool buffered = h->buf_k > 0;
  if ((!d_cqi && !trace_row) || !dt || n_ttis < 0 || cqi_refresh < 1) return fail(RS_ERR_ARG, "rs_run_device: bad argument");
  if (h->d.rand_stride > 0 && !d_rand2) return fail(RS_ERR_ARG, "ids 8/9/11 need the rand() draws");
  if (!trace_row && (((uintptr_t)d_cqi & 3) || (cqi_tti_stride & 3))) return fail(RS_ERR_ARG, "cqi must be 4-byte aligned");
  if (trace_row && !h->trace_tab.p) return fail(RS_ERR_ARG, "no traces loaded: call rs_set_traces first");
  if (h->d.nb == 2 && !d_queue && !buffered) return fail(RS_ERR_ARG, "two bearers per UE: every run call needs rs_set_queues");
  if (n_ttis == 0) return RS_OK;
  CU(cudaSetDevice(h->device));
  if (trace_row) { const int rc = check_trace_rows(h, trace_row, n_ttis); if (rc != RS_OK) return rc; }
  if (ttis_per_launch <= 0) ttis_per_launch = 16;
  ttis_per_launch = std::min<int>(ttis_per_launch, rs::kMaxTtisPerLaunch);
  const size_t B = h->B, U = h->d.U;
  /* buffered: the kernels write the queue / HoL each TTI shows into queue_out / hol_out, or into one launch's worth of
   * scratch that every launch of the call reuses (launches of one part run in order; parts own disjoint cells) */
  size_t q_tti = B * U * h->d.nb, h_tti = q_tti;
  if (buffered) {
    const size_t per_launch = (size_t)std::min(ttis_per_launch, n_ttis) * B * U * h->d.nb;
    if (tr.queue_out) d_queue = tr.queue_out; else { CU(h->shown_q.alloc(per_launch)); d_queue = h->shown_q.p; q_tti = 0; }
    if (tr.hol_out) d_hol = tr.hol_out; else { CU(h->shown_hol.alloc(per_launch)); d_hol = h->shown_hol.p; h_tti = 0; }
  }
  /* more than one launch in this call and a big batch: the two halves of the batch go down two streams (forked
   * here, joined at the end of the call), so the tail of one launch overlaps the head of the next */
  const bool split = h->parts > 1 && n_ttis > ttis_per_launch;
  const int P = split ? h->parts : 1;
  if (split) {
    CU(cudaEventRecord(h->fork_ev, h->stream));
    for (int q = 1; q < P; ++q) CU(cudaStreamWaitEvent(h->xs[q - 1], h->fork_ev, 0));
  }
  for (int t0 = 0; t0 < n_ttis; t0 += ttis_per_launch) {
    rs::RunArgs a{};
    a.T = std::min(ttis_per_launch, n_ttis - t0);
    a.cqi = d_cqi;
    a.cqi_tti_stride = cqi_tti_stride;
    a.t0 = t0;
    a.cqi_refresh = cqi_refresh;
    a.rand2 = (d_rand2 && h->d.rand_stride) ? d_rand2 + (size_t)t0 * B * h->d.rand_stride : nullptr;
    a.active = d_active ? d_active + (size_t)t0 * active_tti_stride : nullptr;
    a.active_tti_stride = active_tti_stride;
    fill_scalars(h, &a, dt + t0, trace_row ? trace_row + t0 : nullptr, a.T);
    a.queue = d_queue ? d_queue + (size_t)t0 * q_tti : nullptr;
    a.hol = d_hol ? d_hol + (size_t)t0 * h_tti : nullptr;
    if (buffered) {
      a.arrivals = tr.arrivals + (size_t)t0 * B * U * h->d.nb;
      fill_buffers(h, &a, tr, t0, a.T);
    }
    a.stage = h->stage_ok && (trace_row || ((((uintptr_t)d_cqi) & 15) == 0 && (cqi_tti_stride & 15) == 0)) ? 1 : 0;
    point_outputs(h, &a, d_out, (size_t)t0);
    int rc = launch_ttis(h, a, trace_row != nullptr, nullptr, split ? 0 : -1);
    for (int q = 1; q < P && rc == RS_OK; ++q) rc = launch_ttis(h, a, trace_row != nullptr, nullptr, q);
    if (rc != RS_OK) { for (auto st : h->xs) cudaStreamSynchronize(st); return rc; }
  }
  for (int q = 1; q < P; ++q) {
    CU(cudaEventRecord(h->join_evs[q - 1], h->xs[q - 1]));
    CU(cudaStreamWaitEvent(h->stream, h->join_evs[q - 1], 0));
  }
  if (buffered) h->last_now = tr.now[n_ttis - 1];
  return RS_OK;
}

/* trace_row == NULL: CQI slabs from the host; else trace-driven (cqi unused, nothing but rand2/active goes up).
 * Enqueues the whole call on the handle's three streams and returns a ticket; `wait` blocks until the call's
 * results are in the caller's buffers.  The slot ring is NOT drained at the end of a call: the first chunks of
 * the next call overlap the last kernels and copies of this one. */
int run_host_impl(rs_handle* h, int32_t n_ttis, const uint8_t* cqi, int32_t cqi_refresh, const int32_t* trace_row,
                  const int32_t* rand2, const uint8_t* active, const double* dt, const rs_outputs* out,
                  int32_t ttis_per_launch, bool wait, int64_t* ticket) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  /* rs_set_queues: consumed by this call whether it succeeds or not */
  const int32_t* queue = h->q_next;
  const double* hol = h->hol_next;
  h->q_next = nullptr;
  h->hol_next = nullptr;
  if (ticket) *ticket = -1;
  rs_traffic tr;
  if (const int rc = take_traffic(h, n_ttis, &tr); rc != RS_OK) return rc;
  const bool buffered = h->buf_k > 0;   /* the slot's queue / hol arrays are written by the kernel, not copied in */
  if ((!cqi && !trace_row) || !dt || n_ttis < 0 || cqi_refresh < 1) return fail(RS_ERR_ARG, "rs_run_host: bad argument");
  if (h->d.rand_stride > 0 && !rand2) return fail(RS_ERR_ARG, "ids 8/9/11 need the rand() draws");
  if (trace_row && !h->trace_tab.p) return fail(RS_ERR_ARG, "no traces loaded: call rs_set_traces first");
  if (h->d.nb == 2 && !queue && !buffered) return fail(RS_ERR_ARG, "two bearers per UE: every run call needs rs_set_queues");
  CU(cudaSetDevice(h->device));
  if (trace_row) { const int rc = check_trace_rows(h, trace_row, n_ttis); if (rc != RS_OK) return rc; }
  if (ttis_per_launch <= 0) ttis_per_launch = trace_row ? 16 : 8;
  const size_t NB = (size_t)h->d.nb;
  const int TC = std::max(1, std::min(std::min<int>(ttis_per_launch, rs::kMaxTtisPerLaunch), n_ttis));
  const size_t B = h->B, U = h->d.U, S = h->d.S, G = h->d.G, C = h->cqi_cols, NL = h->d.grant_len;
  const bool slabs = !trace_row && cqi_refresh > 1;   /* consecutive chunks share a CQI slab */
  const bool split = h->parts > 1;
  const int P = h->parts;
  if (split) {   /* the extra streams join whatever the caller's stream has seen so far (state uploads, earlier device calls) */
    CU(cudaEventRecord(h->fork_ev, h->stream));
    for (int q = 1; q < P; ++q) CU(cudaStreamWaitEvent(h->xs[q - 1], h->fork_ev, 0));
  }
  for (auto& s : h->slot) {
    const int rc = alloc_slot(h, s, TC, out, active != nullptr, !trace_row && !slabs, queue != nullptr || buffered,
                              hol != nullptr || buffered, buffered);
    if (rc != RS_OK) { drain(h); return rc; }
  }
  if (slabs)
    for (auto& sl : h->slab) {
      CU_DRAIN(sl.cqi.alloc(B * U * C));
      if (!sl.used) CU_DRAIN(cudaEventCreateWithFlags(&sl.used, cudaEventDisableTiming));
      for (auto& e : sl.used_x) if (!e) CU_DRAIN(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      sl.index = -1;   /* slab numbers are relative to this call's cqi pointer */
    }
  for (auto& e : h->call_done)
    if (!e) CU_DRAIN(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  int next_slab_buf = 0;
  for (int t0 = 0, T = 0; t0 < n_ttis; t0 += T) {
    rs_handle::Slot& s = h->slot[h->chunk_seq % rs_handle::kSlots];
    T = std::min(TC, n_ttis - t0);
    /* with a refresh > 1 a chunk ends at the next refresh boundary: it reads exactly one slab */
    if (slabs) T = std::min(T, (t0 / cqi_refresh + 1) * cqi_refresh - t0);
    const int slab0 = t0 / cqi_refresh;
    /* inputs: the slot's previous kernel must be done with them */
    if (s.k_rec) {
      CU_DRAIN(cudaStreamWaitEvent(h->copy_in, s.k_done, 0));
      for (int q = 1; q < P; ++q) CU_DRAIN(cudaStreamWaitEvent(h->copy_in, s.k_done_x[q - 1], 0));
    }
    const uint8_t* d_cqi = nullptr;
    rs_handle::Slab* sl = nullptr;
    if (slabs) {
      for (auto& c : h->slab) if (c.index == slab0) sl = &c;
      if (!sl) {
        sl = &h->slab[next_slab_buf];
        next_slab_buf ^= 1;
        if (sl->used_rec) {
          CU_DRAIN(cudaStreamWaitEvent(h->copy_in, sl->used, 0));
          for (int q = 1; q < P; ++q) CU_DRAIN(cudaStreamWaitEvent(h->copy_in, sl->used_x[q - 1], 0));
        }
        CU_DRAIN(cudaMemcpyAsync(sl->cqi.p, cqi + (size_t)slab0 * B * U * C, B * U * C, cudaMemcpyHostToDevice, h->copy_in));
        sl->index = slab0;
      }
      d_cqi = sl->cqi.p;
    } else if (!trace_row) {
      CU_DRAIN(cudaMemcpyAsync(s.cqi.p, cqi + (size_t)t0 * B * U * C, (size_t)T * B * U * C, cudaMemcpyHostToDevice, h->copy_in));
      d_cqi = s.cqi.p;
    }
    const size_t RS = (size_t)h->d.rand_stride;
    if (rand2 && RS) CU_DRAIN(cudaMemcpyAsync(s.rand2.p, rand2 + (size_t)t0 * B * RS, (size_t)T * B * RS * 4, cudaMemcpyHostToDevice, h->copy_in));
    if (active) CU_DRAIN(cudaMemcpyAsync(s.active.p, active + (size_t)t0 * B * U, (size_t)T * B * U, cudaMemcpyHostToDevice, h->copy_in));
    if (queue) CU_DRAIN(cudaMemcpyAsync(s.queue.p, queue + (size_t)t0 * B * U * NB, (size_t)T * B * U * NB * 4, cudaMemcpyHostToDevice, h->copy_in));
    if (hol) CU_DRAIN(cudaMemcpyAsync(s.hol.p, hol + (size_t)t0 * B * U * NB, (size_t)T * B * U * NB * 8, cudaMemcpyHostToDevice, h->copy_in));
    if (buffered) CU_DRAIN(cudaMemcpyAsync(s.arrivals.p, tr.arrivals + (size_t)t0 * B * U * NB, (size_t)T * B * U * NB * 4, cudaMemcpyHostToDevice, h->copy_in));
    CU_DRAIN(cudaEventRecord(s.in_done, h->copy_in));
    /* kernel(s): inputs in, and the slot's previous outputs drained; a big batch runs as two half-batches, each half
     * chained on its own stream from chunk to chunk (the copies wait for both) */
    CU_DRAIN(cudaStreamWaitEvent(h->stream, s.in_done, 0));
    if (s.out_rec) CU_DRAIN(cudaStreamWaitEvent(h->stream, s.out_done, 0));
    for (int q = 1; q < P; ++q) {
      CU_DRAIN(cudaStreamWaitEvent(h->xs[q - 1], s.in_done, 0));
      if (s.out_rec) CU_DRAIN(cudaStreamWaitEvent(h->xs[q - 1], s.out_done, 0));
    }
    rs::RunArgs a{};
    a.T = T;
    a.cqi = d_cqi; a.cqi_tti_stride = (long long)(B * U * C);
    a.t0 = 0; a.cqi_refresh = slabs ? cqi_refresh : 1;   /* one resident slab, or one slab per TTI of the chunk */
    a.rand2 = (rand2 && RS) ? s.rand2.p : nullptr;
    a.active = active ? s.active.p : nullptr; a.active_tti_stride = (long long)(B * U);
    fill_scalars(h, &a, dt + t0, trace_row ? trace_row + t0 : nullptr, T);
    a.queue = (queue || buffered) ? s.queue.p : nullptr;
    a.hol = (hol || buffered) ? s.hol.p : nullptr;
    if (buffered) {
      a.arrivals = s.arrivals.p;
      fill_buffers(h, &a, tr, t0, T);
    }
    a.stage = h->stage_ok ? 1 : 0;   /* slot buffers come from cudaMalloc; B*U*C is a multiple of 16 when stage_ok */
    rs_outputs so{};
    if (out) {
      so.rbg_to_ue = out->rbg_to_ue ? s.rbg_to_ue.p : nullptr;
      so.tbs_bits = out->tbs_bits ? s.tbs_bits.p : nullptr;
      so.mcs = out->mcs ? s.mcs.p : nullptr;
      so.final_cqi = out->final_cqi ? s.final_cqi.p : nullptr;
      so.slice_target = out->slice_target ? s.slice_target.p : nullptr;
      so.slice_quota = out->slice_quota ? s.slice_quota.p : nullptr;
      so.nvs_slice = out->nvs_slice ? s.nvs_slice.p : nullptr;
      so.alloc_n = out->alloc_n ? s.alloc_n.p : nullptr;
      so.alloc_ue = out->alloc_ue ? s.alloc_ue.p : nullptr;
      so.alloc_rbg = out->alloc_rbg ? s.alloc_rbg.p : nullptr;
      point_outputs(h, &a, &so, 0);
    }
    int rc = launch_ttis(h, a, trace_row != nullptr, nullptr, split ? 0 : -1);
    for (int q = 1; q < P && rc == RS_OK; ++q) rc = launch_ttis(h, a, trace_row != nullptr, nullptr, q);
    if (rc != RS_OK) { drain(h); return rc; }
    CU_DRAIN(cudaEventRecord(s.k_done, h->stream));
    for (int q = 1; q < P; ++q) CU_DRAIN(cudaEventRecord(s.k_done_x[q - 1], h->xs[q - 1]));
    s.k_rec = true;
    if (sl) {
      CU_DRAIN(cudaEventRecord(sl->used, h->stream));
      for (int q = 1; q < P; ++q) CU_DRAIN(cudaEventRecord(sl->used_x[q - 1], h->xs[q - 1]));
      sl->used_rec = true;
    }
    /* outputs */
    CU_DRAIN(cudaStreamWaitEvent(h->copy_out, s.k_done, 0));
    for (int q = 1; q < P; ++q) CU_DRAIN(cudaStreamWaitEvent(h->copy_out, s.k_done_x[q - 1], 0));
    if (out) {
      if (a.rbg_to_ue) CU_DRAIN(cudaMemcpyAsync(out->rbg_to_ue + (size_t)t0 * B * G, s.rbg_to_ue.p, (size_t)T * B * G * 2, cudaMemcpyDeviceToHost, h->copy_out));
      if (a.tbs_bits) CU_DRAIN(cudaMemcpyAsync(out->tbs_bits + (size_t)t0 * B * U, s.tbs_bits.p, (size_t)T * B * U * 4, cudaMemcpyDeviceToHost, h->copy_out));
      if (a.mcs) CU_DRAIN(cudaMemcpyAsync(out->mcs + (size_t)t0 * B * U, s.mcs.p, (size_t)T * B * U, cudaMemcpyDeviceToHost, h->copy_out));
      if (a.final_cqi) CU_DRAIN(cudaMemcpyAsync(out->final_cqi + (size_t)t0 * B * U, s.final_cqi.p, (size_t)T * B * U, cudaMemcpyDeviceToHost, h->copy_out));
      if (a.slice_target) CU_DRAIN(cudaMemcpyAsync(out->slice_target + (size_t)t0 * B * S, s.slice_target.p, (size_t)T * B * S * 4, cudaMemcpyDeviceToHost, h->copy_out));
      if (a.slice_quota) CU_DRAIN(cudaMemcpyAsync(out->slice_quota + (size_t)t0 * B * S, s.slice_quota.p, (size_t)T * B * S * 4, cudaMemcpyDeviceToHost, h->copy_out));
      if (a.nvs_slice) CU_DRAIN(cudaMemcpyAsync(out->nvs_slice + (size_t)t0 * B, s.nvs_slice.p, (size_t)T * B * 4, cudaMemcpyDeviceToHost, h->copy_out));
      if (a.alloc_n) CU_DRAIN(cudaMemcpyAsync(out->alloc_n + (size_t)t0 * B, s.alloc_n.p, (size_t)T * B * 4, cudaMemcpyDeviceToHost, h->copy_out));
      if (a.alloc_ue) CU_DRAIN(cudaMemcpyAsync(out->alloc_ue + (size_t)t0 * B * NL, s.alloc_ue.p, (size_t)T * B * NL * 2, cudaMemcpyDeviceToHost, h->copy_out));
      if (a.alloc_rbg) CU_DRAIN(cudaMemcpyAsync(out->alloc_rbg + (size_t)t0 * B * NL, s.alloc_rbg.p, (size_t)T * B * NL * 2, cudaMemcpyDeviceToHost, h->copy_out));
    }
    if (tr.queue_out) CU_DRAIN(cudaMemcpyAsync(tr.queue_out + (size_t)t0 * B * U * NB, s.queue.p, (size_t)T * B * U * NB * 4, cudaMemcpyDeviceToHost, h->copy_out));
    if (tr.hol_out) CU_DRAIN(cudaMemcpyAsync(tr.hol_out + (size_t)t0 * B * U * NB, s.hol.p, (size_t)T * B * U * NB * 8, cudaMemcpyDeviceToHost, h->copy_out));
    CU_DRAIN(cudaEventRecord(s.out_done, h->copy_out));
    s.out_rec = true;
    h->chunk_seq++;
  }
  for (int q = 1; q < P; ++q) {   /* the handle's stream is behind every part's kernels again (rs_get_state, the next device call) */
    CU_DRAIN(cudaEventRecord(h->join_evs[q - 1], h->xs[q - 1]));
    CU_DRAIN(cudaStreamWaitEvent(h->stream, h->join_evs[q - 1], 0));
  }
  if (buffered && n_ttis > 0) h->last_now = tr.now[n_ttis - 1];
  /* copy_out is behind every kernel of the call (it waited on each k_done), and every kernel is behind its inputs */
  const int64_t tk = h->calls++;
  CU_DRAIN(cudaEventRecord(h->call_done[tk % rs_handle::kTickets], h->copy_out));
  if (ticket) *ticket = tk;
  if (wait) CU_DRAIN(cudaEventSynchronize(h->call_done[tk % rs_handle::kTickets]));
  return RS_OK;
}
}  // namespace

extern "C" {

int rs_run_device(rs_handle* h, int32_t n_ttis, const uint8_t* d_cqi, int64_t cqi_tti_stride, int32_t cqi_refresh,
                  const int32_t* d_rand2, const uint8_t* d_active, int64_t active_tti_stride,
                  const double* dt, const rs_outputs* d_out, int32_t ttis_per_launch) {
  if (!d_cqi) return fail(RS_ERR_ARG, "rs_run_device: bad argument");
  return run_device_impl(h, n_ttis, d_cqi, cqi_tti_stride, cqi_refresh, nullptr, d_rand2, d_active, active_tti_stride,
                         dt, d_out, ttis_per_launch);
}

int rs_run_host(rs_handle* h, int32_t n_ttis, const uint8_t* cqi, int32_t cqi_refresh, const int32_t* rand2,
                const uint8_t* active, const double* dt, const rs_outputs* out, int32_t ttis_per_launch) {
  if (!cqi) return fail(RS_ERR_ARG, "rs_run_host: bad argument");
  return run_host_impl(h, n_ttis, cqi, cqi_refresh, nullptr, rand2, active, dt, out, ttis_per_launch, true, nullptr);
}

int rs_run_host_async(rs_handle* h, int32_t n_ttis, const uint8_t* cqi, int32_t cqi_refresh, const int32_t* rand2,
                      const uint8_t* active, const double* dt, const rs_outputs* out, int32_t ttis_per_launch,
                      int64_t* ticket) {
  if (!cqi || !ticket) return fail(RS_ERR_ARG, "rs_run_host_async: bad argument");
  return run_host_impl(h, n_ttis, cqi, cqi_refresh, nullptr, rand2, active, dt, out, ttis_per_launch, false, ticket);
}

int rs_run_traces_device(rs_handle* h, int32_t n_ttis, const int32_t* trace_row, const int32_t* d_rand2,
                         const uint8_t* d_active, int64_t active_tti_stride, const double* dt,
                         const rs_outputs* d_out, int32_t ttis_per_launch) {
  if (!trace_row) return fail(RS_ERR_ARG, "rs_run_traces_device: bad argument");
  return run_device_impl(h, n_ttis, nullptr, 0, 1, trace_row, d_rand2, d_active, active_tti_stride, dt, d_out,
                         ttis_per_launch);
}

int rs_run_traces_host(rs_handle* h, int32_t n_ttis, const int32_t* trace_row, const int32_t* rand2,
                       const uint8_t* active, const double* dt, const rs_outputs* out, int32_t ttis_per_launch) {
  if (!trace_row) return fail(RS_ERR_ARG, "rs_run_traces_host: bad argument");
  return run_host_impl(h, n_ttis, nullptr, 1, trace_row, rand2, active, dt, out, ttis_per_launch, true, nullptr);
}

int rs_run_traces_host_async(rs_handle* h, int32_t n_ttis, const int32_t* trace_row, const int32_t* rand2,
                             const uint8_t* active, const double* dt, const rs_outputs* out, int32_t ttis_per_launch,
                             int64_t* ticket) {
  if (!trace_row || !ticket) return fail(RS_ERR_ARG, "rs_run_traces_host_async: bad argument");
  return run_host_impl(h, n_ttis, nullptr, 1, trace_row, rand2, active, dt, out, ttis_per_launch, false, ticket);
}

int rs_wait(rs_handle* h, int64_t ticket) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  if (ticket < 0 || ticket >= h->calls) return fail(RS_ERR_ARG, "rs_wait: ticket %lld was never issued", (long long)ticket);
  CU(cudaSetDevice(h->device));
  /* an event that has been re-used by a later call completes after the earlier call did */
  CU(cudaEventSynchronize(h->call_done[ticket % rs_handle::kTickets]));
  return RS_OK;
}

/* EnbMacEntity::ReceiveCqiIdealControlMessage under USE_REAL_TRACE, enb-mac-entity.cc:189-191:
 * int time_stamp = Now()*1000 / CQI_INTERVAL; row = time_stamp % cqi_traces.size() */
int32_t rs_trace_row(double now_seconds, int32_t n_rows) {
  if (n_rows <= 0) return -1;
  volatile double x = now_seconds * 1000;
  const int time_stamp = (int)(x / 40);
  return (int32_t)(time_stamp % n_rows);
}

/* One ue<id>.log as the reference reads it (enb-mac-entity.cc:169-187): n_rows lines, the first n_rbs
 * integers of each (operator>> semantics: a short or unreadable line repeats the last value read). */
int rs_parse_trace_file(const char* path, int32_t n_rows, int32_t n_rbs, uint8_t* out) {
  if (!path || !out || n_rows < 1 || n_rbs < 1) return fail(RS_ERR_ARG, "rs_parse_trace_file: bad argument");
  FILE* f = fopen(path, "r");
  if (!f) return fail(RS_ERR_ARG, "cannot open %s", path);
  std::vector<char> line(1 << 16);
  int cqi = 0;
  for (int i = 0; i < n_rows; ++i) {
    const char* p = "";
    if (fgets(line.data(), (int)line.size(), f)) p = line.data();
    for (int j = 0; j < n_rbs; ++j) {
      char* end = nullptr;
      const long v = strtol(p, &end, 10);
      if (end != p) { cqi = (int)v; p = end; }
      if (cqi < 0 || cqi > 15) { fclose(f); return fail(RS_ERR_ARG, "%s line %d: CQI %d outside 0..15", path, i + 1, cqi); }
      out[(size_t)i * n_rbs + j] = (uint8_t)cqi;
    }
  }
  fclose(f);
  return RS_OK;
}

/* mapping.config as the reference reads it (enb-mac-entity.cc:48-55): pairs "uid tid"; the uid is
 * ignored, entry k of the map is the k-th tid in file order. */
int rs_parse_mapping_file(const char* path, int32_t* out, int32_t cap, int32_t* n_out) {
  if (!path || !n_out || cap < 0 || (cap > 0 && !out)) return fail(RS_ERR_ARG, "rs_parse_mapping_file: bad argument");
  FILE* f = fopen(path, "r");
  if (!f) return fail(RS_ERR_ARG, "cannot open %s", path);
  int uid, tid, n = 0;
  while (fscanf(f, "%d %d", &uid, &tid) == 2) {
    if (n < cap) out[n] = tid;
    n++;
  }
  fclose(f);
  *n_out = n;
  return RS_OK;
}

int rs_set_traces(rs_handle* h, const uint8_t* traces, int32_t n_traces, int32_t n_rows, const int32_t* ue_trace) {
  if (!h || !traces || !ue_trace || n_traces < 1 || n_rows < 1) return fail(RS_ERR_ARG, "rs_set_traces: bad argument");
  const int R = h->d.R, G = h->d.G, rbg = h->d.rbg, C = h->cqi_cols, lay = h->d.cqi_per_rb;
  const size_t per_trace = (size_t)(n_rows + 1) * C;
  if (per_trace * ((size_t)n_traces + 1) > 0x7fffffffull) return fail(RS_ERR_UNSUPPORTED, "trace table larger than 2 GiB");
  /* pseudo-trace n_traces: CQI 10 on every line, for UEs whose reports never arrive (ue_trace = -1) */
  std::vector<uint8_t> tab(per_trace * ((size_t)n_traces + 1), (uint8_t)(lay == 2 ? 0xAA : 10));
  for (int k = 0; k < n_traces; ++k)
    for (int i = 0; i <= n_rows; ++i) {
      uint8_t* dst = tab.data() + (size_t)k * per_trace + (size_t)i * C;
      const uint8_t* src = traces + ((size_t)k * n_rows + i) * R;
      for (int g = 0; g < G; ++g) {
        int v0 = 10;   /* row n_rows: UserEquipmentRecord's initial feedback, ENodeB.cpp:207-217 */
        for (int r = 0; r < rbg; ++r) {
          const int v = (i < n_rows) ? src[(size_t)g * rbg + r] : 10;
          if (v < 1 || v > 15) return fail(RS_ERR_ARG, "trace %d row %d RB %d: CQI %d outside 1..15", k, i, g * rbg + r, v);
          if (r == 0) v0 = v;
          if (lay == 1) dst[(size_t)g * rbg + r] = (uint8_t)v;
          else if (v != v0)
            return fail(RS_ERR_UNSUPPORTED, "trace %d row %d: CQI varies inside RBG %d; create the handle with cqi_per_rb = 1", k, i, g);
        }
        if (lay == 0) dst[g] = (uint8_t)v0;
        else if (lay == 2) dst[g >> 1] = (uint8_t)((g & 1) ? (dst[g >> 1] | (v0 << 4)) : v0);
      }
    }
  const size_t BU = (size_t)h->B * h->d.U;
  std::vector<int> off(BU);
  for (size_t i = 0; i < BU; ++i) {
    if (ue_trace[i] < -1 || ue_trace[i] >= n_traces) return fail(RS_ERR_ARG, "ue_trace[%zu] = %d outside -1..%d", i, ue_trace[i], n_traces - 1);
    off[i] = (int)((size_t)(ue_trace[i] < 0 ? n_traces : ue_trace[i]) * per_trace);
  }
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  int rc = upload(h->trace_tab, tab);
  if (rc != RS_OK) return rc;
  rc = upload(h->ue_trace_off, off);
  if (rc != RS_OK) return rc;
  h->n_traces = n_traces;
  h->trace_rows = n_rows;
  h->d.trace_tab = h->trace_tab.p;
  h->d.ue_trace_off = h->ue_trace_off.p;
  h->d.trace_rows = n_rows;
  return RS_OK;
}

/* ---- log-compatible writer (host only) --------------------------------------------------------
 * Regenerates, from the batch results, the text the reference prints per TTI so that its own plotters
 * (NSDI23-radiosaber-experiments/ ... /plot_throughput.py:35-47) work unchanged. */
struct rs_log {
  int algo = 9, S = 0, U = 0, G = 0, R = 0, rbg = 0, layout = 0, row = 0, data = 0;
  int nb = 1;                   /* bearers per UE; the per-bearer arrays below are [U][nb], slot i = the bearer of priority i */
  std::vector<int> u2s;
  std::vector<int32_t> app;     /* application id of every bearer (rs_log_set_app_ids; default u * nb + i), < 0 = no such bearer */
  std::vector<uint64_t> cum_bytes, cum_rbs;
  std::vector<int32_t> queue;   /* per-bearer dataToTransmit for the next rs_log_tti (rs_log_set_queues), empty = cfg's */
  std::vector<double> hol;
  double eff[16];
  std::string out, err;
};

int rs_log_create(const rs_config* cfg, rs_log** out) {
  if (!cfg || !out || !cfg->ue_to_slice) return fail(RS_ERR_ARG, "rs_log_create: bad argument");
  if (cfg->rbg_size < 1 || cfg->n_rbs < cfg->rbg_size || cfg->n_rbs % cfg->rbg_size != 0 || cfg->n_ues < 1 ||
      cfg->n_slices < 1 || cfg->cqi_per_rb < 0 || cfg->cqi_per_rb > 2)
    return fail(RS_ERR_ARG, "rs_log_create: bad configuration");
  rs_log* lg = new (std::nothrow) rs_log;
  if (!lg) return fail(RS_ERR_ARG, "out of memory");
  lg->algo = cfg->algo; lg->S = cfg->n_slices; lg->U = cfg->n_ues; lg->R = cfg->n_rbs; lg->rbg = cfg->rbg_size;
  lg->G = lg->R / lg->rbg; lg->layout = cfg->cqi_per_rb; lg->data = cfg->data_to_transmit;
  lg->row = lg->layout == 1 ? lg->R : (lg->layout == 2 ? lg->G / 2 : lg->G);
  lg->nb = cfg->n_bearers == 2 ? 2 : 1;
  if (lg->nb == 2 && lg->algo == 1) {   /* id 1 schedules flows: log a two-bearer cell as one user per bearer */
    delete lg;
    return fail(RS_ERR_UNSUPPORTED, "rs_log_create: id 1 schedules flows; give it one user per bearer");
  }
  lg->u2s.assign(cfg->ue_to_slice, cfg->ue_to_slice + lg->U);
  lg->app.resize((size_t)lg->U * lg->nb);
  for (size_t k = 0; k < lg->app.size(); ++k) lg->app[k] = (int32_t)k;
  lg->cum_bytes.assign((size_t)lg->U * lg->nb, 0);
  lg->cum_rbs.assign((size_t)lg->U * lg->nb, 0);
  lg->eff[0] = 0.0;
  for (int c = 1; c <= 15; ++c) lg->eff[c] = eff_from_cqi(c);
  *out = lg;
  return RS_OK;
}

void rs_log_destroy(rs_log* lg) { delete lg; }

int rs_log_set_counters(rs_log* lg, const uint64_t* cum_bytes, const uint64_t* cum_rbs) {
  if (!lg) return fail(RS_ERR_ARG, "null log");
  if (cum_bytes) lg->cum_bytes.assign(cum_bytes, cum_bytes + (size_t)lg->U * lg->nb);
  if (cum_rbs) lg->cum_rbs.assign(cum_rbs, cum_rbs + (size_t)lg->U * lg->nb);
  return RS_OK;
}

int rs_log_set_app_ids(rs_log* lg, const int32_t* app_ids) {
  if (!lg || !app_ids) return fail(RS_ERR_ARG, "rs_log_set_app_ids: bad argument");
  lg->app.assign(app_ids, app_ids + (size_t)lg->U * lg->nb);
  return RS_OK;
}

int rs_log_set_queues(rs_log* lg, const int32_t* queue_bytes, const double* hol_delay) {
  if (!lg) return fail(RS_ERR_ARG, "null log");
  if (queue_bytes) lg->queue.assign(queue_bytes, queue_bytes + (size_t)lg->U * lg->nb); else lg->queue.clear();
  if (hol_delay) lg->hol.assign(hol_delay, hol_delay + (size_t)lg->U * lg->nb); else lg->hol.clear();
  return RS_OK;
}

/* Shared by rs_log_tti and rs_log_tti_grants: rbgs[u] = the RBGs of user u in the order of its RB list,
 * sum_bits = the efficiency sum of the inter-slice algorithm's all_bytes line (in the reference's order). */
static int log_tti_core(rs_log* lg, uint64_t timestamp, const uint8_t* cqi, const std::vector<std::vector<int>>& rbgs,
                        double sum_bits, const int32_t* tbs_bits, const uint8_t* final_cqi, const int32_t* slice_target,
                        const int32_t* slice_quota) {
  const int U = lg->U, S = lg->S, algo = lg->algo;
  const bool tr = algo == 8 || algo == 9 || algo == 10 || algo == 101 || algo == 103;   /* RBsAllocation's log lines */
  char buf[256];
  auto cqi_at = [&](int u, int g) -> int {   /* CQI on the first RB of RBG g, what :641 prints */
    const uint8_t* p = cqi + (size_t)u * lg->row;
    if (lg->layout == 2) return (p[g >> 1] >> (4 * (g & 1))) & 15;
    return lg->layout == 1 ? p[(size_t)g * lg->rbg] : p[g];
  };
  int scheduled = 0;
  for (int u = 0; u < U; ++u) scheduled += (int)rbgs[u].size();
  /* RBsAllocation only runs (and prints) when at least one user is schedulable (transport.cpp:152-168);
   * with every bearer idle nothing is allocated and nothing is printed */
  bool ran = scheduled > 0;
  if (!ran && tr)
    for (int s = 0; s < S; ++s) ran = ran || slice_target[s] != 0 || slice_quota[s] != 0;
  if (ran && algo != 1) {
    if (tr) {
      /* stdout, downlink-transport-scheduler.cpp:523-527 */
      lg->out += "slice_id, target_rbs, quota_rbgs: ";
      for (int s = 0; s < S; ++s) {
        snprintf(buf, sizeof buf, "(%d, %d, %d) ", s, slice_target[s], slice_quota[s]);
        lg->out += buf;
      }
      lg->out += "\n";
      /* stderr, :244 / :270 / :347 / :374 / :449 */
      snprintf(buf, sizeof buf, "all_bytes: %.0f\n", sum_bits * 180 / 8 * 4);
      lg->err += buf;
    }
    /* stdout, :631-649 (NVS: downlink-nvs-scheduler.cpp:314-332) */
    snprintf(buf, sizeof buf, "%llu\n", (unsigned long long)timestamp);
    lg->out += buf;
    for (int u = 0; u < U; ++u) {
      if (rbgs[u].empty()) continue;
      snprintf(buf, sizeof buf, "User(%d) allocated RBGS:", u);
      lg->out += buf;
      for (int g : rbgs[u]) {
        snprintf(buf, sizeof buf, " %d(%d)", g, cqi_at(u, g));
        lg->out += buf;
      }
      snprintf(buf, sizeof buf, " final_cqi: %d\n", (int)final_cqi[u]);
      lg->out += buf;
    }
  }
  /* stderr, DoStopSchedule: transport.cpp:177-199, nvs.cpp:226-251, dl-pf-packet-scheduler.cpp:80-96.
   * Application id: rs_log_set_app_ids, by default bearer k = u * nb + i is application k (== the user id with one bearer
   * per UE); the head-of-line delay (0 for an infinite buffer) is printed the way operator<< prints a double, i.e. %g. */
  const int nb = lg->nb;
  for (int u = 0; u < U; ++u) {
    int avail = tbs_bits[u] / 8;
    /* the bearer of priority 1 is served first, what is left goes to the other one; every bearer that sends is booked
     * the user's whole RB count (transport.cpp:179-191, nvs.cpp:231-243) */
    for (int i = nb - 1; i >= 0; --i) {
      if (avail <= 0) break;
      const size_t k = (size_t)u * nb + i;
      if (lg->app[k] < 0) continue;
      int sent = avail;
      if (algo != 1) {
        const int data = lg->queue.empty() ? lg->data : lg->queue[k];
        if (data <= 0) continue;
        sent = std::min(avail, data);
      }
      avail -= sent;
      lg->cum_bytes[k] += (uint64_t)sent;
      lg->cum_rbs[k] += (uint64_t)rbgs[u].size() * lg->rbg;
      snprintf(buf, sizeof buf, "%llu app: %d cumu_bytes: %llu cumu_rbs: %llu hol_delay: %g user: %d slice: %d\n",
               (unsigned long long)timestamp, (int)lg->app[k], (unsigned long long)lg->cum_bytes[k],
               (unsigned long long)lg->cum_rbs[k], lg->hol.empty() ? 0.0 : lg->hol[k], u, lg->u2s[u]);
      lg->err += buf;
    }
  }
  lg->queue.clear();
  lg->hol.clear();
  return RS_OK;
}

static int log_cqi_at(const rs_log* lg, const uint8_t* cqi, int u, int g) {
  const uint8_t* p = cqi + (size_t)u * lg->row;
  if (lg->layout == 2) return (p[g >> 1] >> (4 * (g & 1))) & 15;
  return lg->layout == 1 ? p[(size_t)g * lg->rbg] : p[g];
}

int rs_log_tti(rs_log* lg, uint64_t timestamp, const uint8_t* cqi, const int16_t* rbg_to_ue, const int32_t* tbs_bits,
               const uint8_t* final_cqi, const int32_t* slice_target, const int32_t* slice_quota) {
  if (!lg || !cqi || !rbg_to_ue || !tbs_bits) return fail(RS_ERR_ARG, "rs_log_tti: bad argument");
  const int U = lg->U, G = lg->G, algo = lg->algo;
  if (algo == 10) return fail(RS_ERR_ARG, "rs_log_tti: id 10 books an RBG to several users, use rs_log_tti_grants");
  const bool tr = algo == 8 || algo == 9 || algo == 101 || algo == 103;
  if (tr && (!slice_target || !slice_quota)) return fail(RS_ERR_ARG, "rs_log_tti: ids 8/9/101/103 need targets and quotas");
  if (algo != 1 && !final_cqi) return fail(RS_ERR_ARG, "rs_log_tti: final_cqi missing");
  std::vector<std::vector<int>> rbgs(U);
  double sum_bits = 0;   /* :366-374 / :265-270: sum over RBGs of the winner's efficiency, in RBG order */
  for (int g = 0; g < G; ++g) {
    const int u = rbg_to_ue[g];
    if (u < -1 || u >= U) return fail(RS_ERR_ARG, "rs_log_tti: rbg_to_ue[%d] = %d", g, u);
    if (u >= 0) rbgs[u].push_back(g);
    sum_bits += u >= 0 ? lg->eff[log_cqi_at(lg, cqi, u, g)] : 0.0;
  }
  return log_tti_core(lg, timestamp, cqi, rbgs, sum_bits, tbs_bits, final_cqi, slice_target, slice_quota);
}

int rs_log_tti_grants(rs_log* lg, uint64_t timestamp, const uint8_t* cqi, int32_t n_grants, const int16_t* grant_ue,
                      const int16_t* grant_rbg, const int32_t* tbs_bits, const uint8_t* final_cqi,
                      const int32_t* slice_target, const int32_t* slice_quota) {
  if (!lg || !cqi || n_grants < 0 || (n_grants > 0 && (!grant_ue || !grant_rbg)) || !tbs_bits || !final_cqi || !slice_target ||
      !slice_quota)
    return fail(RS_ERR_ARG, "rs_log_tti_grants: bad argument");
  if (lg->algo != 10) return fail(RS_ERR_ARG, "rs_log_tti_grants: the grant list is id 10's output");
  const int U = lg->U, G = lg->G;
  std::vector<std::vector<int>> rbgs(U);
  double sum_bits = 0;   /* :240-244: sum over the grants in the order they were made (slice by slice) */
  for (int e = 0; e < n_grants; ++e) {
    const int u = grant_ue[e], g = grant_rbg[e];
    if (u < 0) continue;   /* a slice without a listed user on that RBG: efficiency 0, nobody's RB list grows */
    if (u >= U || g < 0 || g >= G) return fail(RS_ERR_ARG, "rs_log_tti_grants: grant %d = (%d, %d)", e, u, g);
    rbgs[u].push_back(g);
    sum_bits += lg->eff[log_cqi_at(lg, cqi, u, g)];
  }
  return log_tti_core(lg, timestamp, cqi, rbgs, sum_bits, tbs_bits, final_cqi, slice_target, slice_quota);
}

const char* rs_log_stdout(rs_log* lg, int64_t* len) {
  if (!lg) return "";
  if (len) *len = (int64_t)lg->out.size();
  return lg->out.c_str();
}
const char* rs_log_stderr(rs_log* lg, int64_t* len) {
  if (!lg) return "";
  if (len) *len = (int64_t)lg->err.size();
  return lg->err.c_str();
}
void rs_log_clear(rs_log* lg) {
  if (lg) { lg->out.clear(); lg->err.clear(); }
}
int rs_log_get_counters(rs_log* lg, uint64_t* cum_bytes, uint64_t* cum_rbs) {
  if (!lg) return fail(RS_ERR_ARG, "null log");
  if (cum_bytes) memcpy(cum_bytes, lg->cum_bytes.data(), sizeof(uint64_t) * lg->U * lg->nb);
  if (cum_rbs) memcpy(cum_rbs, lg->cum_rbs.data(), sizeof(uint64_t) * lg->U * lg->nb);
  return RS_OK;
}

int rs_set_queues(rs_handle* h, const int32_t* queue_bytes, const double* hol_delay) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  if (hol_delay && !queue_bytes) return fail(RS_ERR_ARG, "rs_set_queues: head-of-line delays without queue sizes");
  if (h->buf_k > 0 && queue_bytes)
    return fail(RS_ERR_ARG, "rs_set_queues: the handle keeps its own buffers (rs_enable_buffers); give it rs_set_traffic");
  h->q_next = queue_bytes;
  h->hol_next = hol_delay;
  return RS_OK;
}

int rs_enable_buffers(rs_handle* h, int32_t max_records, const uint8_t* backlogged) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  if (max_records < 0 || max_records > RS_MAX_BUFFER_RECORDS)
    return fail(RS_ERR_ARG, "rs_enable_buffers: max_records %d outside 0..%d", max_records, RS_MAX_BUFFER_RECORDS);
  const int rc = rs_sync(h);   /* the launches in flight read the old buffers */
  if (rc != RS_OK) return rc;
  h->q_next = nullptr;
  h->hol_next = nullptr;
  h->traffic_set = false;
  h->buf_k = 0;
  h->buf_meta.release(); h->buf_time.release(); h->buf_bytes.release(); h->shown_q.release(); h->shown_hol.release();
  h->buf_backlogged.clear();
  h->last_now = -HUGE_VAL;
  if (max_records == 0) return RS_OK;
  const size_t n = (size_t)h->B * h->d.U * h->d.nb;
  CU(h->buf_meta.alloc(n));
  cudaError_t e = h->buf_time.alloc(n * (size_t)max_records);
  if (e == cudaSuccess) e = h->buf_bytes.alloc(n * (size_t)max_records);
  if (e != cudaSuccess) {
    h->buf_meta.release(); h->buf_time.release(); h->buf_bytes.release();
    return fail(RS_ERR_CUDA, "rs_enable_buffers: cudaMalloc of %zu bearers x %d records: %s", n, max_records, cudaGetErrorString(e));
  }
  if (backlogged) h->buf_backlogged.assign(backlogged, backlogged + n); else h->buf_backlogged.assign(n, 0);
  h->buf_k = max_records;
  return buf_empty(h);
}

int rs_set_traffic(rs_handle* h, const rs_traffic* traffic) {
  if (!h || !traffic) return fail(RS_ERR_ARG, "rs_set_traffic: bad argument");
  if (h->buf_k == 0) return fail(RS_ERR_ARG, "rs_set_traffic: the handle has no buffers (rs_enable_buffers)");
  h->traffic = *traffic;
  h->traffic_set = true;
  return RS_OK;
}

int rs_get_buffers(rs_handle* h, int64_t* queued, int32_t* n_records, double* head_time, uint64_t* dropped) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  if (h->buf_k == 0) return fail(RS_ERR_ARG, "rs_get_buffers: the handle has no buffers (rs_enable_buffers)");
  const int rc = rs_sync(h);
  if (rc != RS_OK) return rc;
  const size_t n = h->buf_backlogged.size();
  std::vector<rs::BufMeta> m(n);
  CU(cudaMemcpy(m.data(), h->buf_meta.p, n * sizeof(rs::BufMeta), cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < n; ++i) {
    const bool fifo = m[i].n >= 0;
    if (queued) queued[i] = fifo ? m[i].queued : 0;
    if (n_records) n_records[i] = fifo ? m[i].n : 0;
    if (dropped) dropped[i] = fifo ? m[i].dropped : 0;
  }
  if (head_time) {
    CU(h->buf_scratch.alloc(n * sizeof(double)));
    const int blocks = (int)std::min<size_t>((n + 255) / 256, 148 * 4);
    rs::rs_buf_heads_kernel<<<blocks, 256, 0, h->stream>>>(h->buf_meta.p, h->buf_time.p, h->buf_k, n, (double*)h->buf_scratch.p);
    CU(cudaGetLastError());
    h->launches++;
    CU(cudaMemcpyAsync(head_time, h->buf_scratch.p, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  return RS_OK;
}

int rs_synth_arrivals(rs_handle* h, uint64_t seed, int64_t cell0, int64_t tti0, int32_t n_ttis, const int32_t* pkt_bytes,
                      const int32_t* pkts_q16, int32_t* d_out) {
  if (!h || !pkt_bytes || !pkts_q16 || !d_out || n_ttis < 0) return fail(RS_ERR_ARG, "rs_synth_arrivals: bad argument");
  const int P = h->P, S = h->d.S;
  std::vector<int> spec((size_t)2 * P * S);
  for (int i = 0; i < P * S; ++i) {
    if (pkt_bytes[i] < 0 || pkts_q16[i] < 0)
      return fail(RS_ERR_ARG, "rs_synth_arrivals: profile %d slice %d: negative packet size or rate", i / S, i % S);
    if ((long long)pkt_bytes[i] * ((pkts_q16[i] >> 16) + 1) > 0x7fffffffLL)
      return fail(RS_ERR_ARG, "rs_synth_arrivals: profile %d slice %d: a TTI's bytes overflow int32", i / S, i % S);
    spec[2 * i] = pkt_bytes[i];
    spec[2 * i + 1] = pkts_q16[i];
  }
  CU(cudaSetDevice(h->device));
  CU(h->synth_spec.alloc(spec.size()));
  /* pageable source: the copy is staged before the call returns; ordered with earlier kernels that read the table */
  CU(cudaMemcpyAsync(h->synth_spec.p, spec.data(), spec.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  auto sm64 = [](unsigned long long x) {
    unsigned long long z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  };
  const unsigned long long key = sm64((seed & 0xFFFFFFFFull) | (0x41525200ull << 32));   /* "ARR\0" */
  const size_t total_n = (size_t)n_ttis * h->B * h->d.U * h->d.nb;
  if (total_n == 0) return RS_OK;
  const int blocks = (int)std::min<size_t>((total_n + 255) / 256, 148 * 16);
  rs::rs_synth_arrivals_kernel<<<blocks, 256, 0, h->stream>>>(d_out, key, cell0, tti0, n_ttis, h->d, h->synth_spec.p);
  CU(cudaGetLastError());
  h->launches++;
  return RS_OK;
}

int rs_arrival_spec(double pkt_bytes, double pkts_per_tti, int32_t* pkt_bytes_out, int32_t* pkts_q16) {
  if (!pkt_bytes_out || !pkts_q16) return fail(RS_ERR_ARG, "rs_arrival_spec: bad argument");
  if (!(pkt_bytes >= 0 && pkt_bytes <= 0x7fffffff) || pkt_bytes != std::floor(pkt_bytes))
    return fail(RS_ERR_ARG, "pkt_bytes %g is not an integer 0..2147483647", pkt_bytes);
  if (!std::isfinite(pkts_per_tti) || pkts_per_tti < 0)
    return fail(RS_ERR_ARG, "pkts_per_tti %g is not a finite rate >= 0", pkts_per_tti);
  const double q = std::round(pkts_per_tti * 65536.0);   /* the product is exact: a power-of-two scale */
  if (q > 0x7fffffff) return fail(RS_ERR_ARG, "pkts_per_tti %g does not fit 16.16 fixed point (under 32768 packets per TTI)", pkts_per_tti);
  if (pkts_per_tti > 0 && q == 0)
    return fail(RS_ERR_ARG, "pkts_per_tti %g is below 1/65536 packet per TTI (16.16 fixed point)", pkts_per_tti);
  const long long qi = (long long)q;
  if ((long long)pkt_bytes * ((qi >> 16) + 1) > 0x7fffffffLL)
    return fail(RS_ERR_ARG, "pkt_bytes %g at %g packets per TTI: a TTI's bytes overflow int32", pkt_bytes, pkts_per_tti);
  *pkt_bytes_out = (int32_t)pkt_bytes;
  *pkts_q16 = (int32_t)qi;
  return RS_OK;
}

int rs_step(rs_handle* h, const uint8_t* cqi, const int32_t* rand2, const uint8_t* active, double dt,
            const rs_outputs* out) {
  return rs_run_host(h, 1, cqi, 1, rand2, active, &dt, out, 1);
}

/* One TTI with everything the in-simulator plug-in moves per TTI in ONE host-to-device copy, one launch, one
 * device-to-host copy and one synchronisation: the mailbox is [inputs | state | outputs], the state part goes up
 * and comes back. */
int rs_step_cell(rs_handle* h, const rs_cell_io* io) {
  if (!h || !io || !io->cqi) return fail(RS_ERR_ARG, "rs_step_cell: bad argument");
  h->q_next = nullptr;
  h->hol_next = nullptr;
  h->traffic_set = false;
  if (h->buf_k > 0)
    return fail(RS_ERR_ARG, "rs_step_cell: the handle keeps its own buffers; inside a simulator the simulator owns the queues");
  if (io->hol_delay && !io->queue_bytes) return fail(RS_ERR_ARG, "rs_step_cell: head-of-line delays without queue sizes");
  if (h->d.rand_stride > 0 && !io->rand2) return fail(RS_ERR_ARG, "ids 8/9/11 need the rand() draws");
  if (h->d.nb == 2 && !io->queue_bytes) return fail(RS_ERR_ARG, "two bearers per UE: the call needs queue_bytes");
  CU(cudaSetDevice(h->device));
  const size_t B = h->B, U = h->d.U, S = h->d.S, G = h->d.G, C = h->cqi_cols, RS = (size_t)h->d.rand_stride;
  const size_t NB = (size_t)h->d.nb;
  const rs_outputs& o = io->out;
  const bool nvs = h->d.algo == 7 || h->d.algo == 11, tr = is_transport(h->d.algo);
  size_t off = 0;
  auto take = [&](bool want, size_t bytes) { const size_t at = off; if (want) off += (bytes + 15) & ~(size_t)15; return at; };
  const size_t o_cqi = take(true, B * U * C), o_rand = take(io->rand2 && RS, B * RS * 4), o_act = take(io->active, B * U),
               o_q = take(io->queue_bytes, B * U * NB * 4), o_hol = take(io->hol_delay, B * U * NB * 8);
  const size_t state0 = off;
  const bool st = io->slice_state && (nvs || tr);
  const size_t o_avg = take(io->avg_rate, B * U * NB * 8), o_st = take(st, B * S * 8);
  const size_t out0 = off;
  const size_t o_rbg = take(o.rbg_to_ue, B * G * 2), o_bits = take(o.tbs_bits, B * U * 4), o_mcs = take(o.mcs, B * U),
               o_fc = take(o.final_cqi, B * U), o_tgt = take(o.slice_target && tr, B * S * 4),
               o_quo = take(o.slice_quota && tr, B * S * 4), o_nvs = take(o.nvs_slice && nvs, B * 4),
               o_an = take(o.alloc_n && h->d.algo == 10, B * 4), o_au = take(o.alloc_ue && h->d.algo == 10, B * h->d.grant_len * 2),
               o_ar = take(o.alloc_rbg && h->d.algo == 10, B * h->d.grant_len * 2);
  const size_t total = off;
  if (h->mb_bytes < total) {
    CU(cudaStreamSynchronize(h->stream));
    if (h->mb_host) cudaFreeHost(h->mb_host);
    h->mb_host = nullptr;
    h->mb_bytes = 0;
    CU(cudaMallocHost((void**)&h->mb_host, total));
    CU(h->mb_dev.alloc(total));
    h->mb_bytes = total;
  }
  unsigned char* m = h->mb_host;
  unsigned char* dm = h->mb_dev.p;
  memcpy(m + o_cqi, io->cqi, B * U * C);
  if (io->rand2 && RS) memcpy(m + o_rand, io->rand2, B * RS * 4);
  if (io->active) memcpy(m + o_act, io->active, B * U);
  if (io->queue_bytes) memcpy(m + o_q, io->queue_bytes, B * U * NB * 4);
  if (io->hol_delay) memcpy(m + o_hol, io->hol_delay, B * U * NB * 8);
  if (io->avg_rate) memcpy(m + o_avg, io->avg_rate, B * U * NB * 8);
  if (st) memcpy(m + o_st, io->slice_state, B * S * 8);
  CU(cudaMemcpyAsync(dm, m, out0, cudaMemcpyHostToDevice, h->stream));
  rs::DevCfg d = h->d;
  if (io->avg_rate) d.avg = (double*)(dm + o_avg);
  if (st) { if (nvs) d.ewma = (double*)(dm + o_st); else d.offset = (double*)(dm + o_st); }
  rs::RunArgs a{};
  a.T = 1;
  a.cqi = dm + o_cqi; a.cqi_tti_stride = (long long)(B * U * C);
  a.t0 = 0; a.cqi_refresh = 1;
  a.rand2 = (io->rand2 && RS) ? (const int*)(dm + o_rand) : nullptr;
  a.active = io->active ? dm + o_act : nullptr; a.active_tti_stride = (long long)(B * U);
  a.dt[0] = io->dt;
  a.queue = io->queue_bytes ? (const int*)(dm + o_q) : nullptr;
  a.hol = io->hol_delay ? (const double*)(dm + o_hol) : nullptr;
  a.stage = h->stage_ok ? 1 : 0;
  rs_outputs so{};
  so.rbg_to_ue = o.rbg_to_ue ? (int16_t*)(dm + o_rbg) : nullptr;
  so.tbs_bits = o.tbs_bits ? (int32_t*)(dm + o_bits) : nullptr;
  so.mcs = o.mcs ? dm + o_mcs : nullptr;
  so.final_cqi = o.final_cqi ? dm + o_fc : nullptr;
  so.slice_target = (o.slice_target && tr) ? (int32_t*)(dm + o_tgt) : nullptr;
  so.slice_quota = (o.slice_quota && tr) ? (int32_t*)(dm + o_quo) : nullptr;
  so.nvs_slice = (o.nvs_slice && nvs) ? (int32_t*)(dm + o_nvs) : nullptr;
  if (h->d.algo == 10) {
    so.alloc_n = o.alloc_n ? (int32_t*)(dm + o_an) : nullptr;
    so.alloc_ue = o.alloc_ue ? (int16_t*)(dm + o_au) : nullptr;
    so.alloc_rbg = o.alloc_rbg ? (int16_t*)(dm + o_ar) : nullptr;
  }
  point_outputs(h, &a, &so, 0);
  const int rc = launch_ttis(h, a, false, &d);
  if (rc != RS_OK) { cudaStreamSynchronize(h->stream); return rc; }
  if (total > state0) CU(cudaMemcpyAsync(m + state0, dm + state0, total - state0, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (io->avg_rate) memcpy(io->avg_rate, m + o_avg, B * U * NB * 8);
  if (st) memcpy(io->slice_state, m + o_st, B * S * 8);
  if (so.rbg_to_ue) memcpy(o.rbg_to_ue, m + o_rbg, B * G * 2);
  if (so.tbs_bits) memcpy(o.tbs_bits, m + o_bits, B * U * 4);
  if (so.mcs) memcpy(o.mcs, m + o_mcs, B * U);
  if (so.final_cqi) memcpy(o.final_cqi, m + o_fc, B * U);
  if (so.slice_target) memcpy(o.slice_target, m + o_tgt, B * S * 4);
  if (so.slice_quota) memcpy(o.slice_quota, m + o_quo, B * S * 4);
  if (so.nvs_slice) memcpy(o.nvs_slice, m + o_nvs, B * 4);
  if (so.alloc_n) memcpy(o.alloc_n, m + o_an, B * 4);
  if (so.alloc_ue) memcpy(o.alloc_ue, m + o_au, B * h->d.grant_len * 2);
  if (so.alloc_rbg) memcpy(o.alloc_rbg, m + o_ar, B * h->d.grant_len * 2);
  return RS_OK;
}

int rs_synth_cqi(rs_handle* h, uint64_t seed, int64_t cell0, int64_t epoch0, int32_t n_slabs, uint8_t* d_out) {
  if (!h || !d_out || n_slabs < 0) return fail(RS_ERR_ARG, "rs_synth_cqi: bad argument");
  if (h->d.cqi_per_rb == 1) return fail(RS_ERR_UNSUPPORTED, "synthetic CQI is one value per RBG");
  CU(cudaSetDevice(h->device));
  /* histogram of cqi-traces-noise0 (SURVEY 8d); thresholds as in radiosaber_b200/workload.py */
  static const unsigned long long hist[15] = {19075, 7082, 33860, 261099, 438688, 199446, 518174, 661977,
                                              237928, 861279, 596358, 355319, 447453, 12000, 153462};
  unsigned long long total = 0, cum = 0;
  for (int i = 0; i < 15; ++i) total += hist[i];
  rs::CdfTable cdf;
  for (int i = 0; i < 14; ++i) {
    cum += hist[i];
    cdf.thr[i] = (unsigned)(unsigned long long)(((double)cum / (double)total) * 4294967296.0);
  }
  auto sm64 = [](unsigned long long x) {
    unsigned long long z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  };
  const unsigned long long key = sm64((seed & 0xFFFFFFFFull) | (0x43514900ull << 32));
  const size_t total_n = (size_t)n_slabs * h->B * h->d.U * h->cqi_cols;
  if (total_n == 0) return RS_OK;
  const int blocks = (int)std::min<size_t>((total_n + 255) / 256, 148 * 16);
  rs::rs_synth_cqi_kernel<<<blocks, 256, 0, h->stream>>>(d_out, key, cell0, epoch0, n_slabs, h->B, h->d.U, h->d.G,
                                                         h->d.cqi_per_rb == 2 ? 1 : 0, cdf);
  CU(cudaGetLastError());
  h->launches++;
  return RS_OK;
}

int rs_synth_rand2(rs_handle* h, uint64_t seed, int64_t cell0, int64_t tti0, int32_t n_ttis, int32_t* d_out) {
  if (!h || !d_out || n_ttis < 0) return fail(RS_ERR_ARG, "rs_synth_rand2: bad argument");
  CU(cudaSetDevice(h->device));
  auto sm64 = [](unsigned long long x) {
    unsigned long long z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  };
  const unsigned long long key = sm64((seed & 0xFFFFFFFFull) | (0x524E4400ull << 32));
  const int stride = std::max(h->d.rand_stride, 2);
  const size_t total_n = (size_t)n_ttis * h->B * stride;
  if (total_n == 0) return RS_OK;
  const int blocks = (int)std::min<size_t>((total_n + 255) / 256, 148 * 8);
  rs::rs_synth_rand2_kernel<<<blocks, 256, 0, h->stream>>>(d_out, key, cell0, tti0, n_ttis, h->B, h->d.S, stride);
  CU(cudaGetLastError());
  h->launches++;
  return RS_OK;
}

int rs_stats_device(rs_handle* h, uint64_t* d_stats) {
  if (!h || !d_stats) return fail(RS_ERR_ARG, "rs_stats_device: bad argument");
  CU(cudaSetDevice(h->device));
  const int S = h->d.S;
  const size_t words = (size_t)4 * S * h->P;   /* [P][4][S] */
  CU(cudaMemsetAsync(d_stats, 0, sizeof(uint64_t) * words, h->stream));
  const size_t total = (size_t)h->B * h->d.U;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 4);
  /* per-block sums in shared memory while they fit the default 48 KB: up to 1536 (slice, profile) pairs */
  const int in_smem = words * sizeof(unsigned long long) <= 48 * 1024 ? 1 : 0;
  rs::rs_stats_kernel<<<blocks, 256, in_smem ? sizeof(unsigned long long) * words : 0, h->stream>>>(
      h->d, (unsigned long long*)d_stats, h->P, in_smem);
  CU(cudaGetLastError());
  h->launches++;
  return RS_OK;
}

int rs_buffer_stats_device(rs_handle* h, uint64_t* d_stats) {
  if (!h || !d_stats) return fail(RS_ERR_ARG, "rs_buffer_stats_device: bad argument");
  if (h->buf_k == 0) return fail(RS_ERR_ARG, "rs_buffer_stats_device: the handle has no buffers (rs_enable_buffers)");
  CU(cudaSetDevice(h->device));
  const size_t words = (size_t)3 * h->d.S * h->P;   /* [P][3][S] */
  CU(cudaMemsetAsync(d_stats, 0, sizeof(uint64_t) * words, h->stream));
  const size_t total = (size_t)h->B * h->d.U * h->d.nb;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 4);
  const int in_smem = words * sizeof(unsigned long long) <= 48 * 1024 ? 1 : 0;   /* as rs_stats_device */
  rs::rs_buffer_stats_kernel<<<blocks, 256, in_smem ? sizeof(unsigned long long) * words : 0, h->stream>>>(
      h->buf_meta.p, h->d, (unsigned long long*)d_stats, h->P, in_smem);
  CU(cudaGetLastError());
  h->launches++;
  return RS_OK;
}

int rs_get_buffer_stats(rs_handle* h, uint64_t* stats) {
  if (!h || !stats) return fail(RS_ERR_ARG, "rs_get_buffer_stats: bad argument");
  int rc = rs_buffer_stats_device(h, (uint64_t*)h->stats.p);   /* [P][3][S] fits the [P][4][S] scratch */
  if (rc != RS_OK) return rc;
  CU(cudaMemcpyAsync(stats, h->stats.p, sizeof(uint64_t) * 3 * h->d.S * h->P, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return RS_OK;
}

int rs_get_stats(rs_handle* h, uint64_t* stats) {
  if (!h || !stats) return fail(RS_ERR_ARG, "rs_get_stats: bad argument");
  int rc = rs_stats_device(h, (uint64_t*)h->stats.p);
  if (rc != RS_OK) return rc;
  CU(cudaMemcpyAsync(stats, h->stats.p, sizeof(uint64_t) * 4 * h->d.S * h->P, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return RS_OK;
}

int rs_dims(const rs_handle* h, int32_t* n_cells, int32_t* n_slices, int32_t* n_ues, int32_t* n_rbgs, int32_t* device) {
  if (!h) return fail(RS_ERR_ARG, "null handle");
  if (n_cells) *n_cells = h->B;
  if (n_slices) *n_slices = h->d.S;
  if (n_ues) *n_ues = h->d.U;
  if (n_rbgs) *n_rbgs = h->d.G;
  if (device) *device = h->device;
  return RS_OK;
}
int32_t rs_n_profiles(const rs_handle* h) { return h ? h->P : 0; }
int32_t rs_rand_draws_per_cell_tti(const rs_handle* h) { return h ? h->d.rand_stride : 0; }
int64_t rs_launch_count(const rs_handle* h) { return h ? h->launches : 0; }
int32_t rs_smem_bytes(const rs_handle* h) { return h ? h->layout.total : 0; }
int32_t rs_threads_per_cta(const rs_handle* h) { return (h && h->wide) ? rsw::kThreads : rs::kThreads; }
int32_t rs_fixed_shape(const rs_handle* h) { return h ? h->fixed : -1; }
int32_t rs_direct_metric(const rs_handle* h) { return h ? h->d.direct : 0; }
int64_t rs_algorithmic_bytes_per_cell_tti(const rs_handle* h) {
  if (!h) return 0;
  const int64_t U = h->d.U, G = h->d.G, S = h->d.S;
  return U * (G + 20) + 16 * S + 2 * G + 8;
}

int rs_test_sort(int32_t device, const uint8_t* keys, int32_t n_arrays, int32_t n, int32_t depth_limit,
                 int32_t* perm_out) {
  return rs_test_sort_timed(device, keys, n_arrays, n, depth_limit, perm_out, 1, nullptr);
}

int rs_test_sort_timed(int32_t device, const uint8_t* keys, int32_t n_arrays, int32_t n, int32_t depth_limit,
                       int32_t* perm_out, int32_t reps, float* ms_per_launch) {
  if (!keys || !perm_out || n_arrays < 1 || n < 1 || n > 4096 || reps < 1) return fail(RS_ERR_ARG, "rs_test_sort: bad argument");
  CU(cudaSetDevice(device));
  if (depth_limit < 0) { int lg = 0; for (int m = n; m > 1; m >>= 1) lg++; depth_limit = 2 * lg; }
  const rs::Layout L = rs::make_layout(1, 0, n, 0);
  CU(cudaFuncSetAttribute(rs::rs_sort_test_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
  uint8_t* dk = nullptr;
  int* dp = nullptr;
  unsigned short* de = nullptr;
  const int eq_max = std::min(n, kEqMax);
  if (eq_max >= 17) {
    std::vector<unsigned short> eq;
    build_eq_table(eq_max, &eq);
    CU(cudaMalloc((void**)&de, eq.size() * 2));
    cudaError_t e0 = cudaMemcpy(de, eq.data(), eq.size() * 2, cudaMemcpyHostToDevice);
    if (e0 != cudaSuccess) { cudaFree(de); return fail(RS_ERR_CUDA, "cudaMemcpy: %s", cudaGetErrorString(e0)); }
  }
  CU(cudaMalloc((void**)&dk, (size_t)n_arrays * n));
  cudaError_t e = cudaMalloc((void**)&dp, (size_t)n_arrays * n * 4);
  if (e != cudaSuccess) { cudaFree(dk); return fail(RS_ERR_CUDA, "cudaMalloc: %s", cudaGetErrorString(e)); }
  e = cudaMemcpy(dk, keys, (size_t)n_arrays * n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    rs::rs_sort_test_kernel<<<n_arrays, rs::kThreads, L.total>>>(dk, n, depth_limit, dp, de, de ? eq_max : 0, L);
    cudaEventRecord(e0);
    for (int r = 1; r < reps; ++r)
      rs::rs_sort_test_kernel<<<n_arrays, rs::kThreads, L.total>>>(dk, n, depth_limit, dp, de, de ? eq_max : 0, L);
    cudaEventRecord(e1);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaEventSynchronize(e1);
    if (e == cudaSuccess && ms_per_launch && reps > 1) {
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      *ms_per_launch = ms / (float)(reps - 1);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
  }
  if (e == cudaSuccess) e = cudaMemcpy(perm_out, dp, (size_t)n_arrays * n * 4, cudaMemcpyDeviceToHost);
  cudaFree(dk);
  cudaFree(dp);
  if (de) cudaFree(de);
  if (e != cudaSuccess) return fail(RS_ERR_CUDA, "rs_test_sort: %s", cudaGetErrorString(e));
  return RS_OK;
}

}  /* extern "C" */
