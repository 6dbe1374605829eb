/* rs_device.cuh -- sm_100a kernels of the per-TTI downlink RBG allocation, one CTA per cell.
 *
 * Reference behaviour reproduced (paths under /root/reference/src/protocolStack/mac/packet-scheduler
 * unless a directory is given; "transport.cpp" = downlink-transport-scheduler.cpp, "nvs.cpp" =
 * downlink-nvs-scheduler.cpp, "dlps.cpp" = downlink-packet-scheduler.cpp):
 *   EWMA of the served rate        flows/radio-bearer.cpp:138-164
 *   scheduling metric              transport.cpp:677-713, nvs.cpp:360-390, dl-pf-packet-scheduler.cpp:128-140
 *   per-slice enterprise argmax    transport.cpp:543-567
 *   slice targets / RBG quotas     transport.cpp:463-521
 *   RadioSaber MaximizeCell        transport.cpp:351-376 (std::sort order, SURVEY H1)
 *   Sequential GreedyByRow         transport.cpp:249-272
 *   NVS slice selection / argmax   nvs.cpp:94-142, 275-311
 *   No-slicing PF argmax           dlps.cpp:179-271 (flow-satisfied cut-off :264-269 with finite queues)
 *   UpperBound / SubOpt / Vogel    transport.cpp:223-246, 274-349, 378-451
 *   NVS non-greedy PF search       nvs.cpp:405-528
 *   queue-aware metrics            transport.cpp:694-711, nvs.cpp:384-386, packet-scheduler.cpp:321-334
 *   trace-driven CQI               protocolStack/mac/enb-mac-entity.cc:160-193
 *   EESM -> CQI -> MCS -> TBS      transport.cpp:632-660, utility/eesm-effective-sinr.h:33-46,
 *                                  protocolStack/mac/AMCModule.cpp:252-317
 *   byte / RB accounting           transport.cpp:170-199, dl-pf-packet-scheduler.cpp:64-96,
 *                                  flows/radio-bearer.cpp:100-123
 *
 * Everything that decides an assignment is integer or IEEE-754 double arithmetic with explicit
 * rounding (__dmul_rn/__dadd_rn/__ddiv_rn: no FMA contraction), so results are bit-identical to the
 * reference's x86-64 build; libm values (pow/exp/log/log10) enter only through tables computed on
 * the host with glibc (rs_sched.cu).
 */
/* No include guard: rs_sched.cu includes this file twice, once per CTA width (RS_NS = the namespace,
 * RS_THREADS = threads per cell, RS_MIN_BLOCKS = cells per SM the register budget must allow). */
#include <cuda_runtime.h>
#include <stdint.h>
#include <cstdio>

#ifndef RS_NS
#define RS_NS rs
#endif
namespace RS_NS {

#ifdef RS_PHASE_TIMING
#define RS_TICK(k) do { if (threadIdx.x == 0) { long long now_ = clock64(); ph_[k] += now_ - last_; last_ = now_; } } while (0)
#else
#define RS_TICK(k) do {} while (0)
#endif

#ifndef RS_THREADS
#define RS_THREADS 128
#endif
#ifndef RS_MIN_BLOCKS
#define RS_MIN_BLOCKS 8
#endif
constexpr int kThreads = RS_THREADS;   /* threads per CTA (one CTA = one cell) */
constexpr int kWarps = kThreads / 32;
constexpr int kSortThreshold = 16;     /* libstdc++ _S_threshold, bits/stl_algo.h:1848 */
constexpr int kMStride = 16;           /* metric table row: entries for CQI 0..15 */
constexpr unsigned kFull = 0xffffffffu;
constexpr unsigned short kNoUe = 0xffff;
constexpr int kMaxQueueBytes = 268435455;  /* queue sizes saturate here: data * 8 is an int in the reference (2^31 overflows there) */
constexpr int kMaxTtisPerLaunch = 64;  /* TTIs one launch can take (their dt / trace row ride in the kernel parameters) */

/* ---- tables that are the same for every handle (set once per device) ------------------------- */
struct ConstTables {
  double tval[16];   /* exp(-10^(SINR[cqi]/10)), the EESM summand of a CQI (eesm-effective-sinr.h:39-41) */
  double eff[16];    /* AMCModule::GetEfficiencyFromCQI per CQI (AMCModule.cpp:319-327), eff[0] = 0: the
                        flow_spectraleff of a (rbg, slice) pair (ids 101/103 work on differences of it) */
  double cut[16];    /* cut[k], k=1..14: largest mean with 10*log10(-log(mean)) >= SINRForCQIIndex[k]
                        (AMCModule.cpp:252-261 expressed on the EESM mean) */
};
static __constant__ ConstTables c_tab;   /* one copy per translation unit that holds kernels (rs_kernels.cu sets its own) */

/* One bearer's byte FIFO (rs_enable_buffers): `n` records from ring slot `head` on, `queued` = the sum of their bytes;
 * n = -1 = a backlogged bearer (no FIFO, the infinite buffer). */
struct BufMeta {
  long long queued;
  unsigned long long dropped;   /* bytes of arrivals refused because the FIFO held its K records */
  int head, n;
};

/* ---- per-handle description (lives in kernel parameter space) -------------------------------- */
struct Layout {
  int avg, den, mtab, tx, mask, seg0, seg1, cnt, a, win, posl, posr,
      target, quota, frb, wd, outsl, off, tval, misc, utr, sptr, sues, cq, mbar, ng_hc, ng_list, ng_mcs, ng_red, done, total;
};

struct DevCfg {
  int algo, S, U, G, R, rbg, cqi_per_rb, data;   /* cqi_per_rb: 0 u8/RBG, 1 u8/RB, 2 two RBGs per byte */
  int cqi_row;             /* bytes of CQI per UE: G, R or G/2 */
  Layout lay;              /* shared-memory offsets, computed once on the host (make_layout) */
  int n_cells;
  int n_chunks;            /* metric-table chunks (ranges of slices) */
  int m_cap;               /* metric-table capacity in UEs */
  int sort_n;              /* G*S */
  int sort_depth;          /* 2*floor(log2(G*S)) */
  int nvs_guard;           /* 1: NVS required-RBs guard can bind (finite data) -> unsupported for now */
  const int* ue_to_slice;  /* [U] */
  const int* slice_ptr;    /* [S+1] CSR over UEs sorted by (slice, ue); algo 1: one "slice" = all UEs */
  const int* slice_ues;    /* [U] */
  const int* chunk_slice;  /* [n_chunks+1] first slice of each chunk */
  const double* weight;    /* [S] */
  const double* epow;      /* [S][16]: pow(eff(c)*180000/1000, epsilon_s) (ids 7/8/9); [1][16] eff*180000 (id 1) */
  const unsigned char* psi;/* [S] 0/1 */
  const int* tbs_n;        /* [G+1][16]: GetTBSizeFromMCS(mcs(cqi), k*rbg) */
  const unsigned short* eq_tab; /* id 9: permutations of all-equal ranges (SortBufs::eq_tab) */
  int eq_max;
  /* trace-driven CQI (enb-mac-entity.cc:160-193): [n_traces][trace_rows + 1][cqi_row] in the handle's
   * CQI layout, row trace_rows = the all-10 vector a UE record holds before its first report
   * (ENodeB.cpp:207-217); ue_trace_off[b][u] = byte offset of the trace UE u of cell b replays */
  const uint8_t* trace_tab;
  const int* ue_trace_off;
  int trace_rows;
  int rand_stride;         /* int32 rand() draws per cell-TTI in RunArgs::rand2: 2 (ids 8/9), 300 x max UEs per slice (id 11) */
  int ng_ues;              /* id 11: largest slice */
  const unsigned char* holmul; /* [S] 1: the slice's metric carries the head-of-line delay (transport.cpp:702-706
                                  when alpha and beta are set; nvs.cpp:384-386 whenever alpha is set) */
  const int* tbs1;             /* [16] GetTBSizeFromMCS(mcs(cqi)) for one RB: m_requiredRBs, packet-scheduler.cpp:334 */
  const short* vogel_tab;      /* id 103: [kVogelTab] built on the host from the doubles the reference subtracts (rs_sched.cu build_vogel_tab) */
  int sort_depth_g;        /* id 10: 2*floor(log2(G)), the depth limit of a per-slice sort of G entries */
  int direct;              /* 1: big slices, the per-slice argmax divides its metrics on the fly instead of tabulating them per
                              chunk (rs_tti_kernel, "P2 for big slices"); the table area then holds Epow's S rows */
  int nb;                  /* bearers per UE (MAX_BEARERS, packet-scheduler.h:31): 1, or 2 = slot i holds the bearer of priority i;
                              state arrays are then [B][U][2] and the queue-aware kernels (QUEUE) are the only ones used */
  /* state, [B][U][nb] / [B][S] */
  double* avg; int* tx; unsigned long long* cum_bytes; unsigned long long* cum_rbs;
  double* offset; double* ewma;
  /* slice profiles (rs_create_profiles): weight, epow (ids 7/8/9/10/101/103), psi and holmul are [P][S] ([P][S][16]),
   * ue_to_slice and slice_ues [P][U], slice_ptr [P][S+1] ([P][2] for id 1), chunk_slice [P][n_chunks+1] (profiles with
   * fewer chunks end in empty ones); cell b uses row cell_profile[b], null = row 0 for every cell */
  const int* cell_profile;
  int grant_len;           /* id 10: entries per cell of the alloc_ue / alloc_rbg outputs (rs_set_grant_list_len), 2G..S*G */
};

/* The dimensions of a cell as the device code reads them (see rs_tti_kernel and the shape policies below). */
struct Dims {
  int S, U, G, R, rbg, cqi_per_rb, cqi_row, n_chunks, m_cap, sort_n, sort_depth, nb, direct;
  Layout lay;
};

struct RunArgs {
  const uint8_t* cqi; long long cqi_tti_stride;   /* TTI t reads slab (t0 + t) / cqi_refresh */
  int t0, cqi_refresh;
  int stage;               /* 1: every TTI's CQI is copied to shared memory with cp.async first */
  const int* queue;        /* [T][B][U][nb] bytes queued on each UE's bearer(s) (its dataToTransmit; 0 = not listed), or null:
                              DevCfg::data for everybody */
  const double* hol;       /* [T][B][U][nb] head-of-line delay of the bearer(s), or null (0) */
  const int* rand2;
  const uint8_t* active; long long active_tti_stride;
  /* per-TTI scalars travel in the kernel parameters (no copy, no staging buffer): at most kMaxTtisPerLaunch TTIs */
  double dt[kMaxTtisPerLaunch];       /* Now - lastUpdate of the EWMA at TTI t (flows/radio-bearer.cpp:150) */
  int trace_row[kMaxTtisPerLaunch];   /* trace mode: row of every UE's trace in force at TTI t */
  int T;
  int cell_off;            /* first cell of this launch (the host may run the two halves of a batch on two streams) */
  short* rbg_to_ue; int* tbs_bits; uint8_t* mcs; uint8_t* final_cqi;
  int* slice_target; int* slice_quota; int* nvs_slice;
  int* alloc_n; short* alloc_ue; short* alloc_rbg;   /* id 10: [T][B], [T][B][grant_len], [T][B][grant_len] */
  /* Per-bearer byte FIFOs (rs_enable_buffers), used by the queue-aware kernels only (the fields sit behind every other
   * parameter, so the other kernels' parameter offsets are those of a handle without them).  buf_k records per bearer,
   * 0 = off; buf_meta [B][U][nb], buf_time / buf_bytes [B][U][nb][buf_k] (a ring per bearer); arrivals [T][B][U][nb]
   * bytes arriving at each bearer.  `queue` / `hol` are then written by the kernel (what each TTI shows the scheduler)
   * before they are read. */
  int buf_k;
  BufMeta* buf_meta;
  double* buf_time;
  int* buf_bytes;
  const int* arrivals;
  double now[kMaxTtisPerLaunch];        /* simulator time of TTI t: HoL delay = now - arrival time of the head record */
  double arr_time[kMaxTtisPerLaunch];   /* arrival time stamped on the records TTI t pushes */
};

/* ---- shared-memory layout (same function on host and device) --------------------------------- */
__host__ __device__ constexpr inline int rs_align(int x, int a) { return (x + a - 1) / a * a; }
/* The cumulative byte / RB counters stay in HBM (touched only for the few UEs a TTI serves); the
 * metric table is dead once the sort starts, so it shares the bytes of the sort's slot arrays
 * when it fits there. */
/* cq_bytes: room for one TTI of the cell's CQI ([U][cqi_row], staged with cp.async); 0 = CQI is read
 * from global memory where it lies. */
/* ng_ues: id 11 only, the largest number of UEs in a slice (scratch of the 300-sample search). */
/* min_sort_n: id 10 sorts its slices' G entries on up to five warps at a time next to the parked grants: it needs
 * the slot arrays at least max(16 G, 1024) entries long whatever S is (rs_sched.cu). */
/* den_in_cnt: the metric denominators (written in P0, last read by the per-slice argmax) share the bytes of the sort's
 * counters (first written by the sort) -- every id but 10, whose EESM sums reuse `den` while its warp sorts count
 * (den_shares_cnt below).  The 800 B are what lets a tenth headline cell (one CQI byte per RBG) fit an SM. */
__host__ __device__ constexpr inline bool den_shares_cnt(int algo) { return algo != 10; }
__host__ __device__ constexpr inline Layout make_layout(int S, int U, int G, int m_cap, int cq_bytes = 0, int ng_ues = 0,
                                                        int min_sort_n = 0, int nb = 1, bool den_in_cnt = false) {
  Layout L{};
  const int n = (S * G > min_sort_n) ? S * G : min_sort_n;
  const int nw = (n + 31) / 32;
  int o = 0;
  L.avg = o;  o += 8 * U * nb;
  const bool share_den = den_in_cnt && 8 * U <= 2 * 16 * nw;
  L.den = o;  o += share_den ? 0 : 8 * U;
  L.off = o;  o += 8 * S;
  L.tval = o; o += 8 * 16;
  L.posl = o; o += 2 * n;
  L.posr = o; o += 2 * n;
  o = rs_align(o, 8);
  if (8 * kMStride * m_cap <= 4 * n) {
    L.mtab = L.posl;
  } else {
    L.mtab = o; o += 8 * kMStride * m_cap;
  }
  L.tx = o;   o += 4 * U * nb;
  L.utr = o;  o += 4 * U;
  L.mask = o; o += 8 * U;
  L.seg0 = o; o += 4 * (n / 16 + 2);
  L.seg1 = o; o += 4 * (n / 16 + 2);
  L.target = o; o += 4 * S;
  L.quota = o;  o += 4 * S;
  L.frb = o;    o += 4 * S;
  L.wd = o;     o += 4 * S;
  L.misc = o;   o += 4 * 48;
  L.a = o;    o += 2 * n;
  L.win = o;  o += 2 * n;
  o = rs_align(o, 8);
  L.cnt = o;  o += 2 * 16 * nw;
  if (share_den) L.den = L.cnt;
  L.outsl = o; o += G;
  L.sptr = rs_align(o, 4); o = L.sptr + 4 * (S + 1);
  L.sues = o; o += 2 * U;
  L.cq = rs_align(o, 16); o = L.cq + cq_bytes;
  L.mbar = rs_align(o, 8); o = L.mbar + 8;   /* mbarrier of the bulk copy that stages the CQI */
  L.ng_red = rs_align(o, 8); o = L.ng_red + (ng_ues ? 16 * (RS_THREADS / 32) : 0);
  L.ng_list = o; o += 2 * ng_ues;
  L.ng_hc = o;   o += ng_ues;
  L.ng_mcs = rs_align(o, 4); o = L.ng_mcs + ng_ues * RS_THREADS;
  L.done = o;    o += U;
  L.total = rs_align(o, 16);
  return L;
}

/* ---- shape policies of the TTI kernel ------------------------------------------------------------
 * DynShape: every dimension, the shared-memory layout and the slice tables come from DevCfg at run time (any cell).
 * FixedShape: a cell of S slices x UPS UEs each (UE u in slice u / UPS), G RBGs of RBG RBs, CQI layout LAY, one
 * bearer per UE, staged CQI -- known when the kernel is compiled, so shared-memory addresses are immediates, the
 * slice tables are arithmetic, divisions are shifts / multiplies and the short loops unroll.  The host picks a
 * FixedShape instantiation when a handle's configuration AND its host-computed layout match it bit for bit
 * (rs_sched.cu fixed_kernel_for), otherwise the DynShape kernel runs; results are identical either way
 * (tests/test_gpu_parity.py::test_fixed_shape_equals_dynamic). */
struct DynShape {
  static constexpr bool kStatic = false;
};
/* UEs one chunk of the per-slice metric table holds: at least the largest slice; otherwise as many as still fit the
 * bytes of the sort's slot arrays, which the table borrows (make_layout: 8 * 16 * cap <= 4 * n), and at least 32.  The
 * headline cell: 40 UEs = 8 slices per chunk, 128 (slice, RBG quad) items per chunk for 128 threads, three chunks. */
__host__ __device__ constexpr inline int metric_table_cap(int max_slice, int U, int sort_n) {
  const int fit = sort_n / 32 > 32 ? sort_n / 32 : 32;
  const int want = U < fit ? U : fit;
  return max_slice > want ? max_slice : want;
}
template <int S_, int UPS_, int G_, int RBG_, int LAY_>
struct FixedShape {
  static constexpr bool kStatic = true;
  static constexpr int S = S_, UPS = UPS_, U = S_ * UPS_, G = G_, RBG = RBG_, R = G_ * RBG_, LAY = LAY_;
  static constexpr int kCqiRow = LAY_ == 1 ? R : (LAY_ == 2 ? G_ / 2 : G_);
  /* metric-table chunks as rs_create packs them: consecutive slices while their UEs fit metric_table_cap() */
  static constexpr int kCap = metric_table_cap(UPS_, U, S_ * G_);
  static constexpr int kSlicesPerChunk = kCap / UPS_;
  static constexpr int kChunks = (S_ + kSlicesPerChunk - 1) / kSlicesPerChunk;
  static constexpr int kMCap = (S_ < kSlicesPerChunk ? S_ : kSlicesPerChunk) * UPS_;
  static constexpr int kSortN = G_ * S_;
  __host__ __device__ static constexpr int log2_floor(int v) { int lg = 0; while (v > 1) { v >>= 1; ++lg; } return lg; }
  static constexpr int kSortDepth = 2 * log2_floor(kSortN);
  /* NVS (ids 7, 11) tabulates the served slice only: one "chunk" of UPS UEs, plus the scratch of the served slice's users */
  __host__ __device__ static constexpr bool nvs(int algo) { return algo == 7 || algo == 11; }
  __host__ __device__ static constexpr int chunks(int algo) { return nvs(algo) ? 1 : kChunks; }
  __host__ __device__ static constexpr int mcap(int algo) { return nvs(algo) ? UPS_ : kMCap; }
  __host__ __device__ static constexpr Layout layout(int algo) {
    return make_layout(S_, U, G_, mcap(algo), U * kCqiRow, nvs(algo) ? UPS_ : 0, 0, 1, den_shares_cnt(algo));
  }
};

/* ================================================================================================
 * libstdc++ std::sort (introsort) order of n entries, key = bits 12..15 (descending), payload =
 * bits 0..11, evaluated level by level over all ranges of one recursion depth at once
 * (tests/sort_model.py is the executable statement of this formulation).
 * ============================================================================================== */
__device__ __forceinline__ bool before(unsigned short x, unsigned short y) { return (x >> 12) > (y >> 12); }

/* std::__partial_sort(first,last,last): __make_heap + __sort_heap (bits/stl_heap.h), comp = before.
 * Sequential; reached only when the depth limit runs out (never seen on real inputs). */
static __device__ void heap_adjust(unsigned short* f, int hole, int len, unsigned short v) {
  const int top = hole;
  int child = hole;
  while (child < (len - 1) / 2) {
    child = 2 * (child + 1);
    if (before(f[child], f[child - 1])) child--;
    f[hole] = f[child];
    hole = child;
  }
  if ((len & 1) == 0 && child == (len - 2) / 2) {
    child = 2 * (child + 1);
    f[hole] = f[child - 1];
    hole = child - 1;
  }
  int parent = (hole - 1) / 2;
  while (hole > top && before(f[parent], v)) {
    f[hole] = f[parent];
    hole = parent;
    parent = (hole - 1) / 2;
  }
  f[hole] = v;
}
static __device__ void heap_sort(unsigned short* f, int len) {
  if (len >= 2) {
    int parent = (len - 2) / 2;
    while (true) {
      heap_adjust(f, parent, len, f[parent]);
      if (parent == 0) break;
      parent--;
    }
  }
  int last = len;
  while (last > 1) {
    --last;
    unsigned short v = f[last];
    f[last] = f[0];
    heap_adjust(f, 0, last, v);
  }
}

/* std::__move_median_to_first(first, first+1, mid, last-1), bits/stl_algo.h:1893-1899 (g++ 13) */
__device__ __forceinline__ void median_to_first(unsigned short* a, int first, int last) {
  const int pa = first + 1, pb = first + (last - first) / 2, pc = last - 1;
  const unsigned short xa = a[pa], xb = a[pb], xc = a[pc];
  int pick;
  if (before(xa, xb)) pick = before(xb, xc) ? pb : (before(xa, xc) ? pc : pa);
  else if (before(xa, xc)) pick = pa;
  else if (before(xb, xc)) pick = pc;
  else pick = pb;
  const unsigned short t = a[first];
  a[first] = a[pick];
  a[pick] = t;
}

/* atomicAdd on shared memory as ONE instruction: around a one-lane atomicAdd the compiler builds its warp aggregation
 * (vote, popc, leader election) for nothing. */
__device__ __forceinline__ unsigned smem_add(unsigned* p, unsigned v) {
  unsigned old;
  asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"((unsigned)__cvta_generic_to_shared(p)), "r"(v) : "memory");
  return old;
}

struct SortBufs {
  unsigned short* a;     /* [n] in: entries in insertion order; scratch afterwards */
  unsigned short* out;   /* [n] result, sorted (== posr) */
  unsigned short* posl;  /* [n] */
  unsigned short* posr;  /* [n] */
  unsigned* seg0;        /* [n/16+2] ranges still to partition, ping */
  unsigned* seg1;        /* [n/16+2] pong */
  unsigned short* cnt;   /* [16*nw] */
  unsigned* misc;        /* [48]: 0 the cell's slice profile, 8..10 rotating list counters, 13..15 per-TTI scalars of the
                            kernel, 16.. warp totals */
  const unsigned short* eq_tab;  /* all-equal-keys permutations, see eq_offset(); may be null */
  int eq_max;            /* longest range the table covers */
};

/* Offset of the permutation for a range of `len` equal keys (len = 17..eq_max) in eq_tab. */
__host__ __device__ inline size_t eq_offset(int len) { return (size_t)(len - 1) * len / 2 - 136; }

/* One warp partitions the range [f,l) exactly like std::__unguarded_partition_pivot and returns
 * the cut.  Stoppers of the left scan (key <= pivot) and of the right scan (key >= pivot) are
 * listed in slots of the range itself; pair k = (k-th from the left, k-th from the right) is
 * swapped while the former lies left of the latter. */
__device__ __forceinline__ int warp_partition(const SortBufs& b, int f, int l, int lane, int levels_left) {
  unsigned short* a = b.a;
  if (lane == 0) median_to_first(a, f, l);
  __syncwarp();
  const int p = a[f] >> 12;
  const int m = l - f - 1, base = f + 1;
  const unsigned lt = (1u << lane) - 1u;
  int nl = 0, nr = 0;
  /* four chunks per trip while the range is long (the four loads are independent, so their
   * latencies overlap), then one chunk at a time */
  int c0 = 0;
  for (; c0 + 96 < m; c0 += 128) {
    int k[4];
    bool v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int idx = c0 + 32 * q + lane;
      v[q] = idx < m;
      k[q] = v[q] ? (a[base + idx] >> 12) : 0;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int idx = c0 + 32 * q + lane;
      const bool fl = v[q] && k[q] <= p, fr = v[q] && k[q] >= p;
      const unsigned bl = __ballot_sync(kFull, fl), br = __ballot_sync(kFull, fr);
      if (fl) b.posl[base + nl + __popc(bl & lt)] = (unsigned short)(base + idx);
      if (fr) b.posr[base + nr + __popc(br & lt)] = (unsigned short)(base + idx);
      nl += __popc(bl);
      nr += __popc(br);
    }
  }
  for (; c0 < m; c0 += 32) {
    const int idx = c0 + lane;
    const bool valid = idx < m;
    const int k = valid ? (a[base + idx] >> 12) : 0;
    const bool fl = valid && k <= p, fr = valid && k >= p;
    const unsigned bl = __ballot_sync(kFull, fl), br = __ballot_sync(kFull, fr);
    if (fl) b.posl[base + nl + __popc(bl & lt)] = (unsigned short)(base + idx);
    if (fr) b.posr[base + nr + __popc(br & lt)] = (unsigned short)(base + idx);
    nl += __popc(bl);
    nr += __popc(br);
  }
  __syncwarp();
  /* Every key equals the pivot: from here on no comparison depends on the data, so what the rest of
   * the recursion does to this range is a fixed permutation of its length (built on the host by
   * running the same loop, rs_sched.cu build_eq_table).  Apply it in one gather. */
  if (nl == m && nr == m && l - f <= b.eq_max && 32 - __clz(l - f) <= levels_left) {
    const int len = l - f;
    const unsigned short* tab = b.eq_tab + eq_offset(len);
    if (len <= 64) {   /* two entries per lane: permute through registers */
      const bool h0 = lane < len, h1 = lane + 32 < len;
      const unsigned short v0 = h0 ? a[f + tab[lane]] : (unsigned short)0;
      const unsigned short v1 = h1 ? a[f + tab[lane + 32]] : (unsigned short)0;
      __syncwarp();
      if (h0) a[f + lane] = v0;
      if (h1) a[f + lane + 32] = v1;
    } else {
      for (int i = lane; i < len; i += 32) b.posl[f + i] = a[f + i];
      __syncwarp();
      for (int i = lane; i < len; i += 32) a[f + i] = b.posl[f + tab[i]];
    }
    __syncwarp();
    return -1;
  }
  /* k-th right stopper counted from the right = posr[base + nr - 1 - k] */
  const int nmin = min(nl, nr);
  int K = 0;
  for (int c0 = 0;; c0 += 64) {   /* two chunks per trip; pairs stop swapping at one k and never resume */
    bool sw[2];
    int lp[2], rp[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int k = c0 + 32 * q + lane;
      sw[q] = false;
      lp[q] = 0;
      rp[q] = 0;
      if (k < nmin) {
        lp[q] = b.posl[base + k];
        rp[q] = b.posr[base + nr - 1 - k];
        sw[q] = lp[q] < rp[q];
      }
    }
    unsigned short t0[2], t1[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      t0[q] = a[lp[q]];
      t1[q] = a[rp[q]];
    }
#pragma unroll
    for (int q = 0; q < 2; ++q)
      if (sw[q]) {
        a[lp[q]] = t1[q];
        a[rp[q]] = t0[q];
      }
    const unsigned bs0 = __ballot_sync(kFull, sw[0]), bs1 = __ballot_sync(kFull, sw[1]);
    if (bs0 != kFull) { K = c0 + __ffs(~bs0) - 1; break; }
    if (bs1 != kFull) { K = c0 + 32 + __ffs(~bs1) - 1; break; }
  }
  int cut = (K < nl) ? (int)b.posl[base + K] : 0x7fffffff;
  if (K >= 1) cut = min(cut, (int)b.posr[base + nr - K]);
  __syncwarp();
  return cut;
}

#ifdef RS_SORT_TIMING   /* tools/sort_prof.cu: clock64() per level, thread 0 of CTA 0 (each tick is a global read-modify-write:
                           compare builds, not absolute cycles) */
static __device__ long long g_sort_prof[64];
#define RS_STICK(slot) do { if (tid == 0 && blockIdx.x == 0) { const long long now_ = clock64(); g_sort_prof[slot] += now_ - slast_; slast_ = now_; } } while (0)
#else
#define RS_STICK(slot) do {} while (0)
#endif
/* All kThreads threads of the CTA call this. On return b.out[0..n) holds the entries in the order
 * std::sort leaves them.  Ranges of one recursion depth are independent, so each level hands the
 * ranges longer than _S_threshold to the warps, one range per warp at a time. */
/* `rot` rotates which warp takes which range: warp w of every CTA sits on SM sub-partition w % 4, so
 * without it the single-range levels of all resident cells would pile up on one scheduler. */
__device__ __forceinline__ void sort_desc(const SortBufs& b, int n, int depth_limit, int rot) {
  const int tid = threadIdx.x, lane = tid & 31, warp = ((tid >> 5) + rot) % kWarps;
  const int nw = (n + 31) >> 5;
#ifdef RS_SORT_TIMING
  long long slast_ = clock64();
#endif
  if (tid == 0) {
    b.seg0[0] = (unsigned)n << 16;
    b.misc[8] = (n > kSortThreshold) ? 1u : 0u;
    b.misc[9] = 0;
    b.misc[10] = 0;
  }
  __syncthreads();
  RS_STICK(0);
  int c_cur = 8, c_nxt = 9, c_old = 10;   /* misc[8..10]: range counters of this level, the next, the one after (rotating) */
  for (int level = 0;; ++level) {
    unsigned* cur = (level & 1) ? b.seg1 : b.seg0;
    unsigned* nxt = (level & 1) ? b.seg0 : b.seg1;
    const int nseg = (int)b.misc[c_cur];
    if (nseg == 0) break;
    if (level >= depth_limit) {      /* __introsort_loop's depth_limit == 0: heap sort what is left */
      for (int s = tid; s < nseg; s += kThreads) {
        const unsigned sg = cur[s];
        heap_sort(b.a + (sg & 0xffff), (int)(sg >> 16) - (int)(sg & 0xffff));
      }
      break;
    }
    if (tid == 0) b.misc[c_old] = 0;   /* last read before the previous barrier; next used after this one */
    for (int s = warp; s < nseg; s += kWarps) {
      const unsigned sg = cur[s];
      const int f = sg & 0xffff, l = sg >> 16;
      const int cut = warp_partition(b, f, l, lane, depth_limit - level);
      if (lane == 0 && cut >= 0) {   /* one slot request for both parts */
        const int nl_ = cut - f > kSortThreshold, nr_ = l - cut > kSortThreshold;
        if (nl_ + nr_) {
          unsigned at = smem_add(&b.misc[c_nxt], (unsigned)(nl_ + nr_));
          if (nl_) nxt[at++] = (unsigned)f | ((unsigned)cut << 16);
          if (nr_) nxt[at] = (unsigned)cut | ((unsigned)l << 16);
        }
      }
    }
    RS_STICK(1 + 4 * (level < 12 ? level : 12));
    __syncthreads();
    RS_STICK(4 + 4 * (level < 12 ? level : 12));
    { const int t = c_cur; c_cur = c_nxt; c_nxt = c_old; c_old = t; }
  }
  __syncthreads();
  RS_STICK(60);

  /* __final_insertion_sort == stable sort by key of what is in a[] now: counting sort, 16 keys */
  for (int q = tid; q < 16 * nw; q += kThreads) b.cnt[q] = 0;
  __syncthreads();
  for (int w = warp; w < nw; w += kWarps) {
    const int i = w * 32 + lane;
    const bool valid = i < n;
    const int k = valid ? (b.a[i] >> 12) : 16;
    const unsigned m = __match_any_sync(kFull, k);
    const int rk = __popc(m & ((1u << lane) - 1u));
    if (valid) {
      b.posl[i] = (unsigned short)rk;
      if (rk == 0) b.cnt[(15 - k) * nw + w] = (unsigned short)__popc(m);
    }
  }
  __syncthreads();
  { /* exclusive scan of cnt[0..16*nw) in place */
    const int Q = 16 * nw;
    const int per = (Q + kThreads - 1) / kThreads;
    const int q0 = tid * per;
    int s = 0;
    for (int q = q0; q < q0 + per && q < Q; ++q) s += (int)b.cnt[q];
    int incl = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(kFull, incl, d);
      if (lane >= d) incl += v;
    }
    const int pw = tid >> 5;   /* physical warp: the scan runs over threads in tid order */
    if (lane == 31) b.misc[16 + pw] = (unsigned)incl;
    __syncthreads();
    int base = incl - s;
    for (int w = 0; w < pw; ++w) base += (int)b.misc[16 + w];
    for (int q = q0; q < q0 + per && q < Q; ++q) {
      const int c = (int)b.cnt[q];
      b.cnt[q] = (unsigned short)base;
      base += c;
    }
  }
  __syncthreads();
  for (int w = warp; w < nw; w += kWarps) {
    const int i = w * 32 + lane;
    if (i < n) {
      const unsigned short e = b.a[i];
      b.out[b.cnt[(15 - (e >> 12)) * nw + w] + b.posl[i]] = e;
    }
  }
  __syncthreads();
  RS_STICK(61);
}

/* The same sort by ONE warp on private buffers, for short arrays (n <= 64: UpperBound sorts one slice's G entries,
 * several slices at a time on different warps).  Ranges are taken depth first from a small stack -- the order in
 * which disjoint ranges are partitioned does not change the result, only a range's depth matters (the heap-sort
 * fallback at the depth limit).  stack: >= 16 entries of this warp; b.cnt: >= 32 entries; b.out = b.posr. */
__device__ __forceinline__ void warp_sort_desc(const SortBufs& b, unsigned* stack, int n, int depth_limit, int lane) {
  int sp = 0;
  if (n > kSortThreshold) {
    if (lane == 0) stack[0] = (unsigned)n << 12;   /* f | l << 12 | depth << 24 */
    sp = 1;
  }
  __syncwarp();
  while (sp > 0) {
    const unsigned e = stack[--sp];
    const int f = e & 0xfff, l = (e >> 12) & 0xfff, depth = (int)(e >> 24);
    __syncwarp();
    if (depth >= depth_limit) {
      if (lane == 0) heap_sort(b.a + f, l - f);
      __syncwarp();
      continue;
    }
    const int cut = warp_partition(b, f, l, lane, depth_limit - depth);
    if (cut >= 0) {
      if (l - cut > kSortThreshold) {
        if (lane == 0) stack[sp] = (unsigned)cut | ((unsigned)l << 12) | ((unsigned)(depth + 1) << 24);
        sp++;
      }
      if (cut - f > kSortThreshold) {
        if (lane == 0) stack[sp] = (unsigned)f | ((unsigned)cut << 12) | ((unsigned)(depth + 1) << 24);
        sp++;
      }
    }
    __syncwarp();
  }
  /* __final_insertion_sort == stable counting sort on the 4-bit key, two 32-entry chunks at most */
  const int nw = (n + 31) >> 5;
  b.cnt[lane] = 0;
  __syncwarp();
  for (int w = 0; w < nw; ++w) {
    const int i = w * 32 + lane;
    const bool valid = i < n;
    const int k = valid ? (b.a[i] >> 12) : 16;
    const unsigned mm = __match_any_sync(kFull, k);
    const int rk = __popc(mm & ((1u << lane) - 1u));
    if (valid) {
      b.posl[i] = (unsigned short)rk;
      if (rk == 0) b.cnt[(15 - k) * nw + w] = (unsigned short)__popc(mm);
    }
  }
  __syncwarp();
  {
    const int mine = lane < 16 * nw ? (int)b.cnt[lane] : 0;   /* 16 * nw <= 32 counters: one per lane */
    int incl = mine;
#pragma unroll
    for (int dd = 1; dd < 32; dd <<= 1) {
      const int v = __shfl_up_sync(kFull, incl, dd);
      if (lane >= dd) incl += v;
    }
    __syncwarp();
    b.cnt[lane] = (unsigned short)(incl - mine);
  }
  __syncwarp();
  for (int w = 0; w < nw; ++w) {
    const int i = w * 32 + lane;
    if (i < n) {
      const unsigned short e = b.a[i];
      b.out[b.cnt[(15 - (e >> 12)) * nw + w] + b.posl[i]] = e;
    }
  }
  __syncwarp();
}

/* ================================================================================================
 * helpers shared by the four schedulers
 * ============================================================================================== */

/* RadioBearer::UpdateAverageTransmissionRate, flows/radio-bearer.cpp:138-164 */
__device__ __forceinline__ double ewma_update(double avg, int tx_bytes, double dt) {
  const double rate = __ddiv_rn((double)(tx_bytes * 8), dt);
  const double beta = 0.02;
  double v = __dadd_rn(__dmul_rn(1 - beta, avg), __dmul_rn(beta, rate));
  if (v < 1) v = 1;
  return v;
}

/* AMCModule::GetCQIFromSinr(GetEesmEffectiveSinr(...)), AMCModule.cpp:252-261 on the EESM mean:
 * SINRForCQIIndex[k] <= 10*log10(-log(mean))  <=>  mean <= cut[k] (host bisection against glibc). */
__device__ __forceinline__ int cqi_from_mean(double mean) {
  /* cut[] decreases with k, so the conditions are nested and the reference's loop is a count */
  int cqi = 1;
#pragma unroll
  for (int k = 1; k <= 14; ++k) cqi += (mean <= c_tab.cut[k]) ? 1 : 0;
  return cqi;
}

struct Cell {
  /* shared-memory views */
  double* avg; double* den; double* mtab; double* off;
  unsigned long long* cumb; unsigned long long* cumr;   /* this cell's rows of the HBM counters */
  double* tval; int* tx; int* utr; int* sptr; unsigned short* sues; uint8_t* cq; unsigned* mask; int* target; int* quota; int* frb; int* wd;
  unsigned short* win; unsigned char* outsl; unsigned* misc;
  unsigned short* ng_list; unsigned char* ng_hc; unsigned char* ng_mcs; unsigned char* ng_red; unsigned char* done;
  unsigned long long* mbar;
  SortBufs sb;
};

__device__ __forceinline__ Cell carve(unsigned char* smem, const Layout& L) {
  Cell c;
  c.avg = (double*)(smem + L.avg);
  c.den = (double*)(smem + L.den);
  c.mtab = (double*)(smem + L.mtab);
  c.cumb = nullptr;
  c.cumr = nullptr;
  c.off = (double*)(smem + L.off);
  c.tval = (double*)(smem + L.tval);
  c.tx = (int*)(smem + L.tx);
  c.utr = (int*)(smem + L.utr);
  c.sptr = (int*)(smem + L.sptr);
  c.sues = (unsigned short*)(smem + L.sues);
  c.cq = smem + L.cq;
  c.mbar = (unsigned long long*)(smem + L.mbar);
  c.ng_list = (unsigned short*)(smem + L.ng_list);
  c.ng_hc = smem + L.ng_hc;
  c.ng_mcs = smem + L.ng_mcs;
  c.ng_red = smem + L.ng_red;
  c.done = smem + L.done;
  c.mask = (unsigned*)(smem + L.mask);
  c.target = (int*)(smem + L.target);
  c.quota = (int*)(smem + L.quota);
  c.frb = (int*)(smem + L.frb);
  c.wd = (int*)(smem + L.wd);
  c.win = (unsigned short*)(smem + L.win);
  c.outsl = (unsigned char*)(smem + L.outsl);
  c.misc = (unsigned*)(smem + L.misc);
  c.sb.a = (unsigned short*)(smem + L.a);
  c.sb.out = (unsigned short*)(smem + L.posr);
  c.sb.seg0 = (unsigned*)(smem + L.seg0);
  c.sb.seg1 = (unsigned*)(smem + L.seg1);
  c.sb.posl = (unsigned short*)(smem + L.posl);
  c.sb.posr = (unsigned short*)(smem + L.posr);
  c.sb.cnt = (unsigned short*)(smem + L.cnt);
  c.sb.misc = c.misc;
  c.sb.eq_tab = nullptr;
  c.sb.eq_max = 0;
  return c;
}

#ifdef RS_NO_BULK
/* Ampere-style asynchronous 16-byte copy global -> shared (LDGSTS); both addresses 16-byte aligned */
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
#else
/* Bulk asynchronous copy global -> shared through the TMA unit (cp.async.bulk, SASS UBLKCP): one instruction moves
 * a whole contiguous block (the cell's CQI slab, 3.2-6.4 KB at the headline shape) and reports the bytes landed to
 * an mbarrier in shared memory; the consumers sleep on the barrier's phase instead of a wait_group + CTA barrier.
 * Addresses and size are multiples of 16. */
__device__ __forceinline__ void mbar_init(void* mbar, unsigned count) {
  const unsigned ma = (unsigned)__cvta_generic_to_shared(mbar);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ma), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void* mbar, unsigned bytes) {
  const unsigned ma = (unsigned)__cvta_generic_to_shared(mbar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ma), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, unsigned bytes, void* mbar) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst), ma = (unsigned)__cvta_generic_to_shared(mbar);
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(sa), "l"(gsrc), "r"(bytes), "r"(ma) : "memory");
}
__device__ __forceinline__ void mbar_wait(void* mbar, unsigned parity) {
  const unsigned ma = (unsigned)__cvta_generic_to_shared(mbar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "RS_MBAR_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra RS_MBAR_DONE;\n"
      "bra RS_MBAR_WAIT;\n"
      "RS_MBAR_DONE:\n"
      "}\n" ::"r"(ma), "r"(parity) : "memory");
}
#endif

/* Where UE u's CQI vector of this TTI starts: row u of the [U][cqi_row] slab, or (trace mode) the
 * current row of the trace the UE replays (cqi then points at that row of trace 0). */
template <bool TRACE>
__device__ __forceinline__ const uint8_t* ue_cqi(const DevCfg& d, const Dims& dm, const Cell& c, const uint8_t* cqi, int u) {
  return TRACE ? cqi + c.utr[u] : cqi + (size_t)u * dm.cqi_row;
}
/* CQI on the first RB of RBG g (the RB the metric is evaluated on, transport.cpp:536); p = ue_cqi() */
__device__ __forceinline__ int cqi_first_rb(const Dims& dm, const uint8_t* p, int g) {
  if (dm.cqi_per_rb == 2) return (p[g >> 1] >> (4 * (g & 1))) & 15;
  return dm.cqi_per_rb ? (p[(size_t)g * dm.rbg] & 15) : (p[g] & 15);
}

/* First entry of the cell's slice profile in a table of n entries per profile.  The profile sits in shared memory
 * (misc[0], written at cell start) rather than in a register that would stay live across the whole kernel. */
__device__ __forceinline__ int prof_row(const DevCfg& d, const Cell& c, int n) {
  return d.cell_profile ? (int)c.misc[0] * n : 0;   /* one profile (null): row 0 without the load */
}

/* Slice targets and RBG quotas, transport.cpp:463-521, by one warp (lane s and lane s+32). */
__device__ __forceinline__ void slice_quotas(const DevCfg& d, const Dims& dm, const Cell& c, int r0, int r1, int lane, int* g_target, int* g_quota) {
  const int S = dm.S;
  const int nb_rbs = dm.G * dm.rbg;
  const double* weight = d.weight + prof_row(d, c, S);
  int tgt[2], wd[2];
  int sum = 0, nonempty = 0;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int s = lane + 32 * h;
    tgt[h] = 0;
    wd[h] = 0;
    if (s < S) {
      wd[h] = c.wd[s] & 1;   /* bit 8: the slice's bearer priority of this TTI */
      if (wd[h]) tgt[h] = (int)__dadd_rn(__dmul_rn((double)nb_rbs, weight[s]), c.off[s]);   /* :475 */
    }
    sum += tgt[h];
    nonempty += wd[h];
  }
  sum = __reduce_add_sync(kFull, sum);
  nonempty = __reduce_add_sync(kFull, nonempty);
  if (lane == 0) c.misc[14] = (unsigned)nonempty;
  if (nonempty == 0) return;   /* RBsAllocation only runs with >= 1 user (transport.cpp:152-168) */
  int extra = nb_rbs - sum;
  /* first non-empty slice in rotation order k = (i + rand) % S, i = 0..S-1   (:489-500) */
  const int b0 = r0 % S;
  int rot[2];
  unsigned best = 0xffffffffu;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int s = lane + 32 * h;
    rot[h] = (s - b0 + S) % S;
    if (s < S && wd[h]) best = min(best, (unsigned)rot[h]);
  }
  best = __reduce_min_sync(kFull, best);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int s = lane + 32 * h;
    if (s < S && wd[h]) {
      tgt[h] += extra / nonempty;
      if ((unsigned)rot[h] == best) tgt[h] += extra % nonempty;
    }
  }
  /* quotas (:501-521) */
  int q[2];
  int qsum = 0;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int s = lane + 32 * h;
    q[h] = (s < S) ? tgt[h] / dm.rbg : 0;
    qsum += q[h];
  }
  qsum = __reduce_add_sync(kFull, qsum);
  const int extra_rbgs = dm.G - qsum;
  const int b1 = r1 % S;
  best = 0xffffffffu;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int s = lane + 32 * h;
    rot[h] = (s - b1 + S) % S;
    if (s < S && wd[h]) best = min(best, (unsigned)rot[h]);
  }
  best = __reduce_min_sync(kFull, best);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int s = lane + 32 * h;
    if (s < S) {
      if (wd[h]) {
        q[h] += extra_rbgs / nonempty;
        if ((unsigned)rot[h] == best) q[h] += extra_rbgs % nonempty;
      }
      c.target[s] = tgt[h];
      c.quota[s] = q[h];
      if (g_target) g_target[s] = tgt[h];
      if (g_quota) g_quota[s] = q[h];
    }
  }
}

/* MaximizeCell's first-fit scan over the sorted (rbg,slice) entries, transport.cpp:362-375, by one
 * warp, 32 entries at a time.  Remaining quotas (c.quota) and the RBG->slice map (c.outsl, 0xff =
 * free) live in shared memory between chunks; inside a chunk every lane keeps the remaining quota
 * of its own entry's slice in a register, one redux.sync(min) finds the lowest feasible lane and
 * broadcasts its (rbg,slice), and the other lanes drop out if they lost their RBG or their slice
 * ran out.  c.quota is consumed (the host-visible quotas were written by slice_quotas). */
__device__ __forceinline__ void greedy_maxcell(const DevCfg& d, const Dims& dm, const Cell& c, const unsigned short* sorted, int lane) {
  const int n = dm.sort_n;
  int nfree = dm.G;
  for (int base = 0; base < n && nfree > 0; base += 32) {
    const int i = base + lane;
    const unsigned e = (i < n) ? sorted[i] : 0u;
    const int g = (e >> 6) & 63, s = e & 63;
    int rem = c.quota[s];
    bool feas = (i < n) && c.outsl[g] == 0xff && rem > 0;
    unsigned v = feas ? (((unsigned)lane << 12) | (e & 0xfffu)) : 0xffffffffu;
    unsigned w = __reduce_min_sync(kFull, v);
    while (w != 0xffffffffu) {
      const int pg = (w >> 6) & 63, ps = w & 63, ld = (int)(w >> 12);
      if (s == ps) rem--;
      if (lane == ld) {
        c.outsl[pg] = (unsigned char)ps;
        c.quota[ps] = rem;
      }
      nfree--;
      feas = feas && lane != ld && g != pg && rem > 0;
      if (!feas) v = 0xffffffffu;
      w = __reduce_min_sync(kFull, v);
    }
    __syncwarp();
  }
}

/* GreedyByRow, transport.cpp:249-272, by one warp. a[] holds the unsorted (rbg-major) entries. */
__device__ __forceinline__ void greedy_by_row(const DevCfg& d, const Dims& dm, const Cell& c, const unsigned short* a, int lane) {
  const int S = dm.S;
  int rem_a = (lane < S) ? c.quota[lane] : 0;
  int rem_b = (lane + 32 < S) ? c.quota[lane + 32] : 0;
  for (int g = 0; g < dm.G; ++g) {
    unsigned v = 0;
    if (lane < S && rem_a > 0) v = ((unsigned)(a[g * S + lane] >> 12) << 8 | (unsigned)(63 - lane)) + 1u;
    if (lane + 32 < S && rem_b > 0) {
      const unsigned v2 = ((unsigned)(a[g * S + lane + 32] >> 12) << 8 | (unsigned)(63 - lane - 32)) + 1u;
      v = max(v, v2);
    }
    v = __reduce_max_sync(kFull, v);
    if (v) {
      const int ps = 63 - (int)((v - 1u) & 0xffu);
      if (lane == 0) c.outsl[g] = (unsigned char)ps;
      if (lane == (ps & 31)) { if (ps < 32) rem_a--; else rem_b--; }
    }
  }
}

/* Link adaptation + accounting for UE u holding the RBGs in mask (transport.cpp:632-660 and 170-199;
 * dl-pf-packet-scheduler.cpp:64-96 for id 1). */
__device__ __forceinline__ void finalize_ue(const DevCfg& d, const Dims& dm, const Cell& c, const uint8_t* row, int u,
                                            unsigned m_lo, unsigned m_hi, int* o_bits, uint8_t* o_mcs, uint8_t* o_fc,
                                            int data_u, const double* presum = nullptr, const int* qd2 = nullptr) {
  int bits = 0, mcs = 0xff, fc = 0;
  const int nrbg = __popc(m_lo) + __popc(m_hi);
  if (nrbg > 0) {
    double sum = 0;
    unsigned long long m = ((unsigned long long)m_hi << 32) | m_lo;
    if (presum) {   /* id 10: the RB list is not in RBG order; the caller summed it in list order */
      sum = presum[u];
      m = 0;
    }
    while (m) {
      const int g = __ffsll((long long)m) - 1;
      m &= m - 1;
      if (dm.cqi_per_rb == 1) {
        const uint8_t* p = row + (size_t)g * dm.rbg;
        for (int r = 0; r < dm.rbg; ++r) sum = __dadd_rn(sum, c.tval[p[r] & 15]);
      } else {
        const double t = c.tval[cqi_first_rb(dm, row, g)];
        for (int r = 0; r < dm.rbg; ++r) sum = __dadd_rn(sum, t);
      }
    }
    const int nrb = nrbg * dm.rbg;
    const double mean = __ddiv_rn(sum, (double)nrb);
    fc = cqi_from_mean(mean);
    mcs = 2 * (fc - 1);                        /* MapCQIToMCS, AMCModule.cpp:36-40 */
    bits = d.tbs_n[nrbg * 16 + fc];
    int avail = bits / 8;
    if (avail > 0) {
      if (d.algo == 1) {
        c.tx[u] += avail;
        atomicAdd(&c.cumb[u], (unsigned long long)avail);   /* no value comes back: a fire-and-forget RED instead of a load the TTI would wait for */
        atomicAdd(&c.cumr[u], (unsigned long long)nrb);
      } else if (qd2) {
        /* two bearers: the bearer of the higher priority is served first and what is left goes to the other one;
         * every bearer that sends is booked the user's whole RB count (transport.cpp:179-191, nvs.cpp:229-243) */
        for (int i = 1; i >= 0 && avail > 0; --i) {
          const int data_i = qd2[2 * u + i];
          if (data_i <= 0) continue;
          const int sent = min(avail, data_i);
          avail -= sent;
          c.tx[2 * u + i] += sent;
          atomicAdd(&c.cumb[2 * u + i], (unsigned long long)sent);
          atomicAdd(&c.cumr[2 * u + i], (unsigned long long)nrb);
        }
      } else if (data_u > 0) {
        const int sent = min(avail, data_u);
        c.tx[u] += sent;
        atomicAdd(&c.cumb[u], (unsigned long long)sent);
        atomicAdd(&c.cumr[u], (unsigned long long)nrb);
      }
    }
  }
  if (o_bits) o_bits[u] = bits;
  if (o_mcs) o_mcs[u] = (uint8_t)mcs;
  if (o_fc) o_fc[u] = (uint8_t)fc;
}

/* Per-bearer byte FIFOs (rs_enable_buffers).  m / tm / by: the bearer's metadata and its ring of K records.  Inlined:
 * out of line, the calls made the queue-aware kernels spill up to 72 B around them; inlined they stay within 32 B. */
/* Start of a TTI: the arrival of `a` bytes stamped `at` (tail drop of the whole arrival when K records are held), then
 * the queue size and head-of-line delay the scheduler sees, written to *q / *h. */
static __device__ __forceinline__ void buf_arrive(BufMeta* m, double* tm, int* by, int K, int a, double at, double now, int* q,
                                        double* h) {
  BufMeta x = *m;
  if (x.n < 0) { *q = 100000000; *h = 0.0; return; }   /* backlogged: the reference's infinite buffer */
  if (a > 0) {
    if (x.n == K) {
      m->dropped = x.dropped + (unsigned long long)a;
    } else {
      const int i = x.head + x.n < K ? x.head + x.n : x.head + x.n - K;
      tm[i] = at;
      by[i] = a;
      x.n++;
      x.queued += a;
      m->n = x.n;
      m->queued = x.queued;
    }
  }
  *q = (int)min(x.queued, (long long)0x7fffffff);
  *h = x.n > 0 ? __dsub_rn(now, tm[x.head]) : 0.0;
}
/* End of a TTI: `sent` bytes booked to the bearer leave from the head, clamped to what is queued.  A record sent in
 * part keeps its arrival time. */
static __device__ __forceinline__ void buf_depart(BufMeta* m, int* by, int K, int sent) {
  BufMeta x = *m;
  if (sent <= 0 || x.n <= 0) return;
  long long left = min((long long)sent, x.queued);
  x.queued -= left;
  while (left > 0) {
    const int r = by[x.head];
    if (r > left) { by[x.head] = r - (int)left; break; }
    left -= r;
    x.head = x.head + 1 == K ? 0 : x.head + 1;
    x.n--;
  }
  m->queued = x.queued;
  m->head = x.head;
  m->n = x.n;
}

constexpr int kVogelTab = 16 * 17 + 16 * 17 + 2;   /* id 103: gap ranks [16][17] + acceptance thresholds [ranks + 1], int16 each */
/* Scratch of ids 101 / 103 in the (dead) slot arrays of the sort; inter_scratch_bytes() of it
 * (make_layout's min_sort_n). */
__host__ __device__ inline int inter_scratch_bytes(int G, int S) { return 128 + 20 * (G + S) + 8 * S + S + (S + 1) + 128 + 16 + 2 * kVogelTab; }
struct InterScratch {
  double* eff;             /* [16] AMC efficiency per CQI: lanes index it with different CQIs, which the constant
                              cache would serialise */
  double* val;             /* [G + S] candidate gap / loss */
  int* pick;               /* [G + S] */
  int* k2;                 /* id 103 re-uses val / pick / k2 / todo (20 (G + S) bytes) as six int16 arrays, see vogel_approximate */
  int* todo;
  short* vtab;             /* [kVogelTab] id 103: gap rank of (k1, k2 + 1), then the acceptance threshold of a running maximum */
  int* over;               /* [S] RBGs above quota, 0 = not in the map */
  int* under;              /* [S] RBGs below quota */
  unsigned char* order;    /* [S] the slices below quota in std::unordered_map iteration order */
  unsigned char* nxt;      /* [S + 1] singly linked list of the emulated hashtable, S = before-begin */
  unsigned char* bkt;      /* [128] node before the first node of each bucket, 0xff = empty bucket */
};
__device__ __forceinline__ InterScratch inter_scratch(const DevCfg& d, const Dims& dm, const Cell& c) {
  InterScratch x;
  unsigned char* p = (unsigned char*)c.sb.posl;
  const int n = dm.G + dm.S;
  x.eff = (double*)p;
  p += 128;
  x.val = (double*)p;
  x.pick = (int*)(p + 8 * n);
  x.k2 = x.pick + n;
  x.todo = x.k2 + n;
  x.over = x.todo + n;
  x.under = x.over + dm.S;
  x.order = (unsigned char*)(x.under + dm.S);
  x.nxt = x.order + dm.S;
  x.bkt = x.nxt + dm.S + 1;
  x.vtab = (short*)(((size_t)(x.bkt + 128) + 1) & ~(size_t)1);   /* the 16 spare bytes of inter_scratch_bytes cover the alignment */
  return x;
}
/* efficiency of the (rbg, slice) pair: the slice winner's, 0 for a slice without a listed user */
__device__ __forceinline__ double pair_eff(const Cell& c, const InterScratch& x, int S, int g, int s) {
  return x.eff[c.sb.a[g * S + s] >> 12];
}

/* VogelApproximate, transport.cpp:378-451: up to G rounds; in each, every free RBG (candidate g: a row over the slices
 * with quota left) and every slice with quota left (candidate G + s: a column over the free RBGs) reports the gap
 * between its best and its "second" efficiency exactly as the reference computes them, then the candidates are walked
 * in the reference's order with its int-truncated running maximum, and the last one taken is granted.
 *
 * Lines.  The reference scans a line in order with   if (e1 == -1 || e > e1) { first = k; e1 = e; continue; }
 *                                                    if (e2 == -1 || e > e2) e2 = e;
 * i.e. e1 / first = the first maximum, and e2 = the largest element that was NOT a new strict maximum when it was
 * visited (a displaced maximum is not demoted).  Efficiency is strictly increasing in the CQI, so a line is scanned on
 * its 4-bit CQI keys by one warp, two keys per lane, with redux.max and ballots only: the first maximum is (e1, first);
 * everything behind it is a non-record; in front of it the largest key is a non-record iff it occurs twice, else the
 * search repeats in front of that key (vogel_scan_line).
 *
 * Gaps.  e1 - e2 is one of 16 x 17 doubles (e2 = -1 when there is no second); the host subtracts them and hands down
 * their dense ranks and, for every possible running maximum, the rank of the largest gap not above its truncation
 * (vogel_tab): the walk -- "taken iff gap > (int) largest gap so far", the grant is the last one taken -- is then an
 * integer prefix maximum.
 *
 * Rounds.  Between rounds only two things change: the granted RBG leaves every column, and a slice that reached its
 * quota leaves every row.  Removing element x from a line changes (e1, first, e2) only if key(x) >= key(e2) (or there is
 * no e2): a record below e2 can only promote elements below e2, a non-record below e2 changes nothing.  And a line whose
 * maximum occurs three times or more keeps all three when it loses a maximum other than the first one (e2 IS the maximum
 * then; the candidate carries a count of its maxima).  So a round re-scans just the lines that pass both tests -- with
 * winner CQIs of 12-15 all over a column, the second test is what spares most of them.  One warp walks the candidates and posts the grant (a CTA barrier); every warp keeps
 * the slices' fill and the free-RBG mask in registers, owns the candidates q = warp + kWarps * lane (one packed word each) and re-scans
 * them in place -- the walk lies between the barrier that ends a round and the one that posts the grant, the re-scans
 * between that one and the end of the round.  Result in c.outsl. */
struct VogelBufs {
  unsigned* cand;   /* [n] candidate = gap rank | (grant + 1) << 9 | (CQI key of the second efficiency + 1) << 16 | key of the best
                       << 21 | min(7, how often that key occurs in the line) << 25; grant: the RBG / slice it would grant,
                       0 in that field = candidate out */
  const short* rank_of;   /* [16][17] */
  const short* thr;       /* [ranks + 1], index = running maximum's rank + 1 */
  int n;
};
__device__ __forceinline__ int vogel_pick(unsigned w) { return (int)((w >> 9) & 0x7fu) - 1; }
__device__ __forceinline__ int vogel_k2(unsigned w) { return (int)((w >> 16) & 0x1fu) - 1; }
__device__ __forceinline__ void vogel_scan_line(const Cell& c, const VogelBufs& v, int buf, int S, int G, int q, int lane,
                                                int ha, int qa, int hb, int qb, unsigned long long free_m) {
  const bool is_row = q < G;
  const int n = is_row ? S : G;   /* <= 64: two keys per lane */
  int k1 = -1, first = -1, k2 = -1, n_max = 0;
  bool live;
  if (is_row) live = ((free_m >> q) & 1ull) != 0;
  else {
    const int s = q - G;
    live = __shfl_sync(kFull, s < 32 ? (ha < qa) : (hb < qb), s & 31);
  }
  if (live) {
    int key[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int i = 32 * h + lane;
      bool ok = i < n;
      if (ok) ok = is_row ? (h == 0 ? ha < qa : hb < qb) : (((free_m >> i) & 1ull) != 0);
      key[h] = ok ? (int)((is_row ? c.sb.a[q * S + i] : c.sb.a[i * S + (q - G)]) >> 12) : -1;
    }
    /* e1 / first: the first maximum (the last "record" of the reference's scan) */
    const int M = __reduce_max_sync(kFull, max(key[0], key[1]));
    if (M >= 0) {
      const unsigned b0 = __ballot_sync(kFull, key[0] == M), b1 = __ballot_sync(kFull, key[1] == M);
      const int m = b0 ? __ffs(b0) - 1 : 32 + __ffs(b1) - 1;
      k1 = M;
      first = m;
      n_max = min(__popc(b0) + __popc(b1), 7);
      /* e2 = the largest NON-record.  Everything behind the first maximum is one ... */
      int e2 = __reduce_max_sync(kFull, max(lane > m ? key[0] : -1, 32 + lane > m ? key[1] : -1));
      /* ... and in front of it: M1 = the largest key before `end`; if it occurs twice its second occurrence is a
       * non-record (and nothing in front can be larger); if once, it is a record, everything between it and `end` is a
       * non-record, and the search goes on in front of it.  Keys fall strictly from one trip to the next. */
      int end = m;
      while (true) {
        const int c0 = lane < end ? key[0] : -1, c1 = 32 + lane < end ? key[1] : -1;
        const int M1 = __reduce_max_sync(kFull, max(c0, c1));
        if (M1 <= e2) break;   /* nothing in front of `end` can raise e2 (also: nothing valid there) */
        const unsigned e0 = __ballot_sync(kFull, c0 == M1), e1 = __ballot_sync(kFull, c1 == M1);
        if (__popc(e0) + __popc(e1) >= 2) { e2 = M1; break; }
        const int m1 = e0 ? __ffs(e0) - 1 : 32 + __ffs(e1) - 1;
        e2 = max(e2, __reduce_max_sync(kFull, max((lane > m1 && lane < end) ? key[0] : -1,
                                                   (32 + lane > m1 && 32 + lane < end) ? key[1] : -1)));
        end = m1;
      }
      k2 = e2;
    }
  }
  if (lane == 0)
    v.cand[buf * v.n + q] = (k1 < 0 ? 0u : (unsigned)v.rank_of[k1 * 17 + k2 + 1] | ((unsigned)k1 << 21) | ((unsigned)n_max << 25)) |
                            ((unsigned)(first + 1) << 9) | ((unsigned)(k2 + 1) << 16);
}

static __device__ void vogel_approximate(const DevCfg& d, const Dims& dm, const Cell& c) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, G = dm.G, S = dm.S;
  const InterScratch x = inter_scratch(d, dm, c);
  VogelBufs v;
  v.n = G + S;
  v.cand = (unsigned*)x.val;
  v.rank_of = x.vtab;
  v.thr = x.vtab + 16 * 17;
  for (int i = tid; i < kVogelTab; i += kThreads) x.vtab[i] = d.vogel_tab[i];
  /* every warp's own copy of the state: lane s / s + 32 hold slice s's quota and fill, free_m the RBGs not yet granted */
  const int qa = lane < S ? c.quota[lane] : 0, qb = lane + 32 < S ? c.quota[lane + 32] : 0;
  int ha = 0, hb = 0;
  unsigned long long free_m = G >= 64 ? ~0ull : ((1ull << G) - 1ull);
  __syncthreads();
  for (int q = warp; q < v.n; q += kWarps) vogel_scan_line(c, v, 0, S, G, q, lane, ha, qa, hb, qb, free_m);
  __syncthreads();
  for (int round = 0; round < G; ++round) {
    /* The reference walks the candidates in order and takes candidate q when its gap exceeds max_diff, an int that is
     * set to the (truncated) gap whenever a candidate is taken; the grant is the LAST candidate taken.  max_diff is
     * always the truncated largest gap seen so far, so q is taken iff rank_q > thr[largest rank before q].  Let M be the
     * largest rank and m its first position: thr[x] <= x < M for every x seen before m, so m itself is always taken,
     * and behind m the running maximum is M: the grant is the last q > m with rank_q > thr[M], else m.  No scan.
     * One warp walks and posts the grant; the others wait for it at the barrier. */
    if (warp == 0) {
      int rkq[4], best = -1;
#pragma unroll
      for (int j = 0; j < 4; ++j) {   /* n = G + S <= 128 candidates, four per lane */
        const int q = 32 * j + lane;
        const unsigned w = q < v.n ? v.cand[q] : 0u;
        rkq[j] = (w & 0xfe00u) ? (int)(w & 0x1ffu) : -1;   /* -1: candidate out */
        best = max(best, rkq[j]);
      }
      const int M = __reduce_max_sync(kFull, best);
      int win = -1;
      if (M >= 0) {
        const int T = (int)v.thr[M + 1];
        int m = 0x7fffffff, last = -1;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const unsigned is_max = __ballot_sync(kFull, rkq[j] == M);
          if (is_max && m == 0x7fffffff) m = 32 * j + __ffs(is_max) - 1;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const unsigned over = __ballot_sync(kFull, rkq[j] > T && 32 * j + lane > m);
          if (over) last = 32 * j + 31 - __clz(over);
        }
        win = last >= 0 ? last : m;
      }
      /* the grant travels with the candidate: the candidate's owner may re-scan it while the others still read */
      if (lane == 0) c.misc[13] = win < 0 ? 0xffffffffu : ((unsigned)win | ((unsigned)vogel_pick(v.cand[win]) << 8));
    }
    __syncthreads();
    const unsigned posted = c.misc[13];
    if (posted == 0xffffffffu) break;
    const int win = (int)(posted & 0xffu), pk = (int)(posted >> 8);
    const int gr = win < G ? win : pk, gs = win < G ? pk : win - G;
    if (lane == (gs & 31)) { if (gs < 32) ha++; else hb++; }
    const bool full = __shfl_sync(kFull, gs < 32 ? (ha >= qa) : (hb >= qb), gs & 31);
    free_m &= ~(1ull << gr);
    if (tid == 0) c.outsl[gr] = (unsigned char)gs;
    /* this warp's candidates: carry them over, re-scan the ones the grant can have changed */
    const int qq = warp + kWarps * lane;
    bool redo = false;
    if (qq < v.n) {
      const unsigned w = v.cand[qq];
      if (w & 0xfe00u) {
        /* the line dies, or loses one element x: row qq loses slice gs when that slice is full now, column qq - G loses RBG gr */
        const bool row = qq < G;
        const bool dies = row ? qq == gr : (qq - G == gs && full);
        const bool loses = row ? full : true;
        if (dies) redo = true;
        else if (loses) {
          const int kx = (int)((row ? c.sb.a[qq * S + gs] : c.sb.a[gr * S + (qq - G)]) >> 12);
          if (kx >= vogel_k2(w)) {
            /* x is a maximum behind the first one and at least two maxima stay: first, e1 and e2 (= the maximum) stand;
             * the count is a lower bound (it saturates at 7), so it is simply taken down */
            const int n_max = (int)((w >> 25) & 7u);
            if (kx == (int)((w >> 21) & 15u) && vogel_pick(w) != (row ? gs : gr) && n_max >= 3) v.cand[qq] = w - (1u << 25);
            else redo = true;
          }
        }
      }
    }
    __syncwarp();
    unsigned rm = __ballot_sync(kFull, redo);
    while (rm) {
      const int l = __ffs(rm) - 1;
      rm &= rm - 1;
      vogel_scan_line(c, v, 0, S, G, warp + kWarps * l, lane, ha, qa, hb, qb, free_m);
    }
    __syncthreads();
  }
}

/* SubOpt, transport.cpp:274-349: every RBG to its best slice, then single-RBG moves from slices above their
 * quota to slices below it, each time the move that loses the least efficiency (first in RBG order, then in
 * the iteration order of the reference's std::unordered_map of the slices below quota, which is emulated:
 * libstdc++'s hashtable with its prime bucket counts 13 / 29 / 59 / 127, nodes of an empty bucket go to the
 * front of the list, a rehash re-links the nodes in list order).  Result in c.outsl. */
static __device__ void sub_opt(const DevCfg& d, const Dims& dm, const Cell& c) {
  const int tid = threadIdx.x, G = dm.G, S = dm.S;
  const InterScratch x = inter_scratch(d, dm, c);
  int* held = c.wd;
  for (int s = tid; s < S; s += kThreads) held[s] = 0;
  if (tid < 16) x.eff[tid] = c_tab.eff[tid];
  __syncthreads();
  for (int g = tid; g < G; g += kThreads) {
    double best = -1;
    int pick = 0;
    for (int k = 0; k < S; ++k) {
      const double e = pair_eff(c, x, S, g, k);
      if (e > best) { best = e; pick = k; }
    }
    c.outsl[g] = (unsigned char)pick;
    atomicAdd(&held[pick], 1);
  }
  __syncthreads();
  if (tid == 0) {
    int n_over = 0, n_under = 0, n_bkt = 1, n_elt = 0;
    x.nxt[S] = 0xff;
    x.bkt[0] = 0xff;
    for (int i = 0; i < S; ++i) {
      const int q = max(c.quota[i], 0);
      x.over[i] = 0;
      x.under[i] = 0;
      if (held[i] > q) { x.over[i] = held[i] - q; n_over++; }
      else if (held[i] < q) {
        x.under[i] = q - held[i];
        n_under++;
        /* under[i] = ...: _M_insert_unique_node with the prime rehash policy (max load factor 1) */
        if (n_elt + 1 > (n_bkt == 1 ? 0 : n_bkt)) {
          const int nb = (n_bkt == 1) ? 13 : (n_bkt == 13 ? 29 : (n_bkt == 29 ? 59 : 127));
          for (int b = 0; b < nb; ++b) x.bkt[b] = 0xff;
          int p = x.nxt[S], bbegin = 0;
          x.nxt[S] = 0xff;
          while (p != 0xff) {   /* _M_rehash_aux, unique keys */
            const int nx = x.nxt[p], b = p % nb;
            if (x.bkt[b] == 0xff) {
              x.nxt[p] = x.nxt[S];
              x.nxt[S] = (unsigned char)p;
              x.bkt[b] = (unsigned char)S;
              if (x.nxt[p] != 0xff) x.bkt[bbegin] = (unsigned char)p;
              bbegin = b;
            } else {
              x.nxt[p] = x.nxt[x.bkt[b]];
              x.nxt[x.bkt[b]] = (unsigned char)p;
            }
            p = nx;
          }
          n_bkt = nb;
        }
        const int b = i % n_bkt;   /* _M_insert_bucket_begin */
        if (x.bkt[b] != 0xff) {
          x.nxt[i] = x.nxt[x.bkt[b]];
          x.nxt[x.bkt[b]] = (unsigned char)i;
        } else {
          x.nxt[i] = x.nxt[S];
          x.nxt[S] = (unsigned char)i;
          if (x.nxt[i] != 0xff) x.bkt[x.nxt[i] % n_bkt] = (unsigned char)i;
          x.bkt[b] = (unsigned char)S;
        }
        n_elt++;
      }
    }
    int k = 0;
    for (int p = x.nxt[S]; p != 0xff; p = x.nxt[p]) x.order[k++] = (unsigned char)p;
    c.misc[11] = (unsigned)n_over;
    c.misc[12] = (unsigned)n_under;
  }
  __syncthreads();
  while (c.misc[11] > 0 && c.misc[12] > 0) {
    const int n_under = (int)c.misc[12];
    for (int g = tid; g < G; g += kThreads) {   /* the cheapest move of RBG g, first in map order */
      double least = 1.7976931348623157e308;
      int to = -1;
      const int from = c.outsl[g];
      if (x.over[from] > 0) {
        const double mine = pair_eff(c, x, S, g, from);
        for (int q = 0; q < n_under; ++q) {
          const double loss = __dsub_rn(mine, pair_eff(c, x, S, g, x.order[q]));
          if (loss < least) { least = loss; to = x.order[q]; }
        }
      }
      x.val[g] = least;
      x.pick[g] = to;
    }
    __syncthreads();
    if (tid < 32) {
      /* the first RBG (in RBG order) with the strictly smallest loss: lanes take g = tid, tid + 32, ..., then a
       * butterfly on (loss, rbg) */
      double least = 1.7976931348623157e308;
      int rbg = 0x7fffffff;
      for (int g = tid; g < G; g += 32)
        if (x.pick[g] >= 0 && x.val[g] < least) { least = x.val[g]; rbg = g; }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ol = __shfl_xor_sync(kFull, least, o);
        const int og = __shfl_xor_sync(kFull, rbg, o);
        if (og != 0x7fffffff && (rbg == 0x7fffffff || ol < least || (ol == least && og < rbg))) { least = ol; rbg = og; }
      }
      if (rbg == 0x7fffffff) rbg = -1;
      if (tid != 0) {
        /* lane 0 applies the move */
      } else if (rbg < 0) {
        c.misc[11] = 0;   /* the reference asserts a move exists */
      } else {
        const int from = c.outsl[rbg], to = x.pick[rbg];
        held[from] -= 1;
        held[to] += 1;
        c.outsl[rbg] = (unsigned char)to;
        x.over[from] -= 1;
        x.under[to] -= 1;
        if (x.over[from] <= 0 || held[from] <= 0) { x.over[from] = 0; c.misc[11] -= 1; }
        if (x.under[to] <= 0) {   /* erase keeps the order of the others */
          int w = 0;
          for (int q = 0; q < n_under; ++q)
            if (x.order[q] != to) x.order[w++] = x.order[q];
          c.misc[12] -= 1;
        }
      }
    }
    __syncthreads();
  }
}

/* NVS non-greedy, the 300-sample search (nvs.cpp:436-470) for a served slice of at most NU listed users, one sample per
 * thread at a time.  A sample gives user q the MCS hc_q - rand() % 4 (at least 1); on RBG g the user's metric is
 * mtab[q][mcs_q] if mcs_q <= its CQI there, else 0; the sample's score is the sum over the RBGs, in RBG order, of the
 * largest metric.  "mcs_q <= CQI on g" is bit g of ok[q][mcs_q], and the metric does not depend on g: sort the users by
 * metric (registers, odd-even transposition), give every RBG to the first user in that order whose bit is set, and add
 * the RBGs' values in order -- the same doubles in the same order as the reference adds them (an RBG nobody can use
 * adds 0.0).  The first sample with the largest score wins: this thread's samples come in increasing order. */
template <int NU>
__device__ __forceinline__ void ng_search(const Cell& c, const unsigned* ok, const int* draws, int Ua, int G, int tid,
                                          double& best_pf, int& best_i) {
  for (int i = tid; i < 300; i += kThreads) {
    double M[NU];
    unsigned lo[NU], hi[NU];
#pragma unroll
    for (int q = 0; q < NU; ++q) {
      M[q] = -1.0;
      lo[q] = 0;
      hi[q] = 0;
      if (q < Ua) {
        const int mcs = max((int)c.ng_hc[q] - draws[i * Ua + q] % 4, 1);
        M[q] = c.mtab[q * kMStride + mcs];
        lo[q] = ok[(q * 16 + mcs) * 2];
        hi[q] = ok[(q * 16 + mcs) * 2 + 1];
      }
    }
#pragma unroll
    for (int pass = 0; pass < NU; ++pass)
#pragma unroll
      for (int j = pass & 1; j + 1 < NU; j += 2)
        if (M[j] < M[j + 1]) {
          const double tm = M[j]; M[j] = M[j + 1]; M[j + 1] = tm;
          const unsigned tl = lo[j]; lo[j] = lo[j + 1]; lo[j + 1] = tl;
          const unsigned th = hi[j]; hi[j] = hi[j + 1]; hi[j + 1] = th;
        }
    unsigned seen_lo = 0, seen_hi = 0;
#pragma unroll
    for (int q = 0; q < NU; ++q) {   /* an RBG belongs to the first user (largest metric) that can use it */
      const unsigned l = lo[q] & ~seen_lo, h = hi[q] & ~seen_hi;
      seen_lo |= lo[q];
      seen_hi |= hi[q];
      lo[q] = l;
      hi[q] = h;
    }
    double pf = 0.0;
    unsigned bit = 1u;
    for (int g = 0; g < min(G, 32); ++g, bit <<= 1) {
      double v = 0.0;
#pragma unroll
      for (int q = 0; q < NU; ++q) if (lo[q] & bit) v = M[q];
      pf = __dadd_rn(pf, v);
    }
    bit = 1u;
    for (int g = 32; g < G; ++g, bit <<= 1) {
      double v = 0.0;
#pragma unroll
      for (int q = 0; q < NU; ++q) if (hi[q] & bit) v = M[q];
      pf = __dadd_rn(pf, v);
    }
    if (best_pf < pf) { best_pf = pf; best_i = i; }
  }
}

/* ================================================================================================
 * The TTI kernel: grid = cells, block = kThreads, T TTIs per launch with the cell state on chip.
 * ============================================================================================== */
/* Cells per SM the kernel is compiled for, i.e. its register cap (65536 / kThreads / cells).  The compile-time-shape
 * instantiations of Sequential (8) and of SubOpt / VogelApproximate with streamed CQI (101, 103) fit 48 registers without
 * spilling, so ten of their cells fit an SM (shared memory: 19.8 KB per cell with the packed CQI layout, 22.2 KB with one
 * byte per RBG now that the metric denominators share the sort counters' bytes -- make_layout).  Measured with the packed
 * layout (cell-TTIs/s): id 8 65.2 -> 70.2 M, id 101 18.5 -> 22.9 M (63 registers uncapped: eight cells), id 103 9.8 -> 10.1 M.
 * RadioSaber's kernel (9) is slower with ten cells at 48 registers (19.5 vs 20.25 M: 32 B of cold spills and tighter
 * scheduling cost more than the tenth cell brings) and UpperBound's (10) spills, so those are pinned to nine cells (56
 * registers; they take 50-56) -- pinned, because at 57 the ninth cell is gone (an unrelated edit once cost the headline 7 %
 * that way). */
template <int ALGO, bool TRACE, class SH>
constexpr int min_cells_per_sm() {
  if constexpr (SH::kStatic && RS_MIN_BLOCKS == 8) {
    if (ALGO == 8 || ((ALGO == 101 || ALGO == 103) && !TRACE)) return 10;
    if (ALGO == 11) return 8;   /* the sample search keeps five (metric, mask) pairs in registers: it spills at 56 */
    return 9;
  }
  return RS_MIN_BLOCKS;
}
template <int ALGO, bool TRACE, bool QUEUE, class SH = DynShape>
__global__ void __launch_bounds__(kThreads, min_cells_per_sm<ALGO, TRACE, SH>()) rs_tti_kernel(const DevCfg d, const RunArgs r) {
  extern __shared__ __align__(16) unsigned char smem[];
  /* The dimensions and the layout (Dims) are compile-time constants of a FixedShape instantiation and copies of the
   * launch parameters otherwise; pointers are always read from the parameter block itself (a local copy of the
   * whole DevCfg would cost them their "global memory" provenance: generic LD/ST instead of LDG/STG). */
  Dims dm;
  if constexpr (SH::kStatic) {
    constexpr Layout kLay = SH::layout(ALGO);
    dm.S = SH::S; dm.U = SH::U; dm.G = SH::G; dm.R = SH::R; dm.rbg = SH::RBG;
    dm.cqi_per_rb = SH::LAY; dm.cqi_row = SH::kCqiRow;
    dm.lay = kLay;
    dm.n_chunks = SH::chunks(ALGO); dm.m_cap = SH::mcap(ALGO); dm.sort_n = SH::kSortN; dm.sort_depth = SH::kSortDepth;
    dm.nb = 1;
    dm.direct = 0;
  } else {
    dm.S = d.S; dm.U = d.U; dm.G = d.G; dm.R = d.R; dm.rbg = d.rbg;
    dm.cqi_per_rb = d.cqi_per_rb; dm.cqi_row = d.cqi_row;
    dm.lay = d.lay;
    dm.n_chunks = d.n_chunks; dm.m_cap = d.m_cap; dm.sort_n = d.sort_n; dm.sort_depth = d.sort_depth;
    dm.nb = d.nb;
    dm.direct = d.direct;
  }
  Cell c = carve(smem, dm.lay);
  c.sb.eq_tab = d.eq_tab;
  c.sb.eq_max = d.eq_max;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int S = dm.S, U = dm.U, G = dm.G;
  const int b = blockIdx.x + r.cell_off;   /* a launch covers the cells [cell_off, cell_off + gridDim.x) of the batch */
  constexpr bool NVS = ALGO == 7 || ALGO == 11;   /* DownlinkNVSScheduler, greedy and non-greedy */
  /* DownlinkTransportScheduler with one of its inter-slice algorithms: GreedyByRow (8), MaximizeCell (9),
   * UpperBound (10), SubOpt (101), VogelApproximate (103) */
  constexpr bool TRANSPORT = ALGO == 8 || ALGO == 9 || ALGO == 10 || ALGO == 101 || ALGO == 103;
  if (b >= d.n_cells) return;
  c.cumb = d.cum_bytes + (size_t)b * U * (QUEUE ? dm.nb : 1);
  c.cumr = d.cum_rbs + (size_t)b * U * (QUEUE ? dm.nb : 1);

  /* cell state -> shared memory */
  const int nb = QUEUE ? dm.nb : 1;   /* bearers per UE: the backlogged instantiations know one */
  for (int u = tid; u < U; u += kThreads) {
    const size_t i = (size_t)b * U + u;
    for (int k = 0; k < nb; ++k) {
      c.avg[nb * u + k] = d.avg[nb * i + k];
      c.tx[nb * u + k] = d.tx[nb * i + k];
    }
    c.mask[2 * u] = 0;
    c.mask[2 * u + 1] = 0;
    if (TRACE) c.utr[u] = d.ue_trace_off[i];
  }
  for (int s = tid; s < S; s += kThreads) {
    c.off[s] = NVS ? d.ewma[(size_t)b * S + s] : ((ALGO == 1) ? 0.0 : d.offset[(size_t)b * S + s]);
    c.frb[s] = 0;
    c.wd[s] = 0;
    c.target[s] = 0;
    c.quota[s] = 0;
  }
  if (tid < 16) c.tval[tid] = c_tab.tval[tid];
  for (int g = tid; g < G; g += kThreads) c.outsl[g] = 0xff;
  /* the cell's slice profile: every per-profile table read below goes through prof_row() */
  if constexpr (SH::kStatic) {
    if (tid == 0) c.misc[0] = d.cell_profile ? (unsigned)d.cell_profile[b] : 0u;
  } else {
    const int pf = d.cell_profile ? d.cell_profile[b] : 0;
    if (tid == 0) c.misc[0] = (unsigned)pf;
    {
      const int* sp = d.slice_ptr + pf * ((ALGO == 1) ? 2 : S + 1);
      const int* su = d.slice_ues + pf * U;
      for (int s = tid; s <= ((ALGO == 1) ? 1 : S); s += kThreads) c.sptr[s] = sp[s];
      for (int u = tid; u < U; u += kThreads) c.sues[u] = (unsigned short)su[u];
    }
  }
  /* the slice tables: CSR of the UEs by slice in shared memory, or plain arithmetic for a FixedShape */
  auto slice_of = [&](int u) -> int {
    if constexpr (SH::kStatic) return u / SH::UPS; else return d.ue_to_slice[prof_row(d, c, U) + u];
  };
  auto sptr_of = [&](int s) -> int { if constexpr (SH::kStatic) return s * SH::UPS; else return c.sptr[s]; };
  auto sue_of = [&](int j) -> int { if constexpr (SH::kStatic) return j; else return (int)c.sues[j]; };
  auto chunk_lo = [&](int ch) -> int {
    if constexpr (SH::kStatic) return min(ch * SH::kSlicesPerChunk, SH::S);
    else return d.chunk_slice[prof_row(d, c, dm.n_chunks + 1) + ch];
  };
  __syncthreads();

  /* One TTI of this cell's CQI lands in shared memory while P0 runs: rows [U][cqi_row], from the slab or
   * (trace mode) from the line in force of each UE's trace.  Consecutive TTIs that read the same slab /
   * line keep what is there. */
  const bool stage = r.stage != 0;
  int staged_key = -1;
  auto cqi_key = [&](int t) { return TRACE ? r.trace_row[t] : (r.t0 + t) / r.cqi_refresh; };
#ifdef RS_NO_BULK
  auto stage_cqi = [&](int t) {
    if (TRACE) {
      const uint8_t* base = d.trace_tab + (size_t)r.trace_row[t] * dm.cqi_row;
      const int cpr = dm.cqi_row >> 4;
      for (int q = tid; q < U * cpr; q += kThreads) {
        const int u = q / cpr, part = (q - u * cpr) << 4;
        cp_async16(c.cq + u * dm.cqi_row + part, base + c.utr[u] + part);
      }
    } else {
      const uint8_t* src = r.cqi + (size_t)((r.t0 + t) / r.cqi_refresh) * r.cqi_tti_stride + (size_t)b * U * dm.cqi_row;
      const int n16 = (U * dm.cqi_row) >> 4;
      for (int q = tid; q < n16; q += kThreads) cp_async16(c.cq + (q << 4), src + ((size_t)q << 4));
    }
    cp_async_commit();
  };
  auto stage_wait = [&]() { cp_async_wait_all(); };   /* own copies done; the barrier that follows publishes everybody's */
#else
  /* thread 0 arms the mbarrier with the byte count; the slab is ONE bulk copy, the trace rows of the cell's UEs one
   * bulk copy per UE (issued by the threads in parallel); every thread then waits for the phase to flip */
  unsigned stage_parity = 0;
  bool stage_pending = false;
  if (stage) {
    if (tid == 0) mbar_init(c.mbar, 1);
    __syncthreads();
  }
  auto stage_cqi = [&](int t) {
    const unsigned total = (unsigned)(U * dm.cqi_row);
    if (TRACE) {
      if (tid == 0) mbar_expect_tx(c.mbar, total);
      const uint8_t* base = d.trace_tab + (size_t)r.trace_row[t] * dm.cqi_row;
      for (int u = tid; u < U; u += kThreads) bulk_g2s(c.cq + u * dm.cqi_row, base + c.utr[u], (unsigned)dm.cqi_row, c.mbar);
    } else if (tid == 0) {
      const uint8_t* src = r.cqi + (size_t)((r.t0 + t) / r.cqi_refresh) * r.cqi_tti_stride + (size_t)b * U * dm.cqi_row;
      mbar_expect_tx(c.mbar, total);
      bulk_g2s(c.cq, src, total, c.mbar);
    }
    stage_pending = true;
  };
  auto stage_wait = [&]() {
    if (stage_pending) {
      mbar_wait(c.mbar, stage_parity);
      stage_parity ^= 1u;
      stage_pending = false;
    }
  };
#endif
  if (stage && r.T > 0) { stage_cqi(0); staged_key = cqi_key(0); }

#ifdef RS_PHASE_TIMING
  long long ph_[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  long long last_ = clock64();
#endif
  for (int t = 0; t < r.T; ++t) {
    const uint8_t* cqi = TRACE ? d.trace_tab + (size_t)r.trace_row[t] * dm.cqi_row
                               : r.cqi + (size_t)((r.t0 + t) / r.cqi_refresh) * r.cqi_tti_stride +
                                     (size_t)b * U * dm.cqi_row;
    const uint8_t* act = r.active ? r.active + (size_t)t * r.active_tti_stride + (size_t)b * U : nullptr;
    const double dt = r.dt[t];
    const size_t tb = (size_t)t * d.n_cells + b;
    const int rot = (b + t) % kWarps;   /* which warp plays the single-warp roles this TTI */
    /* queue state of the TTI (SURVEY 8 f3): a bearer is listed when it has packets (transport.cpp:119) */
    const int* qd = QUEUE ? r.queue + tb * U * nb : nullptr;   /* QUEUE = false: the backlogged instantiation, no queue code */
    const double* hl = (QUEUE && r.hol) ? r.hol + tb * U * nb : nullptr;
    const bool two = QUEUE && nb == 2;   /* two bearers per UE, slot i = priority i = position in the bearer container */
    /* a user is listed when one of its bearers has packets (transport.cpp:119, packet-scheduler.cpp:304-318) */
    auto listed = [&](int u) {
      return (!act || act[u]) && (two ? (qd[2 * u] > 0 || qd[2 * u + 1] > 0) : (qd ? qd[u] > 0 : d.data > 0));
    };
    /* dataToTransmit of the bearer that created the user record (m_requiredRBs, packet-scheduler.cpp:333) / of the
     * single bearer */
    auto data_of = [&](int u) { return two ? (qd[2 * u] > 0 ? qd[2 * u] : qd[2 * u + 1]) : (qd ? qd[u] : d.data); };
    /* slice_priority_ (transport.cpp:115, 143-146): the highest priority among the slice's listed bearers, kept in
     * bit 8 of wd[s] next to the "slice has data" flag in bit 0 */
    auto slice_flags = [&](int u) { return 1 | ((two && qd[2 * u + 1] > 0) ? 0x100 : 0); };
    /* metric factor of user u of an alpha slice (hm = holmul): 0 when the bearer of the slice's priority has nothing
     * queued, the bearer's head-of-line delay when the delay is in the metric, else 1 (transport.cpp:694-711) */
    auto prio_gate = [&](int u, int su, int hm, double e) -> double {
      if (two) {
        const int pr = (c.wd[su] >> 8) & 1;
        if (qd[2 * u + pr] == 0) return 0.0;
        return hm == 1 ? __dmul_rn(hl ? hl[2 * u + pr] : 0.0, e) : e;
      }
      if (hm == 1) return __dmul_rn(hl ? hl[u] : 0.0, e);   /* HoL * pow(se, eps) / pow(avg, psi), :702-706 */
      if (hm == 2 && hl && hl[u] < 0.0) return 0.0;          /* the bearer of the slice's priority is empty, :696-698 */
      return e;
    };
    auto row_of = [&](int u) -> const uint8_t* { return stage ? c.cq + u * dm.cqi_row : ue_cqi<TRACE>(d, dm, c, cqi, u); };
    short* o_rbg = r.rbg_to_ue ? r.rbg_to_ue + tb * G : nullptr;
    int* o_bits = r.tbs_bits ? r.tbs_bits + tb * U : nullptr;
    uint8_t* o_mcs = r.mcs ? r.mcs + tb * U : nullptr;
    uint8_t* o_fc = r.final_cqi ? r.final_cqi + tb * U : nullptr;
    int* o_tgt = r.slice_target ? r.slice_target + tb * S : nullptr;
    int* o_quo = r.slice_quota ? r.slice_quota + tb * S : nullptr;

    /* ---- buffered handles: arrivals, and the queue / HoL this TTI shows, from the bearers' FIFOs ---- */
    if (QUEUE && r.buf_k > 0) {
      const int* arr = r.arrivals + tb * U * nb;
      for (int q = tid; q < U * nb; q += kThreads) {
        const size_t i = (size_t)b * U * nb + q;
        buf_arrive(r.buf_meta + i, r.buf_time + i * r.buf_k, r.buf_bytes + i * r.buf_k, r.buf_k, arr[q], r.arr_time[t],
                   r.now[t], const_cast<int*>(qd) + q, const_cast<double*>(hl) + q);
      }
      __syncthreads();
    }

    /* ---- NVS: SelectSliceToServe (nvs.cpp:94-142) runs before the EWMA update ---------------- */
    int served = -1;
    if (NVS) {
      /* slices with at least one queued bearer */
      for (int u = tid; u < U; u += kThreads)
        if (listed(u)) atomicOr(&c.wd[slice_of(u)], slice_flags(u));
      __syncthreads();
      if (tid == 0) {
        int slice_id = 0;
        double max_score = 0;
        const double* weight = d.weight + prof_row(d, c, S);
        for (int i = 0; i < S; ++i) {
          if (!c.wd[i]) continue;
          if (c.off[i] == 0) { slice_id = i; break; }
          const double score = __ddiv_rn(weight[i], c.off[i]);
          if (score >= max_score) { max_score = score; slice_id = i; }
        }
        const double beta = 0.01; /* nvs.h:42 */
        for (int i = 0; i < S; ++i) {
          if (!c.wd[i]) continue;
          double e = __dmul_rn(1 - beta, c.off[i]);
          if (i == slice_id) e = __dadd_rn(e, __dmul_rn(beta, 1.0));
          c.off[i] = e;
        }
        c.misc[15] = (unsigned)slice_id;
        if (r.nvs_slice) r.nvs_slice[tb] = slice_id;
      }
      __syncthreads();
      served = (int)c.misc[15];
    }

    /* ---- P0: EWMA of every bearer; metric denominators; slices with data --------------------- */
    const unsigned char* psi = d.psi + (ALGO == 11 ? 0 : prof_row(d, c, S));   /* id 11: psi all 0, one row will do */
    for (int u = tid; u < U; u += kThreads) {
      double a = c.avg[nb * u];
      if (dt != 0) {
        a = ewma_update(a, c.tx[nb * u], dt);
        c.avg[nb * u] = a;
        c.tx[nb * u] = 0;
      }
      double sum = __dadd_rn(1.0, a);   /* averageRate = 1 + the listed bearers' rates, in slot order (transport.cpp:680-687) */
      if (two) {
        double a1 = c.avg[2 * u + 1];
        if (dt != 0) {
          a1 = ewma_update(a1, c.tx[2 * u + 1], dt);
          c.avg[2 * u + 1] = a1;
          c.tx[2 * u + 1] = 0;
        }
        sum = 1.0;
        if (qd[2 * u] > 0) sum = __dadd_rn(sum, a);
        if (qd[2 * u + 1] > 0) sum = __dadd_rn(sum, a1);
      }
      if (ALGO == 1) {
        c.den[u] = a;                                             /* dl-pf-packet-scheduler.cpp:128-140 */
      } else {
        const int s = slice_of(u);
        /* average_rate = (1 + sum avg) / 1000.0; pow(x, psi) for psi in {0,1}  (transport.cpp:680-692) */
        c.den[u] = psi[s] ? __ddiv_rn(sum, 1000.0) : 1.0;
        if (TRANSPORT && listed(u)) {
          if (two) atomicOr(&c.wd[s], slice_flags(u));
          else c.wd[s] = 1;
        }
      }
    }
    if (stage) stage_wait();
    __syncthreads();

    RS_TICK(0);
    if (TRANSPORT) {
      if (dm.direct) {
        /* ---- P2 for big slices: the per-chunk metric table leaves most of the CTA idle when a chunk holds one or two
         * slices of dozens of UEs (20 x 40 UEs: 16 items per chunk for 512 threads, 20 chunks one after the other).
         * Here every (slice, RBG quad) of the cell is an item at once and the metric of a (UE, RBG) pair is divided
         * where it is compared: Epow[s][cqi] / den[u], the same two doubles and the same IEEE divide as a table
         * entry, so the winners are the same.  Epow's rows are staged in the (otherwise unused) table area. */
        if (warp == (rot + kWarps - 1) % kWarps)
          slice_quotas(d, dm, c, r.rand2[tb * d.rand_stride], r.rand2[tb * d.rand_stride + 1], lane, o_tgt, o_quo);
        double* ep = c.mtab;
        const double* epow = d.epow + prof_row(d, c, S * 16);
        for (int q = tid; q < S * kMStride; q += kThreads) ep[q] = epow[q];
        __syncthreads();
        const bool nib = dm.cqi_per_rb == 2;   /* the host enables this path for one-CQI-per-RBG layouts and G % 4 == 0 */
        const int per = G >> 2;
        for (int q = tid; q < S * per; q += kThreads) {
          const int s = q / per, g0 = (q % per) * 4;
          const int hm = d.holmul[prof_row(d, c, S) + s];
          double best[4] = {-1.0, -1.0, -1.0, -1.0};
          unsigned bu01 = 0xffffffffu, bu23 = 0xffffffffu;   /* winners of RBGs g0..g0+3, 16 bits each (kNoUe = none) */
          auto quad_of = [&](int u) -> unsigned {   /* the CQIs of UE u on the four RBGs, one per byte */
            const uint8_t* row_u = row_of(u);
            if (nib) {
              const unsigned h = *(const unsigned short*)(row_u + (g0 >> 1));
              return (h & 0xfu) | ((h & 0xf0u) << 4) | ((h & 0xf00u) << 8) | ((h & 0xf000u) << 12);
            }
            return *(const unsigned*)(row_u + g0);
          };
          for (int j = sptr_of(s); j < sptr_of(s + 1); ++j) {
            const int u = sue_of(j);
            if (!listed(u)) continue;
            const unsigned w = quad_of(u);
            const double den_u = c.den[u];
#pragma unroll
            for (int x = 0; x < 4; ++x) {
              const int cq = (w >> (8 * x)) & 15;
              double e = ep[s * kMStride + cq];
              if (hm) e = QUEUE ? prio_gate(u, s, hm, e) : (hm == 1 ? __dmul_rn(0.0, e) : e);
              const double mv = cq ? __ddiv_rn(e, den_u) : 0.0;
              if (mv > best[x]) {
                best[x] = mv;
                if (x == 0) bu01 = (bu01 & 0xffff0000u) | (unsigned)u;
                else if (x == 1) bu01 = (bu01 & 0x0000ffffu) | ((unsigned)u << 16);
                else if (x == 2) bu23 = (bu23 & 0xffff0000u) | (unsigned)u;
                else bu23 = (bu23 & 0x0000ffffu) | ((unsigned)u << 16);
              }
            }
          }
#pragma unroll
          for (int x = 0; x < 4; ++x) {
            const int g = g0 + x;
            const unsigned wu = ((x < 2 ? bu01 : bu23) >> (16 * (x & 1))) & 0xffffu;
            const int wc = wu == kNoUe ? 0 : (int)((quad_of((int)wu) >> (8 * x)) & 15);   /* the sort key: the winner's CQI */
            c.sb.a[g * S + s] = (unsigned short)((wc << 12) | (g << 6) | s);
            c.win[g * S + s] = (unsigned short)wu;
          }
        }
        __syncthreads();
      } else
      /* ---- P1/P2: metric table per chunk of slices, per-(rbg,slice) argmax; quotas by the last warp */
      for (int ch = 0; ch < dm.n_chunks; ++ch) {
        const int s0 = chunk_lo(ch), s1 = chunk_lo(ch + 1);
        const int j0 = sptr_of(s0), j1 = sptr_of(s1);
        if (ch == 0 && warp == (rot + kWarps - 1) % kWarps)
          slice_quotas(d, dm, c, r.rand2[tb * d.rand_stride], r.rand2[tb * d.rand_stride + 1], lane, o_tgt, o_quo);
        const double* epow = d.epow + prof_row(d, c, S * 16);
        const unsigned char* holmul = d.holmul + prof_row(d, c, S);
        for (int q = tid; q < (j1 - j0) * kMStride; q += kThreads) {
          const int j = j0 + (q >> 4), cq = q & 15;
          const int u = sue_of(j);
          const int su = slice_of(u);
          double e = epow[su * 16 + cq];
          const int hm = holmul[su];
          /* alpha slices: gate / head-of-line delay of the prioritised bearer; without queue state (backlogged
           * instantiation) the delay of an infinite buffer is 0, so an alpha+beta slice's metric is 0 */
          if (hm) e = QUEUE ? prio_gate(u, su, hm, e) : (hm == 1 ? __dmul_rn(0.0, e) : e);
          c.mtab[q] = cq ? __ddiv_rn(e, c.den[u]) : 0.0;
        }
        __syncthreads();
        /* four RBGs per item (one 32-bit CQI load per UE) while that still gives every thread an item;
         * fewer, bigger slices on a wide CTA go one RBG per item */
        const bool vec4 = dm.cqi_per_rb != 1 && (G % 4 == 0) && (kThreads <= 128 || (s1 - s0) * (G >> 2) >= kThreads);
        const bool nib = dm.cqi_per_rb == 2;
        if (vec4) {
          const int g4 = G >> 2;
          const int items = (s1 - s0) * g4;
          for (int q = tid; q < items; q += kThreads) {
            const int s = s0 + q / g4, g0 = (q % g4) * 4;
            double best[4] = {-1.0, -1.0, -1.0, -1.0};
            int bu[4] = {kNoUe, kNoUe, kNoUe, kNoUe};
            int bc[4] = {0, 0, 0, 0};
            for (int j = sptr_of(s); j < sptr_of(s + 1); ++j) {
              const int u = sue_of(j);
              if (!listed(u)) continue;
              unsigned w;
              const uint8_t* row_u = row_of(u);
              if (nib) {   /* four nibbles -> one per byte, then the same extraction as the u8 layout */
                const unsigned h = *(const unsigned short*)(row_u + (g0 >> 1));
                w = (h & 0xfu) | ((h & 0xf0u) << 4) | ((h & 0xf00u) << 8) | ((h & 0xf000u) << 12);
              } else {
                w = *(const unsigned*)(row_u + g0);
              }
              const double* row = c.mtab + (j - j0) * kMStride;
#pragma unroll
              for (int x = 0; x < 4; ++x) {
                const int cq = (w >> (8 * x)) & 15;
                const double m = row[cq];
                if (m > best[x]) { best[x] = m; bu[x] = u; bc[x] = cq; }
              }
            }
#pragma unroll
            for (int x = 0; x < 4; ++x) {
              const int g = g0 + x;
              c.sb.a[g * S + s] = (unsigned short)((bc[x] << 12) | (g << 6) | s);
              c.win[g * S + s] = (unsigned short)bu[x];
            }
          }
        } else {
          const int items = (s1 - s0) * G;
          for (int q = tid; q < items; q += kThreads) {
            const int s = s0 + q / G, g = q % G;
            double best = -1.0;
            int bu = kNoUe, bc = 0;
            for (int j = sptr_of(s); j < sptr_of(s + 1); ++j) {
              const int u = sue_of(j);
              if (!listed(u)) continue;
              const int cq = cqi_first_rb(dm, row_of(u), g);
              const double m = c.mtab[(j - j0) * kMStride + cq];
              if (m > best) { best = m; bu = u; bc = cq; }
            }
            c.sb.a[g * S + s] = (unsigned short)((bc << 12) | (g << 6) | s);
            c.win[g * S + s] = (unsigned short)bu;
          }
        }
        __syncthreads();
      }

      RS_TICK(1);
      /* ---- P3/P4: inter-slice assignment ---------------------------------------------------- */
      if (ALGO == 10) {
        /* UpperBound (transport.cpp:223-246, 603-616): every slice with a positive quota takes the first
         * quota entries of ITS OWN std::sort of the G (rbg, efficiency) pairs, so an RBG can be granted
         * to several slices.  One sort of G entries per slice (warp_sort_desc); the grants are parked in
         * shared memory (slice-major, sorted order) next to the sort buffers.  Every grant is booked: the slices
         * together make at most S * G of them, and the slot arrays hold n >= S * G entries. */
        /* up to five slices at a time, one warp each, on private buffers in the (dead) right slot array; g_rbg
         * [S*G] (the RBG of grant wd[s] + k, the k-th of slice s) sits in the left one.  The user of that grant is
         * win[g * S + s]; once the sorts are done g_ue [S*G] keeps it in grant order in the (then dead) key array. */
        unsigned short* g_rbg = c.sb.posl;
        unsigned short* g_ue = c.sb.a;
        constexpr int kSorters = kWarps < 5 ? kWarps : 5;
        int base = 0;
        for (int s = 0; s < S; ++s) {   /* every thread: where each slice's grants start */
          const int q = min(c.quota[s], G);
          if (tid == 0) { c.frb[s] = max(q, 0); c.wd[s] = base; }   /* wd is free once the quotas exist: first grant of the slice */
          if (q > 0) base += q;
        }
        __syncthreads();
        if (warp < kSorters) {
          SortBufs s2 = c.sb;
          s2.a = c.sb.posr + warp * 3 * G;
          s2.posl = s2.a + G;
          s2.posr = s2.a + 2 * G;
          s2.out = s2.posr;
          s2.cnt = c.sb.cnt + warp * 32;
          unsigned* stack = c.sb.seg0 + warp * 16;
          for (int s = warp; s < S; s += kSorters) {
            const int q = c.frb[s], b0 = c.wd[s];
            if (q <= 0) continue;
            for (int i = lane; i < G; i += 32) s2.a[i] = (unsigned short)((c.sb.a[i * S + s] & 0xf000u) | (unsigned)i);
            __syncwarp();
            warp_sort_desc(s2, stack, G, d.sort_depth_g, lane);
            for (int k = lane; k < q; k += 32) g_rbg[b0 + k] = s2.out[k] & 0xfff;
            __syncwarp();
          }
        }
        __syncthreads();
        for (int u = tid; u < U; u += kThreads) c.den[u] = 0.0;   /* the metric denominators are dead: EESM sums */
        __syncthreads();
        /* per slice, in grant order: the winner's RB list grows by the RBG's RBs (EESM summand per RB) */
        for (int s = tid; s < S; s += kThreads) {
          const int q = c.frb[s], b0 = c.wd[s];
          int cnt = 0;
          for (int k = 0; k < q; ++k) {
            const int g = g_rbg[b0 + k], ue = c.win[g * S + s];
            g_ue[b0 + k] = (unsigned short)ue;
            if (ue == kNoUe) continue;
            cnt++;
            double sum = c.den[ue];
            const uint8_t* row = row_of(ue);
            if (dm.cqi_per_rb == 1) {
              const uint8_t* p = row + (size_t)g * dm.rbg;
              for (int rr = 0; rr < dm.rbg; ++rr) sum = __dadd_rn(sum, c.tval[p[rr] & 15]);
            } else {
              const double tv = c.tval[cqi_first_rb(dm, row, g)];
              for (int rr = 0; rr < dm.rbg; ++rr) sum = __dadd_rn(sum, tv);
            }
            c.den[ue] = sum;
            c.mask[2 * ue + (g >> 5)] |= 1u << (g & 31);   /* a UE belongs to one slice: no other thread touches it */
          }
          c.frb[s] = cnt;
          if (c.misc[14]) c.off[s] = (double)(c.target[s] - cnt * dm.rbg);   /* :618-620 */
          else { if (o_tgt) o_tgt[s] = 0; if (o_quo) o_quo[s] = 0; }
        }
        __syncthreads();
        /* the reported list: the first grant_len grants (rs_set_grant_list_len), the schedule holds all of them */
        const int n_list = d.grant_len;
        short* o_au = r.alloc_ue ? r.alloc_ue + tb * n_list : nullptr;
        short* o_ar = r.alloc_rbg ? r.alloc_rbg + tb * n_list : nullptr;
        for (int e = tid; e < n_list; e += kThreads) {
          const bool in = e < base && g_ue[e] != kNoUe;
          if (o_au) o_au[e] = in ? (short)g_ue[e] : (short)-1;
          if (o_ar) o_ar[e] = in ? (short)g_rbg[e] : (short)-1;
        }
        if (tid == 0 && r.alloc_n) r.alloc_n[tb] = base;
        /* single-valued view: the highest UE id holding the RBG.  Slice s granted RBG g to its winner w there exactly
         * when w's RB mask has g (w is in slice s only) */
        for (int g = tid; g < G; g += kThreads) {
          int ue = -1;
          for (int s = 0; s < S; ++s) {
            const int w = c.win[g * S + s];
            if (w != kNoUe && ((c.mask[2 * w + (g >> 5)] >> (g & 31)) & 1u)) ue = max(ue, w);
          }
          if (o_rbg) o_rbg[g] = (short)ue;
        }
      } else if (ALGO == 103) {
        vogel_approximate(d, dm, c);
      } else if (ALGO == 101) {
        sub_opt(d, dm, c);
      } else if (ALGO == 9) {
#ifndef RS_SKIP_SORT
        sort_desc(c.sb, dm.sort_n, dm.sort_depth, kWarps - rot);
#endif
        RS_TICK(2);
#ifndef RS_SKIP_GREEDY
        if (warp == rot) greedy_maxcell(d, dm, c, c.sb.out, lane);
#endif
        RS_TICK(3);
      } else {
        if (warp == rot) greedy_by_row(d, dm, c, c.sb.a, lane);
      }
      __syncthreads();

      RS_TICK(4);
      /* ---- P5: RBG -> UE (transport.cpp:589-601) --------------------------------------------- */
      if (ALGO != 10)
      for (int g = tid; g < G; g += kThreads) {
        const int sl = c.outsl[g];
        int ue = -1;
        if (sl != 0xff) {
          const unsigned short w = c.win[g * S + sl];
          if (w != kNoUe) {
            ue = w;
            atomicAdd(&c.frb[sl], 1);
            atomicOr(&c.mask[2 * ue + (g >> 5)], 1u << (g & 31));
          }
        }
        if (o_rbg) o_rbg[g] = (short)ue;
        c.outsl[g] = 0xff;
      }
      __syncthreads();
      /* slice_rbs_offset_ update (:618-620); only when RBsAllocation ran (>= 1 user) */
      if (ALGO != 10)
      for (int s = tid; s < S; s += kThreads) {
        if (c.misc[14]) c.off[s] = (double)(c.target[s] - c.frb[s] * dm.rbg);
        else { if (o_tgt) o_tgt[s] = 0; if (o_quo) o_quo[s] = 0; }
      }
    } else if (ALGO == 11) {
      /* ---- NVS non-greedy (RBsAllocationNonGreedyPF + AssignRBsGivenMCS, nvs.cpp:405-528): 300 samples
       * of per-user CQI back-offs, one sample per thread at a time; the first sample with the largest
       * sum over RBGs of the winning PF metric is kept. */
      const int j0 = sptr_of(served), j1 = sptr_of(served + 1);
      if (warp == 0) {   /* the users the reference lists: bearers of the served slice with packets, in order */
        int cnt = 0;
        for (int jb = j0; jb < j1; jb += 32) {
          const int j = jb + lane;
          const int u = j < j1 ? sue_of(j) : 0;
          const bool in = j < j1 && listed(u);
          const unsigned bal = __ballot_sync(kFull, in);
          if (in) c.ng_list[cnt + __popc(bal & ((1u << lane) - 1u))] = (unsigned short)u;
          cnt += __popc(bal);
        }
        if (lane == 0) c.misc[13] = (unsigned)cnt;
      }
      __syncthreads();
      const int Ua = (int)c.misc[13];
      const bool few = Ua <= 8 && G <= 64;   /* the search on RBG bitmasks (ng_search), else entry by entry */
      unsigned* ok = (unsigned*)c.ng_mcs;    /* few: ok[(q * 16 + t) * 2 + w] = RBGs 32 w .. 32 w + 31 of user q with CQI >= t */
      if (few) {
        for (int q = warp; q < Ua; q += kWarps) {   /* one warp per listed user: a ballot per threshold and half */
          const uint8_t* row = row_of(c.ng_list[q]);
          const int c0 = lane < G ? cqi_first_rb(dm, row, lane) : 0, c1 = lane + 32 < G ? cqi_first_rb(dm, row, lane + 32) : 0;
          int hc = 0;
          for (int t = 1; t < 16; ++t) {
            const unsigned b0 = __ballot_sync(kFull, c0 >= t), b1 = __ballot_sync(kFull, c1 >= t);
            if (lane == 0) {
              ok[(q * 16 + t) * 2] = b0;
              ok[(q * 16 + t) * 2 + 1] = b1;
            }
            if (b0 | b1) hc = t;
          }
          if (lane == 0) c.ng_hc[q] = (unsigned char)hc;   /* user_highest_cqi, nvs.cpp:416-425 */
        }
      } else {
        for (int q = tid; q < Ua; q += kThreads) {   /* user_highest_cqi, nvs.cpp:416-425 */
          const uint8_t* row = row_of(c.ng_list[q]);
          int hc = 0;
          for (int g = 0; g < G; ++g) hc = max(hc, cqi_first_rb(dm, row, g));
          c.ng_hc[q] = (unsigned char)hc;
        }
      }
      for (int q = tid; q < Ua * kMStride; q += kThreads) {   /* sEff * 180000 / (1 + avg), nvs.cpp:512-513 */
        const int cq = q & 15;
        /* UserToSchedule::GetAverageTransmissionRate: 1 + the listed bearers' rates in slot order (packet-scheduler.cpp:423-433) */
        const int un = c.ng_list[q >> 4];
        double rate = __dadd_rn(1.0, c.avg[nb * un]);
        if (two) {
          rate = 1.0;
          if (qd[2 * un] > 0) rate = __dadd_rn(rate, c.avg[2 * un]);
          if (qd[2 * un + 1] > 0) rate = __dadd_rn(rate, c.avg[2 * un + 1]);
        }
        c.mtab[q] = cq ? __ddiv_rn(d.epow[cq], rate) : 0.0;
      }
      __syncthreads();
      const int* draws = r.rand2 + tb * d.rand_stride;
      unsigned char* my = c.ng_mcs + tid * d.ng_ues;
      double best_pf = 0.0;
      int best_i = 0x7fffffff;
      if (Ua > 0 && few) {
        if (Ua <= 5) ng_search<5>(c, ok, draws, Ua, G, tid, best_pf, best_i);
        else ng_search<8>(c, ok, draws, Ua, G, tid, best_pf, best_i);
      } else if (Ua > 0) {
        for (int i = tid; i < 300; i += kThreads) {
          for (int q = 0; q < Ua; ++q) my[q] = (unsigned char)max((int)c.ng_hc[q] - draws[i * Ua + q] % 4, 1);
          double pf = 0.0;
          for (int g = 0; g < G; ++g) {
            double highest = -1.0;
            for (int q = 0; q < Ua; ++q) {
              const int mcs = my[q];
              const double m = (mcs <= cqi_first_rb(dm, row_of(c.ng_list[q]), g)) ? c.mtab[q * kMStride + mcs] : 0.0;
              if (highest < m) highest = m;
            }
            pf = __dadd_rn(pf, highest);
          }
          if (best_pf < pf) { best_pf = pf; best_i = i; }   /* this thread's samples come in increasing order */
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double op = __shfl_xor_sync(kFull, best_pf, o);
        const int oi = __shfl_xor_sync(kFull, best_i, o);
        if (op > best_pf || (op == best_pf && oi < best_i)) { best_pf = op; best_i = oi; }
      }
      if (lane == 0) {
        ((double*)c.ng_red)[warp] = best_pf;
        ((int*)(c.ng_red + 8 * kWarps))[warp] = best_i;
      }
      __syncthreads();
      best_pf = ((double*)c.ng_red)[0];
      best_i = ((int*)(c.ng_red + 8 * kWarps))[0];
      for (int w = 1; w < kWarps; ++w) {
        const double op = ((double*)c.ng_red)[w];
        const int oi = ((int*)(c.ng_red + 8 * kWarps))[w];
        if (op > best_pf || (op == best_pf && oi < best_i)) { best_pf = op; best_i = oi; }
      }
      for (int g = tid; g < G; g += kThreads) {   /* the winning sample's assignment, nvs.cpp:453-460 */
        int bu = -1;
        if (best_i != 0x7fffffff) {
          double highest = -1.0;
          for (int q = 0; q < Ua; ++q) {
            const int mcs = max((int)c.ng_hc[q] - draws[best_i * Ua + q] % 4, 1);
            const int u = c.ng_list[q];
            const double m = (mcs <= cqi_first_rb(dm, row_of(u), g)) ? c.mtab[q * kMStride + mcs] : 0.0;
            if (highest < m) { highest = m; bu = u; }
          }
        }
        if (bu >= 0) atomicOr(&c.mask[2 * bu + (g >> 5)], 1u << (g & 31));
        if (o_rbg) o_rbg[g] = (short)bu;
      }
    } else if (ALGO == 7) {
      /* ---- NVS: enterprise argmax over the served slice's users for every RBG (nvs.cpp:275-311) */
      const int j0 = sptr_of(served), j1 = sptr_of(served + 1);
      for (int q = tid; q < (j1 - j0) * kMStride; q += kThreads) {
        const int j = j0 + (q >> 4), cq = q & 15;
        const int u = sue_of(j);
        double e = d.epow[(prof_row(d, c, S) + served) * 16 + cq];
        if (d.holmul[prof_row(d, c, S) + served]) e = QUEUE ? prio_gate(u, served, 1, e) : 0.0;   /* nvs.cpp:379-386; no queue state: HoL 0 */
        c.mtab[q] = cq ? __ddiv_rn(e, c.den[u]) : 0.0;
      }
      if (qd) {
        /* finite queues: a user stops taking RBGs once it holds m_requiredRBs = dataToTransmit * 8 /
         * TBS(1 RB at its wideband CQI) RBs (packet-scheduler.cpp:321-334, nvs.cpp:299-300), so the RBGs go
         * one after the other (one warp, lanes over the slice's users) */
        int* req = (int*)c.ng_mcs;
        int* alc = req + d.ng_ues;
        for (int j = j0 + tid; j < j1; j += kThreads) {
          const int u = sue_of(j);
          int need = 0;
          if (listed(u)) {
            const uint8_t* row = row_of(u);
            double sum = 0;   /* EESM over every RB of the band, RB order */
            for (int g = 0; g < G; ++g) {
              if (dm.cqi_per_rb == 1) {
                const uint8_t* p = row + (size_t)g * dm.rbg;
                for (int rr = 0; rr < dm.rbg; ++rr) sum = __dadd_rn(sum, c.tval[p[rr] & 15]);
              } else {
                const double tv = c.tval[cqi_first_rb(dm, row, g)];
                for (int rr = 0; rr < dm.rbg; ++rr) sum = __dadd_rn(sum, tv);
              }
            }
            const int wide = cqi_from_mean(__ddiv_rn(sum, (double)(G * dm.rbg)));
            need = min(data_of(u), kMaxQueueBytes) * 8 / d.tbs1[wide];
          }
          req[j - j0] = need;
          alc[j - j0] = 0;
        }
        __syncthreads();
        if (warp == 0) {
          for (int g = 0; g < G; ++g) {
            double best = -1.0;
            int bj = 0x7fffffff;
            for (int j = j0 + lane; j < j1; j += 32) {
              const int u = sue_of(j);
              if (!listed(u) || alc[j - j0] >= req[j - j0]) continue;
              const double m = c.mtab[(j - j0) * kMStride + cqi_first_rb(dm, row_of(u), g)];
              if (m > best) { best = m; bj = j; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              const double om = __shfl_xor_sync(kFull, best, o);
              const int oj = __shfl_xor_sync(kFull, bj, o);
              if (om > best || (om == best && oj < bj)) { best = om; bj = oj; }
            }
            if (lane == 0) {
              int bu = -1;
              if (bj != 0x7fffffff) {
                bu = sue_of(bj);
                alc[bj - j0] += dm.rbg;
                c.mask[2 * bu + (g >> 5)] |= 1u << (g & 31);
              }
              if (o_rbg) o_rbg[g] = (short)bu;
            }
            __syncwarp();
          }
        }
      } else {
      __syncthreads();
      for (int g = tid; g < G; g += kThreads) {
        double best = -1.0;   /* metrics are >= 0, so this behaves like numeric_limits::lowest() */
        int bu = -1;
        for (int j = j0; j < j1; ++j) {
          const int u = sue_of(j);
          if (!listed(u)) continue;
          const int cq = cqi_first_rb(dm, row_of(u), g);
          const double m = c.mtab[(j - j0) * kMStride + cq];
          if (m > best) { best = m; bu = u; }
        }
        if (bu >= 0) atomicOr(&c.mask[2 * bu + (g >> 5)], 1u << (g & 31));
        if (o_rbg) o_rbg[g] = (short)bu;
      }
      }
    } else if (qd) {
      /* ---- No-slicing PF with finite queues (dlps.cpp:227-271): a flow leaves the candidates once the TBS of
       * what it holds covers its queue, so the RBGs go one after the other (one warp, lanes over the flows) */
      double* fsum = c.mtab;   /* running EESM sum of every flow, RB order */
      for (int u = tid; u < U; u += kThreads) { fsum[u] = 0.0; c.done[u] = 0; }
      __syncthreads();
      if (warp == 0) {
        int n_flows = 0;
        for (int u = lane; u < U; u += 32) n_flows += listed(u) ? 1 : 0;
        n_flows = __reduce_add_sync(kFull, n_flows);
        int n_done = 0;
        for (int g = 0; g < G; ++g) {
          int bu = 0x7fffffff;
          if (n_done < n_flows) {
            double best = 0.0;
            for (int u = lane; u < U; u += 32) {
              if (!listed(u) || c.done[u]) continue;
              const double m = __ddiv_rn(d.epow[cqi_first_rb(dm, row_of(u), g)], c.den[u]);
              if (m > best) { best = m; bu = u; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              const double om = __shfl_xor_sync(kFull, best, o);
              const int ou = __shfl_xor_sync(kFull, bu, o);
              if (om > best || (om == best && ou < bu)) { best = om; bu = ou; }
            }
          }
          int finished = 0;
          if (lane == 0) {
            if (bu != 0x7fffffff) {
              c.mask[2 * bu + (g >> 5)] |= 1u << (g & 31);
              const uint8_t* row = row_of(bu);
              double sum = fsum[bu];
              if (dm.cqi_per_rb == 1) {
                const uint8_t* p = row + (size_t)g * dm.rbg;
                for (int rr = 0; rr < dm.rbg; ++rr) sum = __dadd_rn(sum, c.tval[p[rr] & 15]);
              } else {
                const double tv = c.tval[cqi_first_rb(dm, row, g)];
                for (int rr = 0; rr < dm.rbg; ++rr) sum = __dadd_rn(sum, tv);
              }
              fsum[bu] = sum;
              const int nrbg = __popc(c.mask[2 * bu]) + __popc(c.mask[2 * bu + 1]);
              const int fc = cqi_from_mean(__ddiv_rn(sum, (double)(nrbg * dm.rbg)));
              if (d.tbs_n[nrbg * 16 + fc] >= min(qd[bu], kMaxQueueBytes) * 8) {   /* dlps.cpp:264-269 */
                c.done[bu] = 1;
                finished = 1;
              }
            }
            if (o_rbg) o_rbg[g] = (short)(bu == 0x7fffffff ? -1 : bu);
          }
          n_done += __shfl_sync(kFull, finished, 0);
          __syncwarp();
        }
      }
    } else {
      /* ---- No-slicing PF: per RBG, first flow with the strictly largest metric (dlps.cpp:227-246) */
      for (int g = warp; g < G; g += kWarps) {
        double best = 0.0;
        int bu = 0x7fffffff;
        for (int u = lane; u < U; u += 32) {
          if (!listed(u)) continue;
          const int cq = cqi_first_rb(dm, row_of(u), g);
          const double m = __ddiv_rn(d.epow[cq], c.den[u]);
          if (m > best) { best = m; bu = u; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const double om = __shfl_xor_sync(kFull, best, o);
          const int ou = __shfl_xor_sync(kFull, bu, o);
          if (om > best || (om == best && ou < bu)) { best = om; bu = ou; }
        }
        if (lane == 0) {
          const int ue = (bu == 0x7fffffff) ? -1 : bu;
          if (ue >= 0) atomicOr(&c.mask[2 * ue + (g >> 5)], 1u << (g & 31));
          if (o_rbg) o_rbg[g] = (short)ue;
        }
      }
    }
    __syncthreads();

    RS_TICK(5);
    /* ---- P6: link adaptation, accounting, outputs; reset per-TTI scratch ---------------------- */
    for (int u = tid; u < U; u += kThreads) {
      const unsigned m_lo = c.mask[2 * u], m_hi = c.mask[2 * u + 1];
      const bool fifo = QUEUE && r.buf_k > 0;
      int tx0 = 0, tx1 = 0;   /* the bytes finalize_ue books to each bearer are the increments of its tx counter */
      if (fifo) { tx0 = c.tx[nb * u]; if (two) tx1 = c.tx[nb * u + 1]; }
      finalize_ue(d, dm, c, row_of(u), u, m_lo, m_hi, o_bits, o_mcs, o_fc, data_of(u), ALGO == 10 ? c.den : nullptr,
                  two ? qd : nullptr);
      if (fifo)
        for (int k = 0; k < nb; ++k) {
          const size_t i = ((size_t)b * U + u) * nb + k;
          buf_depart(r.buf_meta + i, r.buf_bytes + i * r.buf_k, r.buf_k, c.tx[nb * u + k] - (k ? tx1 : tx0));
        }
      c.mask[2 * u] = 0;
      c.mask[2 * u + 1] = 0;
    }
    for (int s = tid; s < S; s += kThreads) {
      c.frb[s] = 0;
      c.wd[s] = 0;
      c.target[s] = 0;
      c.quota[s] = 0;
    }
    __syncthreads();
    if (stage && t + 1 < r.T && cqi_key(t + 1) != staged_key) { stage_cqi(t + 1); staged_key = cqi_key(t + 1); }
  }

  RS_TICK(6);
#ifdef RS_PHASE_TIMING
  if (threadIdx.x == 0 && (blockIdx.x % 997) == 0)
    printf("cta %d T %d: p0 %lld argmax %lld sort %lld greedy %lld bar %lld p5 %lld p6 %lld (cycles per TTI)\n", blockIdx.x, r.T,
           ph_[0] / r.T, ph_[1] / r.T, ph_[2] / r.T, ph_[3] / r.T, ph_[4] / r.T, ph_[5] / r.T, ph_[6] / r.T);
#endif
  /* cell state -> HBM */
  for (int q = tid; q < U * nb; q += kThreads) {
    const size_t i = (size_t)b * U * nb + q;
    d.avg[i] = c.avg[q];
    d.tx[i] = c.tx[q];
  }
  if (NVS || TRANSPORT) {
    double* dst = NVS ? d.ewma : d.offset;
    for (int s = tid; s < S; s += kThreads) dst[(size_t)b * S + s] = c.off[s];
  }
}

#ifndef RS_CORE_ONLY
/* ---- test hook: the sort alone, one CTA per array --------------------------------------------- */
__global__ void __launch_bounds__(kThreads) rs_sort_test_kernel(const uint8_t* keys, int n, int depth, int* perm,
                                                                const unsigned short* eq_tab, int eq_max, const Layout L) {
  extern __shared__ __align__(16) unsigned char smem[];
  Cell c = carve(smem, L);
  c.sb.eq_tab = eq_tab;
  c.sb.eq_max = eq_max;
  const uint8_t* k = keys + (size_t)blockIdx.x * n;
  for (int i = threadIdx.x; i < n; i += kThreads) c.sb.a[i] = (unsigned short)(((k[i] & 15) << 12) | i);
  __syncthreads();
  sort_desc(c.sb, n, depth, blockIdx.x % kWarps);
  for (int i = threadIdx.x; i < n; i += kThreads) perm[(size_t)blockIdx.x * n + i] = c.sb.out[i] & 0xfff;
}

/* ---- synthetic workload (twin of radiosaber_b200/workload.py) -------------------------------- */
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
  unsigned long long z = x + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
struct CdfTable { unsigned thr[14]; };

__device__ __forceinline__ int synth_one(unsigned long long key, unsigned long long epoch, unsigned long long cell,
                                         unsigned long long ue, unsigned long long rbg, const CdfTable& cdf) {
  unsigned long long ctr = (epoch << 40) ^ (cell << 20) ^ (ue << 8) ^ rbg;
  ctr ^= (ue >> 12) * 0xD6E8FEB86659FD93ull;
  const unsigned u32 = (unsigned)(splitmix64(ctr ^ key) >> 32);
  int cq = 1;
#pragma unroll
  for (int k = 0; k < 14; ++k) cq += (u32 >= cdf.thr[k]);
  return cq;
}

/* n_slabs slabs of [n_cells][U][G] (packed = 0) or [n_cells][U][G/2] (packed = 1, RBG 2k in the low
 * nibble); slab j holds the CQI of TTI epoch epoch0 + j. */
__global__ void rs_synth_cqi_kernel(uint8_t* out, unsigned long long key, long long cell0, long long epoch0,
                                    int n_slabs, int n_cells, int U, int G, int packed, CdfTable cdf) {
  const int row = packed ? G / 2 : G;
  const size_t total = (size_t)n_slabs * n_cells * U * row;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const unsigned long long col = i % row;
    size_t r = i / row;
    const unsigned long long ue = r % U; r /= U;
    const unsigned long long cell = cell0 + (long long)(r % n_cells); r /= n_cells;
    const unsigned long long epoch = (unsigned long long)(epoch0 + (long long)r);
    if (packed) {
      const int lo = synth_one(key, epoch, cell, ue, 2 * col, cdf), hi = synth_one(key, epoch, cell, ue, 2 * col + 1, cdf);
      out[i] = (uint8_t)(lo | (hi << 4));
    } else {
      out[i] = (uint8_t)synth_one(key, epoch, cell, ue, col, cdf);
    }
  }
}

/* stride draws per (tti, cell): 2 for ids 8/9 (the original packing of the counter), more for id 11 */
__global__ void rs_synth_rand2_kernel(int* out, unsigned long long key, long long cell0, long long tti0,
                                      int n_ttis, int n_cells, int S, int stride) {
  const size_t total = (size_t)n_ttis * n_cells * stride;
  const unsigned long long span = (unsigned long long)(2147483647 - S + 1);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const unsigned long long which = i % stride;
    size_t r = i / stride;
    const unsigned long long cell = cell0 + (long long)(r % n_cells);
    const unsigned long long tti = tti0 + (long long)(r / n_cells);
    const unsigned long long ctr = stride == 2 ? ((tti << 32) ^ (cell << 1) ^ which)
                                               : ((tti << 40) ^ (cell << 16) ^ which ^ 0x5EA4C4000000ull);
    out[i] = (int)((splitmix64(ctr ^ key) >> 11) % span);
  }
}

/* Synthetic arrivals (twin of workload.synth_arrivals): int32 [n_ttis][n_cells][U][nb].  spec [P][S][2] = (packet
 * bytes, packets per TTI in 16.16 fixed point) of each profile's slices; a bearer gets (q >> 16) + (draw16 < (q & 0xffff))
 * packets, draw16 the top 16 bits of one counter-based draw per (tti, cell, ue, slot). */
__global__ void rs_synth_arrivals_kernel(int* out, unsigned long long key, long long cell0, long long tti0, int n_ttis,
                                         const DevCfg d, const int* spec) {
  const int nb = d.nb, U = d.U, S = d.S;
  const size_t total = (size_t)n_ttis * d.n_cells * U * nb;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const unsigned long long slot = i % nb;
    size_t r = i / nb;
    const int u = (int)(r % U); r /= U;
    const int b = (int)(r % d.n_cells);
    const unsigned long long cell = cell0 + b;
    const unsigned long long tti = tti0 + (long long)(r / d.n_cells);
    const int pf = d.cell_profile ? d.cell_profile[b] : 0;
    const int* sp = spec + 2 * ((size_t)pf * S + d.ue_to_slice[(size_t)pf * U + u]);
    const unsigned long long ue = (unsigned long long)u;
    const unsigned long long ctr = ((tti << 40) ^ (cell << 20) ^ (ue << 8) ^ slot) ^ ((ue >> 12) * 0xD6E8FEB86659FD93ull);
    const unsigned draw16 = (unsigned)(splitmix64(ctr ^ key) >> 48);
    const int q = sp[1];
    out[i] = sp[0] * ((q >> 16) + (draw16 < (unsigned)(q & 0xffff) ? 1 : 0));
  }
}

/* rs_get_buffers: the arrival time of every bearer's head record (0 when it holds none) */
__global__ void rs_buf_heads_kernel(const BufMeta* meta, const double* tm, int K, size_t n, double* out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = meta[i].n > 0 ? tm[i * K + meta[i].head] : 0.0;
}

/* ---- per-slice totals: uint64 [P][4][S] += over cells (integers: order-independent) ----------- */
/* Row p sums the cells of profile p with profile p's ue_to_slice.  in_smem: the P x 4 x S sums are gathered in shared
 * memory first (the host asks for it while they fit), else added to `stats` directly. */
__global__ void rs_stats_kernel(const DevCfg d, unsigned long long* stats, int n_profiles, int in_smem) {
  extern __shared__ unsigned long long s_acc[];   /* [P][4][S] */
  const int S = d.S;
  unsigned long long* acc = in_smem ? s_acc : stats;
  if (in_smem) {
    for (int i = threadIdx.x; i < 4 * S * n_profiles; i += blockDim.x) s_acc[i] = 0;
    __syncthreads();
  }
  const size_t total = (size_t)d.n_cells * d.U * d.nb;   /* one entry per bearer */
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t cu = i / d.nb;
    const int pf = d.cell_profile ? d.cell_profile[cu / d.U] : 0;
    const int s = d.ue_to_slice[(size_t)pf * d.U + cu % d.U];
    unsigned long long* row = acc + (size_t)pf * 4 * S;
    const unsigned long long by = d.cum_bytes[i], rb = d.cum_rbs[i], q = by >> 10;
    atomicAdd(&row[0 * S + s], by);
    atomicAdd(&row[1 * S + s], rb);
    atomicAdd(&row[2 * S + s], q);
    atomicAdd(&row[3 * S + s], q * q);
  }
  if (in_smem) {
    __syncthreads();
    for (int i = threadIdx.x; i < 4 * S * n_profiles; i += blockDim.x)
      if (s_acc[i]) atomicAdd(&stats[i], s_acc[i]);
  }
}

/* ---- per-slice buffer totals: uint64 [P][3][S] += { queued, dropped, records } over the bearers with a FIFO ---- */
/* Same row and shared-memory rules as rs_stats_kernel; meta [B][U][nb] (BufMeta::n < 0: backlogged, adds nothing). */
__global__ void rs_buffer_stats_kernel(const BufMeta* meta, const DevCfg d, unsigned long long* stats, int n_profiles,
                                       int in_smem) {
  extern __shared__ unsigned long long s_acc[];   /* [P][3][S] */
  const int S = d.S;
  unsigned long long* acc = in_smem ? s_acc : stats;
  if (in_smem) {
    for (int i = threadIdx.x; i < 3 * S * n_profiles; i += blockDim.x) s_acc[i] = 0;
    __syncthreads();
  }
  const size_t total = (size_t)d.n_cells * d.U * d.nb;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const BufMeta m = meta[i];
    if (m.n < 0) continue;   /* backlogged: no FIFO */
    const size_t cu = i / d.nb;
    const int pf = d.cell_profile ? d.cell_profile[cu / d.U] : 0;
    const int s = d.ue_to_slice[(size_t)pf * d.U + cu % d.U];
    unsigned long long* row = acc + (size_t)pf * 3 * S;
    if (m.queued) atomicAdd(&row[0 * S + s], (unsigned long long)m.queued);
    if (m.dropped) atomicAdd(&row[1 * S + s], m.dropped);
    if (m.n) atomicAdd(&row[2 * S + s], (unsigned long long)m.n);
  }
  if (in_smem) {
    __syncthreads();
    for (int i = threadIdx.x; i < 3 * S * n_profiles; i += blockDim.x)
      if (s_acc[i]) atomicAdd(&stats[i], s_acc[i]);
  }
}

#endif  /* RS_CORE_ONLY */

}  // namespace RS_NS
