/* include/rs_sched.h -- C ABI of the B200-native downlink RBG scheduler.
 *
 * What this replaces.  RadioSaber has no FFI: its "plug-in surface" is the C++
 * virtual class PacketScheduler (src/protocolStack/mac/packet-scheduler/
 * packet-scheduler.h:51-174) whose DoSchedule()/RBsAllocation() an ENodeB calls
 * once per 1 ms TTI (src/device/ENodeB.cpp:438-460).  The four behaviours
 * reachable from the SingleCellWithI scenario are selected by id
 * (src/scenarios/single-cell-with-interference.h:94-118):
 *     1  DL_PF_PacketScheduler            downlink-packet-scheduler.cpp:179-331
 *     7  DownlinkNVSScheduler(cfg,false)  downlink-nvs-scheduler.cpp:94-142, 275-358
 *     8  DownlinkTransportScheduler(cfg,0) GreedyByRow   downlink-transport-scheduler.cpp:249-272
 *     9  DownlinkTransportScheduler(cfg,2) MaximizeCell  downlink-transport-scheduler.cpp:351-376
 *    10  DownlinkTransportScheduler(cfg,4) UpperBound    downlink-transport-scheduler.cpp:223-246
 *    11  DownlinkNVSScheduler(cfg,true)   downlink-nvs-scheduler.cpp:405-528 (300-sample non-greedy PF)
 *   101  DownlinkTransportScheduler(cfg,1) SubOpt            downlink-transport-scheduler.cpp:274-349
 *   103  DownlinkTransportScheduler(cfg,3) VogelApproximate  downlink-transport-scheduler.cpp:378-451
 *        (ENodeB::DLScheduler_SUBOPT / DLScheduler_VOGEL, ENodeB.cpp:363-379, have no id in the scenario:
 *        100 + the constructor's second argument)
 * This library is what a host-side subclass of PacketScheduler binds to (see
 * INTEGRATION.md and radiosaber_b200/host/rs_gpu_scheduler.h): every entry
 * point below takes plain pointers and sizes, returns an int status and never
 * throws.  One handle schedules a BATCH of independent cells (one CTA per
 * cell); n_cells = 1 is the in-simulator drop-in.
 *
 * There is no CPU fallback: every compute entry point needs a CUDA device and
 * fails with RS_ERR_CUDA otherwise.
 */
#ifndef RS_SCHED_H_
#define RS_SCHED_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RS_OK 0
#define RS_ERR_ARG 1          /* NULL / out-of-range argument */
#define RS_ERR_UNSUPPORTED 2  /* a configuration the kernels do not cover (message says which) */
#define RS_ERR_CUDA 3         /* CUDA runtime error (message has the CUDA string) */

#define RS_MAX_SLICES 64      /* (rbg,slice) packs into 6+6 bits of a sort entry */
#define RS_MAX_RBGS 64        /* one 64-bit RBG mask per UE; 512 RBs / 8 = 64 at 100 MHz */

/* Static description of the cells.  Mirrors what the reference's scheduler constructors read from the JSON slice
 * config (downlink-transport-scheduler.cpp:55-97, downlink-nvs-scheduler.cpp:46-87, dl-pf-packet-scheduler.cpp:39-57).
 * rs_create gives every cell of the batch the same one; rs_create_profiles takes several that differ in weight, params
 * and ue_to_slice only (a slice PROFILE) and names one per cell. */
typedef struct rs_config {
  int32_t algo;             /* 1 PF, 7 NVS, 8 Sequential, 9 RadioSaber, 10 UpperBound, 11 NVS non-greedy, 101 SubOpt, 103 Vogel */
  int32_t n_slices;         /* S  <= RS_MAX_SLICES */
  int32_t n_ues;            /* U; user j == UE id j (flows/application/Application.cpp:72-123).  1..32767 (user ids are
                               int16), and a cell's shared-memory layout must fit one CTA: some thousands of UEs,
                               fewer for ids 7 / 11 with big slices; else RS_ERR_UNSUPPORTED saying which */
  int32_t n_rbs;            /* 512 for 100 MHz (core/spectrum/bandwidth-manager.cpp:98-102) */
  int32_t rbg_size;         /* get_rbg_size(): 8 (utility/eesm-effective-sinr.h:82-103) */
  int32_t cqi_per_rb;       /* CQI layout per UE: 0 = u8 [G], one value per RBG; 1 = u8 [n_rbs], one per RB
                               (what ENodeB::UserEquipmentRecord::GetCQI holds); 2 = 4-bit [G/2], RBG 2k in the
                               low and 2k+1 in the high nibble of byte k (a CQI is 4 bits on the air) */
  int32_t data_to_transmit; /* bytes queued per bearer; 100000000 = infinite buffer
                               (downlink-transport-scheduler.cpp:123-125) */
  int32_t n_bearers;        /* bearers per UE: 0 or 1 = one (every shipped backlogged config); 2 = MAX_BEARERS
                               (packet-scheduler.h:31, `internet_flow: 2` in exp-customize-20slices/config.json): slot i
                               of a UE holds its bearer of priority i, which is also the order of the two in the eNB's
                               bearer container.  Per-bearer arrays (rates, byte counters, queues, delays) are then
                               [B][U][2], every run call needs rs_set_queues, and the kernels do what
                               SelectFlowsToSchedule / ComputeSchedulingMetric / DoStopSchedule do with two bearers
                               (downlink-transport-scheduler.cpp:115-146, 179-191, 683-711).  Every id but 1, which schedules
                               flows, not users: give it one user per bearer (same CQI row) instead */
  const double* weight;       /* [S] slice_weights_ */
  const int32_t* params;      /* [S][4] alpha,beta,epsilon,psi (SchedulerAlgoParam, packet-scheduler.h:31-49) */
  const int32_t* ue_to_slice; /* [U] user_to_slice_ */
  const int32_t* tbs_row_m1;  /* [27] TransportBlockSizeTable[-1][*] as the reference's -O0 build reads it
                                 (AMCModule.cpp:312-316); NULL = the values of the stock build */
} rs_config;

/* Host (or device, see each call) destinations for one TTI's results; NULL = not wanted. */
typedef struct rs_outputs {
  int16_t* rbg_to_ue;    /* [B][G] winner UE id, -1 = RBG left unallocated
                            (GetListOfAllocatedRBs, downlink-transport-scheduler.cpp:589-601) */
  int32_t* tbs_bits;     /* [B][U] UpdateAllocatedBits value, 0 if unscheduled (:659) */
  uint8_t* mcs;          /* [B][U] MCS of the PDCCH records (:661-668), 0xff if unscheduled */
  uint8_t* final_cqi;    /* [B][U] "final_cqi" of :649, 0 if unscheduled */
  int32_t* slice_target; /* [B][S] slice_target_rbs (ids 8/9, :463-500) */
  int32_t* slice_quota;  /* [B][S] slice_quota_rbgs (ids 8/9, :501-521) */
  int32_t* nvs_slice;    /* [B]    slice served this TTI (ids 7/11, downlink-nvs-scheduler.cpp:94-142) */
  /* id 10 (UpperBound, downlink-transport-scheduler.cpp:223-246, 603-616) grants an RBG to every slice that
   * ranks it among its own best quota RBGs, so the grants are a list: slice-major, each slice's grants in
   * the order of its std::sort (the order the RBs are appended to the winners' lists).  For id 10
   * rbg_to_ue[g] is the highest user id holding RBG g.  The slices can make up to S*G grants; every one is
   * scheduled (RB lists, TBS, counters, slice offsets).  The list arrays hold L = rs_grant_list_len(h) entries per
   * cell (default 2G): grants past L are left out of the list only, and alloc_n still counts them. */
  int32_t* alloc_n;      /* [B]     number of (user, RBG) grants, all of them */
  int16_t* alloc_ue;     /* [B][L]  user of grant e, -1 past alloc_n (or no listed user of the slice on that RBG) */
  int16_t* alloc_rbg;    /* [B][L]  RBG of grant e */
} rs_outputs;

typedef struct rs_handle rs_handle;

/* Message of the last failing call on this thread ("" if none). */
const char* rs_last_error(void);
/* Library/ABI version, bumped when a signature changes. */
int32_t rs_abi_version(void);

/* Replaces the scheduler constructors (ENodeB::SetDLScheduler, ENodeB.cpp:302-391).
 * Allocates device state for n_cells cells on CUDA device `device` and sets it
 * to the reference's initial values (average rate 100000.0, radio-bearer.cpp:54;
 * offsets / NVS credits / byte counters 0). */
int rs_create(const rs_config* cfg, int32_t n_cells, int32_t device, rs_handle** out);
/* Cells with different slice configurations in one batch.  cfgs [n_profiles]: profiles may differ in weight, params and
 * ue_to_slice; every other field (algo, n_slices, n_ues, n_rbs, rbg_size, cqi_per_rb, data_to_transmit, n_bearers and
 * the values of tbs_row_m1) must be the same, else RS_ERR_ARG names the field and the profile.  cell_profile: HOST int32
 * [n_cells], the profile of each cell, values 0..n_profiles-1; NULL only with one profile.  1 <= n_profiles <= n_cells.
 * Cell b is scheduled exactly as a one-profile handle of profile cell_profile[b] schedules it.  rs_create(cfg, ...) is
 * rs_create_profiles(cfg, 1, NULL, ...). */
int rs_create_profiles(const rs_config* cfgs, int32_t n_profiles, const int32_t* cell_profile, int32_t n_cells,
                       int32_t device, rs_handle** out);
/* A new profile for every cell (HOST int32 [B] as in rs_create_profiles).  Synchronous: waits for the handle's work in
 * flight, rs_run_*_async calls included.  The cells' state (rates, offsets / NVS credits, counters) stays as it is. */
int rs_set_cell_profiles(rs_handle* h, const int32_t* cell_profile);
int32_t rs_n_profiles(const rs_handle* h);
void rs_destroy(rs_handle* h);
/* Id 10: entries per cell of the alloc_ue / alloc_rbg outputs, 2G (the default) .. max(S*G, 2G); S*G holds every grant.
 * Only the list changes, never the schedule.  Synchronous: waits for the handle's work in flight.  RS_ERR_ARG for
 * other ids or a length outside the range.  rs_grant_list_len: the current length (0 for other ids). */
int rs_set_grant_list_len(rs_handle* h, int32_t n);
int32_t rs_grant_list_len(const rs_handle* h);

/* Use an existing CUDA stream (a cudaStream_t passed as void*); NULL = the handle's own. */
int rs_set_stream(rs_handle* h, void* cuda_stream);
/* The cudaStream_t (as void*) the handle launches its kernels on. */
void* rs_get_stream(rs_handle* h);
/* Waits for everything the handle has enqueued (kernels and the copies of the *_host calls). */
int rs_sync(rs_handle* h);

/* Page-locked host memory for the buffers of the *_host calls (cudaHostAlloc, portable; write_combined != 0 for
 * buffers the CPU only writes, such as the CQI and rand() inputs).  A process that pins itself to the cores next
 * to its GPU before calling this gets the pages from that NUMA node (first touch). */
int rs_host_alloc(size_t bytes, int32_t write_combined, void** out);
void rs_host_free(void* p);

/* Per-bearer / per-slice state the reference keeps between TTIs (flows/radio-bearer.h:81-85,
 * downlink-transport-scheduler.h:38, downlink-nvs-scheduler.h:38).  Host arrays, [B][U] ([B][U][2] with two
 * bearers per UE) / [B][S]; NULL = leave alone / not wanted.  Synchronous. */
int rs_set_state(rs_handle* h, const double* avg_rate, const int32_t* tx_bytes, const uint64_t* cum_bytes,
                 const uint64_t* cum_rbs, const double* slice_offset, const double* nvs_ewma);
int rs_get_state(rs_handle* h, double* avg_rate, int32_t* tx_bytes, uint64_t* cum_bytes, uint64_t* cum_rbs,
                 double* slice_offset, double* nvs_ewma);
int rs_reset_state(rs_handle* h);

/* One TTI for the whole batch == PacketScheduler::Schedule() (packet-scheduler.cpp:72-90):
 * UpdateAverageTransmissionRate, SelectFlowsToSchedule, RBsAllocation and the byte accounting of
 * DoStopSchedule.  HOST buffers in, HOST buffers out, synchronous.
 *   cqi    [B][U][row] with row = G, n_rbs or G/2 bytes by cfg.cqi_per_rb, values 1..15
 *   rand2  [B][n]  the rand() values the scheduler draws this TTI, in call order, n =
 *                  rs_rand_draws_per_cell_tti(): ids 8/9 n = 2, the two draws of
 *                  downlink-transport-scheduler.cpp:490,511, each in [0, INT32_MAX - S]; id 11 n = 300 x the
 *                  largest slice, sample-major over the served slice's users
 *                  (downlink-nvs-scheduler.cpp:437-446 takes each value % 4); NULL for ids 1 and 7
 *   active [B][U]  1 = bearer has packets (GetDestination()->ACTIVE && HasPackets); NULL = all
 *   dt     Now - lastUpdate seen by RadioBearer::UpdateAverageTransmissionRate
 *          (radio-bearer.cpp:138-164); 0 skips the update like the reference does */
int rs_step(rs_handle* h, const uint8_t* cqi, const int32_t* rand2, const uint8_t* active, double dt,
            const rs_outputs* out);

/* rs_step for the in-simulator drop-in (n_cells = 1, but any batch works): the per-bearer and per-slice state the
 * reference keeps in ITS objects goes up with the TTI's inputs and comes back with the results, in one
 * host-to-device copy, one launch, one device-to-host copy and one synchronisation (rs_set_state + rs_set_queues +
 * rs_step + rs_get_state cost four round trips).  Replaces DownlinkTransportScheduler::RBsAllocation
 * (downlink-transport-scheduler.cpp:453-675) / DownlinkNVSScheduler::RBsAllocation (downlink-nvs-scheduler.cpp:
 * 275-358) / DownlinkPacketScheduler::RBsAllocation (downlink-packet-scheduler.cpp:179-331) as called once per TTI
 * from PacketScheduler::Schedule (packet-scheduler.cpp:72-90).  HOST pointers, synchronous. */
typedef struct rs_cell_io {
  double* avg_rate;           /* [B][U] in/out: m_averageTransmissionRate of each user's bearer(s), radio-bearer.cpp:138-164;
                                 NULL = the handle's own state */
  double* slice_state;        /* [B][S] in/out: slice_rbs_offset_ (ids 8/9/10/101/103, :618-620) or slice_ewma_time_
                                 (ids 7/11, downlink-nvs-scheduler.cpp:128-140); NULL = the handle's own */
  const uint8_t* cqi;         /* as rs_step */
  const int32_t* rand2;       /* as rs_step */
  const uint8_t* active;      /* as rs_step, may be NULL */
  const int32_t* queue_bytes; /* [B][U] as rs_set_queues (one TTI), may be NULL */
  const double* hol_delay;    /* [B][U] as rs_set_queues (one TTI), may be NULL */
  double dt;                  /* as rs_step */
  rs_outputs out;             /* as rs_step */
} rs_cell_io;
int rs_step_cell(rs_handle* h, const rs_cell_io* io);

/* Queue state for the NEXT rs_step / rs_run_* call on this handle (consumed by it): what the reference reads from
 * its bearers each TTI (SURVEY.md section 8 f3; one bearer per UE).
 *   queue_bytes [T][B][U] int32   ([T][B][U][2] with two bearers per UE, here and below) dataToTransmit of each UE's bearer (downlink-transport-scheduler.cpp:119-128):
 *                                 0 = no packets, the bearer is not listed this TTI; 100000000 = infinite buffer;
 *                                 else the queue size (values above 2^28-1 count as 2^28-1 where the reference
 *                                 multiplies by 8 in an int; negative = not listed).  Replaces cfg.data_to_transmit: bytes sent are capped by it
 *                                 (:183-186), id 7 stops granting a user RBGs at m_requiredRBs
 *                                 (packet-scheduler.cpp:321-334, downlink-nvs-scheduler.cpp:299-300), id 1 drops a
 *                                 flow once its TBS covers the queue (downlink-packet-scheduler.cpp:264-269)
 *   hol_delay   [T][B][U] double  RadioBearer::GetHeadOfLinePacketDelay(); multiplied into the metric of slices with
 *                                 alpha and beta set (ids 8/9/10, :702-706) or alpha set (id 7,
 *                                 downlink-nvs-scheduler.cpp:384-386); NULL = 0.  A caller that folds two bearers
 *                                 of a UE into one entry (the LTE-Sim plug-in) marks "the bearer of the slice's
 *                                 priority is empty", which zeroes the metric (:696-698), with a delay of 0 where the
 *                                 delay is in the metric and with a NEGATIVE delay in alpha-without-beta slices
 * HOST pointers for rs_step / rs_run_host / rs_run_traces_host, DEVICE pointers for the *_device calls. */
int rs_set_queues(rs_handle* h, const int32_t* queue_bytes, const double* hol_delay);

/* n_ttis consecutive TTIs with every input and output already in DEVICE memory.
 *   d_cqi   [ceil(T/cqi_refresh)][B][U][row]: TTI t reads slab t / cqi_refresh (the reference refreshes
 *           CQI every 40 TTIs, enb-mac-entity.cc:38; the headline workload every TTI);
 *           cqi_tti_stride = bytes between slabs
 *   d_rand2 [T][B][n], n = rs_rand_draws_per_cell_tti()
 *   d_active [T][B][U] or NULL, active_tti_stride like cqi_tti_stride
 *   dt      HOST array [T]
 *   d_out   device pointers, arrays [T][B][...]; NULL members are skipped
 *   ttis_per_launch  TTIs handled by one kernel launch with the cell state held on chip
 *                    (<= 0: library default 16; at most 64: the TTIs' dt / trace rows ride in the kernel parameters)
 * Asynchronous on the handle's stream; rs_sync() waits. */
int rs_run_device(rs_handle* h, int32_t n_ttis, const uint8_t* d_cqi, int64_t cqi_tti_stride, int32_t cqi_refresh,
                  const int32_t* d_rand2, const uint8_t* d_active, int64_t active_tti_stride,
                  const double* dt, const rs_outputs* d_out, int32_t ttis_per_launch);

/* Same, HOST buffers in and out ([T][B][...]): the library moves them in chunks of ttis_per_launch TTIs (at most
 * 64; <= 0: library default) through a ring of device slots and overlaps the copies with the kernels on three
 * streams.  Page-locked buffers (rs_host_alloc) make the copies asynchronous.  Synchronous: returns when the
 * results are in `out`. */
int rs_run_host(rs_handle* h, int32_t n_ttis, const uint8_t* cqi, int32_t cqi_refresh, const int32_t* rand2,
                const uint8_t* active, const double* dt, const rs_outputs* out, int32_t ttis_per_launch);
/* The same call without the wait: everything is enqueued and *ticket names the call.  The slot ring stays in
 * flight from one call to the next, so the first copies of call n+1 overlap the last kernels of call n.  The
 * caller keeps every buffer of the call untouched until rs_wait(ticket) (or rs_sync) has returned; rs_wait
 * returns once the call's results are in its `out` buffers.  A run loop alternates two sets of buffers:
 *     rs_run_host_async(h, ..., bufs[k & 1], &t[k]);  if (k) { rs_wait(h, t[k-1]); consume(bufs[(k-1) & 1]); } */
int rs_run_host_async(rs_handle* h, int32_t n_ttis, const uint8_t* cqi, int32_t cqi_refresh, const int32_t* rand2,
                      const uint8_t* active, const double* dt, const rs_outputs* out, int32_t ttis_per_launch,
                      int64_t* ticket);
int rs_wait(rs_handle* h, int64_t ticket);

/* ---- trace-driven CQI ingest ---------------------------------------------------------------------
 * Replaces EnbMacEntity's USE_REAL_TRACE path (src/protocolStack/mac/enb-mac-entity.cc:42-56 and
 * 160-193): mapping.config gives every UE a trace, ue<trace>.log holds 475 CQI vectors, and each
 * CQI report (every CQI_INTERVAL = 40 ms) overwrites the UE record's CQI with line
 * (int)(Now*1000/40) % 475.  Here the traces live in HBM once (4-bit packed when the handle's
 * layout is 2: 158 x 476 x 32 B = 2.4 MB, L2-resident) and every (cell, UE) replays one of them, so a
 * trace-driven run streams no CQI at all.
 *
 * rs_parse_trace_file / rs_parse_mapping_file / rs_trace_row are host-only helpers (no GPU needed). */

/* out: uint8 [n_rows][n_rbs], the first n_rows lines x n_rbs integers of a ue<id>.log
 * (enb-mac-entity.cc:169-187). */
int rs_parse_trace_file(const char* path, int32_t n_rows, int32_t n_rbs, uint8_t* out);
/* out[k] = trace id on the k-th line of a mapping.config (the uid column is ignored, as in
 * enb-mac-entity.cc:48-55); at most cap entries are written, *n_out = number of lines.
 * UE u replays out[u % n] (:164). */
int rs_parse_mapping_file(const char* path, int32_t* out, int32_t cap, int32_t* n_out);
/* (int)(Now*1000/CQI_INTERVAL) % n_rows for a report received at simulator time now_seconds
 * (enb-mac-entity.cc:189-191). */
int32_t rs_trace_row(double now_seconds, int32_t n_rows);

/* traces   HOST uint8 [n_traces][n_rows][n_rbs], values 1..15 (what rs_parse_trace_file returns);
 *          converted to the handle's CQI layout (layouts 0 and 2 need one value per RBG, which
 *          holds for every shipped trace; otherwise RS_ERR_UNSUPPORTED asks for cqi_per_rb = 1)
 * ue_trace HOST int32 [B][U]: the trace each UE of each cell replays (the reference:
 *          mapping[u % n_map] for its single cell; a batch gives every cell its own mapping);
 *          -1 = a UE whose reports never reach the eNB: its record keeps the initial CQI 10. */
int rs_set_traces(rs_handle* h, const uint8_t* traces, int32_t n_traces, int32_t n_rows, const int32_t* ue_trace);

/* rs_run_device / rs_run_host with the CQI taken from the loaded traces.
 *   trace_row HOST int32 [T]: the trace line in force at TTI t for every UE (all UEs of a cell report
 *             in the same TTI: they receive the same downlink burst, phy/ue-lte-phy.cpp:215-232),
 *             i.e. rs_trace_row(time of the last report); -1 = no report yet (CQI 10 everywhere,
 *             ENodeB.cpp:207-217)
 * Everything else as in rs_run_device (device pointers, asynchronous) / rs_run_host (host pointers,
 * synchronous). */
int rs_run_traces_device(rs_handle* h, int32_t n_ttis, const int32_t* trace_row, const int32_t* d_rand2,
                         const uint8_t* d_active, int64_t active_tti_stride, const double* dt,
                         const rs_outputs* d_out, int32_t ttis_per_launch);
int rs_run_traces_host(rs_handle* h, int32_t n_ttis, const int32_t* trace_row, const int32_t* rand2,
                       const uint8_t* active, const double* dt, const rs_outputs* out, int32_t ttis_per_launch);
int rs_run_traces_host_async(rs_handle* h, int32_t n_ttis, const int32_t* trace_row, const int32_t* rand2,
                             const uint8_t* active, const double* dt, const rs_outputs* out, int32_t ttis_per_launch,
                             int64_t* ticket);

/* Synthetic workload of SURVEY.md section 8(d), generated on the device (bit-identical twin of
 * radiosaber_b200/workload.py): CQI i.i.d. from the cqi-traces-noise0 histogram, counter-based so
 * any (cell, epoch) shard can be produced on any GPU.  d_out: n_slabs slabs [B][U][row] in the handle's
 * CQI layout (0 or 2); slab j is the CQI of epoch epoch0 + j (epoch = tti / refresh). */
int rs_synth_cqi(rs_handle* h, uint64_t seed, int64_t cell0, int64_t epoch0, int32_t n_slabs, uint8_t* d_out);
/* d_out: int32 [n_ttis][B][n], n = max(2, rs_rand_draws_per_cell_tti()), values in [0, INT32_MAX - S]. */
int rs_synth_rand2(rs_handle* h, uint64_t seed, int64_t cell0, int64_t tti0, int32_t n_ttis, int32_t* d_out);

/* Per-slice totals over every cell of this handle (what the reference's plotters sum from the
 * stderr log, NSDI23-radiosaber-experiments/exp-customization/plot_throughput.py:26-56).
 * stats: uint64 [P][4][S] = { sum cumulative bytes, sum cumulative RBs, sum q, sum q*q } with
 * q = a UE's cumulative bytes >> 10 (integers, so any reduction order gives the same bits); row p sums the cells of
 * profile p with its ue_to_slice ([4][S] with one profile).
 * rs_stats_device writes DEVICE memory (feed it to an NCCL reduce; the buffer holds P x 4 x S uint64); rs_get_stats
 * copies to HOST. */
int rs_stats_device(rs_handle* h, uint64_t* d_stats);
int rs_get_stats(rs_handle* h, uint64_t* stats);

/* ---- log-compatible writer (host only, no GPU needed) ------------------------------------------
 * The reference's only "output format" is what its schedulers print each TTI and what the paper's
 * plotters parse (NSDI23-radiosaber-experiments/exp-customization/plot_throughput.py:35-47):
 *   stdout  "slice_id, target_rbs, quota_rbgs: (i, t, q) ..."   downlink-transport-scheduler.cpp:523-527
 *           "<ts>" and "User(<u>) allocated RBGS: <g>(<cqi>) ... final_cqi: <c>"   :631-649 (NVS :314-332)
 *   stderr  "all_bytes: <n>"                                     :366-374 (id 9), :265-270 (id 8)
 *           "<ts> app: <a> cumu_bytes: <b> cumu_rbs: <r> hol_delay: <d> user: <u> slice: <s>"
 *                                                                :192-199, nvs :244-251, dl-pf :89-96
 * An rs_log regenerates that text, byte for byte, for ONE cell of a batch from the results the device
 * path returns; it keeps the bearer's cumulative byte / RB counters itself.  <ts> is the scheduler's
 * TTI counter (PacketScheduler::m_ts, packet-scheduler.cpp:292-300: +1 per DoStopSchedule since the eNB
 * was created, so the first TTI with bearers of a SingleCellWithI run is 100). */
typedef struct rs_log rs_log;
/* cfg: the configuration of the logged cell -- with slice profiles (rs_create_profiles) that cell's own profile, whose
 * ue_to_slice names the slices in the log lines. */
int rs_log_create(const rs_config* cfg, rs_log** out);
void rs_log_destroy(rs_log* lg);
/* Per-bearer arrays of an rs_log are [U][nb] with nb = 2 when cfg->n_bearers == 2 (slot i = the bearer of priority i,
 * as in the device state), else [U].  Not for id 1 with two bearers (id 1 schedules flows: one user per bearer). */
int rs_log_set_counters(rs_log* lg, const uint64_t* cum_bytes /*[U][nb]*/, const uint64_t* cum_rbs /*[U][nb]*/);
int rs_log_get_counters(rs_log* lg, uint64_t* cum_bytes, uint64_t* cum_rbs);
/* Application id printed for every bearer ([U][nb]; < 0 = the UE has no such bearer).  Default: bearer u * nb + i is
 * application u * nb + i -- the ids SingleCellWithI hands out when every UE has nb flows
 * (single-cell-with-interference.h:411-426: applications are created UE by UE, flow by flow). */
int rs_log_set_app_ids(rs_log* lg, const int32_t* app_ids);
/* Queue state of the cell for the NEXT rs_log_tti (same meaning as rs_set_queues, [U][nb] each, either may be NULL):
 * bytes credited are capped by the queue and the hol_delay field prints the bearer's delay. */
int rs_log_set_queues(rs_log* lg, const int32_t* queue_bytes, const double* hol_delay);
/* Appends one TTI of one cell.  cqi [U][row] in cfg's CQI layout; rbg_to_ue [G]; tbs_bits [U];
 * final_cqi [U] (every id but 1); slice_target / slice_quota [S] (ids 8/9/101/103).  Not for id 10 (next call). */
int rs_log_tti(rs_log* lg, uint64_t timestamp, const uint8_t* cqi, const int16_t* rbg_to_ue, const int32_t* tbs_bits,
               const uint8_t* final_cqi, const int32_t* slice_target, const int32_t* slice_quota);
/* Id 10 (UpperBound, :223-246) books an RBG to several slices: its TTI is logged from the grant list the device
 * returns (rs_outputs.alloc_n / alloc_ue / alloc_rbg of that cell: slice by slice in the order the grants were made,
 * user -1 = a slice without a listed user on that RBG), which is the order of the users' RB lists and of the
 * efficiency sum behind "all_bytes".  grant_ue / grant_rbg hold n_grants entries, every grant of the TTI: set the
 * handle's list length (rs_set_grant_list_len) to S*G, or at least alloc_n, to log a TTI whole. */
int rs_log_tti_grants(rs_log* lg, uint64_t timestamp, const uint8_t* cqi, int32_t n_grants, const int16_t* grant_ue,
                      const int16_t* grant_rbg, const int32_t* tbs_bits, const uint8_t* final_cqi,
                      const int32_t* slice_target, const int32_t* slice_quota);
/* The text accumulated so far (NUL-terminated, owned by the log) and a reset. */
const char* rs_log_stdout(rs_log* lg, int64_t* len);
const char* rs_log_stderr(rs_log* lg, int64_t* len);
void rs_log_clear(rs_log* lg);

/* Introspection for benchmarks and tests. */
/* Shape of the batch behind a handle; any pointer may be NULL. */
int rs_dims(const rs_handle* h, int32_t* n_cells, int32_t* n_slices, int32_t* n_ues, int32_t* n_rbgs, int32_t* device);
int32_t rs_rand_draws_per_cell_tti(const rs_handle* h);   /* int32 values per cell in rand2 (0, 2 or 300 x largest slice
                                                             of any profile) */
int64_t rs_launch_count(const rs_handle* h);      /* kernels launched by this handle so far */
int32_t rs_smem_bytes(const rs_handle* h);        /* dynamic shared memory per CTA of the TTI kernel */
int32_t rs_threads_per_cta(const rs_handle* h);
/* >= 0: the handle's backlogged launches run a compile-time-shape instantiation of the TTI kernel (the headline cell,
 * 20 slices x 5 UEs x 64 RBGs); -1: the general kernel.  Same results either way. */
int32_t rs_fixed_shape(const rs_handle* h);
/* 1: big slices -- the per-slice argmax divides its metrics where it compares them instead of tabulating them per chunk of
 * slices (same doubles, same winners). */
int32_t rs_direct_metric(const rs_handle* h);
int64_t rs_algorithmic_bytes_per_cell_tti(const rs_handle* h); /* U(G+20)+16S+2G+8, SURVEY 8(d) */

/* Device test hook: libstdc++ std::sort order (key descending, comparator of
 * downlink-transport-scheduler.cpp:357-361) of n_arrays arrays of n 4-bit keys, computed by the same
 * device routine the RadioSaber path uses.  keys: HOST uint8 [n_arrays][n]; perm_out: HOST int32
 * [n_arrays][n], perm_out[i] = original index of the element ending at position i.
 * depth_limit < 0 = the library's 2*floor(log2 n). */
int rs_test_sort(int32_t device, const uint8_t* keys, int32_t n_arrays, int32_t n, int32_t depth_limit,
                 int32_t* perm_out);
/* Same, launched `reps` times; *ms_per_launch = mean device time of launches 2..reps (CUDA events). */
int rs_test_sort_timed(int32_t device, const uint8_t* keys, int32_t n_arrays, int32_t n, int32_t depth_limit,
                       int32_t* perm_out, int32_t reps, float* ms_per_launch);

#ifdef __cplusplus
}
#endif
#endif /* RS_SCHED_H_ */
