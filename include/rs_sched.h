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

/* ---- per-bearer buffers kept on the device (closed-loop queues) ----------------------------------
 * rs_set_queues feeds the queue-aware schedulers open loop: the caller says what every bearer holds at every TTI.
 * With buffers the handle keeps, per bearer (cell b, UE u, slot i = priority i), a FIFO of at most K records
 * (arrival time, bytes), the sum `queued` of their bytes and a `dropped` byte counter.  Arrivals are an input;
 * departures are what the scheduler books.  At TTI t of a call, in this order:
 *   1. arrival: a = arrivals[t][b][u][i] > 0 bytes are pushed as one record stamped arrival_time[t] (queued += a), or,
 *      when the FIFO already holds K records, refused whole (dropped += a); a <= 0: nothing arrives;
 *   2. what the scheduler sees, in place of rs_set_queues' values for the TTI: queue min(queued, INT32_MAX) (0 = the
 *      bearer is not listed) and HoL delay now[t] - (arrival time of the head record), 0 when the FIFO is empty;
 *   3. the TTI is scheduled exactly as with those values from rs_set_queues;
 *   4. departure: the bytes booked to the bearer (the increment of its cum_bytes), clamped to queued, leave from the
 *      head; emptied records are dropped, a record sent in part keeps its arrival time with its remaining bytes.
 * A bearer flagged backlogged has no FIFO: it shows queue 100000000 (the infinite buffer) and HoL 0 every TTI.
 * This is a byte FIFO: LTE-Sim's RLC segmentation and header bytes and its application models are not reproduced.
 * rs_step_cell refuses a buffered handle (inside LTE-Sim the simulator owns the queues). */

/* max_records = K, 1..RS_MAX_BUFFER_RECORDS, or 0 to switch the buffers off and free them.  backlogged: HOST uint8
 * [B][U][nb] (nb = 2 with two bearers per UE), nonzero = no FIFO; NULL = none.  Enabling (again) empties every FIFO.
 * Synchronous.  Memory: 24 + 12 K bytes of HBM per bearer. */
#define RS_MAX_BUFFER_RECORDS 65536
int rs_enable_buffers(rs_handle* h, int32_t max_records, const uint8_t* backlogged);

/* Traffic for the NEXT run call on a buffered handle (consumed by it, like rs_set_queues, which a buffered handle
 * refuses).  Every rs_step / rs_run_* call of a buffered handle needs one, with two bearers per UE too.
 *   arrivals     [T][B][U][nb] int32, bytes arriving at each bearer at TTI t (<= 0: none)
 *   now          HOST double [T], simulator time of TTI t; never decreases over the calls of the handle (rs_reset_state
 *                forgets the last one)
 *   arrival_time HOST double [T], the time stamped on the records TTI t pushes; <= now[t]
 *   queue_out    [T][B][U][nb] int32 or NULL: the queue sizes step 2 showed the scheduler
 *   hol_out      [T][B][U][nb] double or NULL: the head-of-line delays step 2 showed (never negative)
 * arrivals / queue_out / hol_out are HOST pointers for rs_step / rs_run_host* / rs_run_traces_host*, DEVICE pointers
 * for rs_run_device / rs_run_traces_device.  Bad times are RS_ERR_ARG before anything runs. */
typedef struct rs_traffic {
  const int32_t* arrivals;
  const double* now;
  const double* arrival_time;
  int32_t* queue_out;
  double* hol_out;
} rs_traffic;
int rs_set_traffic(rs_handle* h, const rs_traffic* traffic);

/* The buffers' state, HOST arrays [B][U][nb], NULL = not wanted: bytes queued, records held, arrival time of the head
 * record (0 when empty) and bytes dropped; a backlogged bearer reports 0 in each.  Synchronous: waits for the handle's
 * work in flight. */
int rs_get_buffers(rs_handle* h, int64_t* queued, int32_t* n_records, double* head_time, uint64_t* dropped);

/* Per-slice totals of the buffers, uint64 [P][3][S] = { sum queued bytes, sum dropped bytes, sum records held } over
 * the bearers with a FIFO (both slots with two bearers per UE; backlogged bearers add 0).  Row p sums the cells of
 * profile p with its ue_to_slice, as rs_stats_device does; integers, so any reduction order gives the same bits.
 * rs_buffer_stats_device writes DEVICE memory (P x 3 x S uint64; feed it to an NCCL reduce, rs_reduce_buffer_stats);
 * rs_get_buffer_stats copies to HOST.  Both are ordered after the handle's earlier work on its stream, like
 * rs_stats_device.  RS_ERR_ARG on a handle without buffers. */
int rs_buffer_stats_device(rs_handle* h, uint64_t* d_stats);
int rs_get_buffer_stats(rs_handle* h, uint64_t* stats);

/* ---- head-of-line delay histograms of a buffered handle ---------------------------------------------
 * With the histogram on, every TTI of every run call (rs_step, rs_run_host(_async), rs_run_device,
 * rs_run_traces_host(_async), rs_run_traces_device) adds samples; the caller changes nothing else.  Only bearers with
 * a FIFO count (backlogged bearers add nothing, as in rs_get_buffer_stats).  With q the queue and h the HoL delay step 2
 * showed the scheduler at that TTI (what queue_out / hol_out receive):
 *   row 0, served   one sample per bearer that sends this TTI, by the rule of rs_log_tti's stderr loop (the reference's
 *                   DoStopSchedule lines): avail = tbs_bits[u] / 8; slots from priority nb-1 down to 0; a slot with
 *                   q <= 0 is skipped (ids other than 1); sent = min(avail, q) (id 1: avail), avail -= sent; the loop
 *                   stops when avail <= 0.  These are the samples of the reference's hol_delay lines, for every cell.
 *   row 1, waiting  one sample per bearer with q > 0, served or not: the time-average view, starved bearers included.
 *   bin             d = floor(h * bins_per_unit + 0.5), a product and a sum each rounded to double (no FMA), then
 *                   min(d, n_bins - 1): the last bin holds every delay of at least n_bins - 1 bins.  With a clock in
 *                   seconds, bins_per_unit = 1000 makes 1-TTI bins.
 *   storage         uint64 [P][2][S][n_bins]; row p sums the cells of profile p, mapped to slices by that profile's
 *                   ue_to_slice, as rs_stats_device does.  Integers, so any order of accumulation gives the same bits.
 * The counts come from a reduction kernel launched after each TTI-kernel launch on the same stream; the schedules,
 * state and buffers are the same bits with the histogram on and off.
 *
 * rs_enable_hol_hist: n_bins 1..RS_MAX_HOL_BINS, or 0 to switch the histogram off and free it; bins_per_unit finite
 * and > 0.  RS_ERR_ARG on a handle without buffers, with 2^30 or more UEs (B x U), or with a [P][2][S][n_bins] block
 * over 2 GiB.  Enabling (again) zeroes the counts, and only that does (rs_reset_state leaves them); rs_enable_buffers
 * (again, or with 0) switches the histogram off.  Synchronous.  rs_hol_hist_bins: n_bins, 0 when off.
 * rs_hol_hist_device writes DEVICE memory (P x 2 x S x n_bins uint64; feed it to an NCCL reduce, rs_reduce_hol_hist);
 * rs_get_hol_hist copies to HOST.  Both are ordered after the handle's earlier work on its stream, like
 * rs_buffer_stats_device; RS_ERR_ARG on a handle without the histogram. */
#define RS_MAX_HOL_BINS 65536
int rs_enable_hol_hist(rs_handle* h, int32_t n_bins, double bins_per_unit);
int32_t rs_hol_hist_bins(const rs_handle* h);
int rs_hol_hist_device(rs_handle* h, uint64_t* d_hist);
int rs_get_hol_hist(rs_handle* h, uint64_t* hist);

/* ---- per-UE throughput histograms over caller-closed windows (any handle) ---------------------------------------
 * The spread of the bytes a slice's UEs receive, cell-edge tail included, summarised on the device window by window.
 * Every handle: backlogged or buffered, any CQI source, every id.  The caller closes each window; integers throughout:
 *   UE bytes        c(b,u) = sum of cum_bytes[b][u][i] over the UE's slots (one, or two with n_bearers = 2), mod 2^64.
 *   snapshot        snap[b][u], uint64 [B][U] in device memory: each UE's c when its open window started.
 *   closing         every UE of every cell adds one sample, backlogged, buffered, idle or inactive alike:
 *                   d = c(b,u) - snap[b][u] (mod 2^64), bin = min(d / bin_bytes, n_bins - 1) (integer division: the
 *                   last bin holds every UE with at least (n_bins - 1) x bin_bytes bytes), then snap[b][u] := c(b,u).
 *                   Two closes with no TTI between them add a bin-0 sample per UE.
 *   row             [p][s]: p = the cell's profile when the window closes (so rs_set_cell_profiles between windows moves
 *                   later samples), s = that profile's ue_to_slice[u], as rs_stats_device maps them.
 *   storage         uint64 [P][S][n_bins]; any order of accumulation gives the same bits.
 *   restarts        rs_reset_state zeroes the counters and sets snap := 0; rs_set_state with a non-NULL cum_bytes sets
 *                   snap := the new counters.  Nothing else moves the snapshot (run calls, rs_step_cell,
 *                   rs_enable_buffers, rs_set_cell_profiles leave it).
 * The schedules, state and buffers are the same bits with the histogram on and off: nothing runs per TTI.
 *
 * rs_enable_ue_rate_hist: n_bins 1..RS_MAX_UE_RATE_BINS, or 0 to switch the histogram off and free it; bin_bytes >= 1.
 * RS_ERR_ARG with 2^30 or more UEs (B x U) or a [P][S][n_bins] block over 2 GiB (32-bit per-CTA counters and
 * indices).  Synchronous: waits for the work in flight, zeroes the counts and takes the snapshot, the first window
 * starting there (warm-up before it is not counted); enabling again does the same.
 * rs_close_ue_rate_window: one kernel on the handle's stream, asynchronous, ordered after the handle's earlier work as
 * rs_stats_device is (the join of a split batch's part streams, the kernels of an rs_run_host_async /
 * rs_run_traces_host_async call not yet waited for).  rs_ue_rate_hist_bins: n_bins, 0 when off.
 * rs_ue_rate_hist_device writes DEVICE memory (P x S x n_bins uint64; feed it to an NCCL reduce,
 * rs_reduce_ue_rate_hist); rs_get_ue_rate_hist copies to HOST; both ordered like rs_hol_hist_device.  Every call but
 * rs_enable_ue_rate_hist returns RS_ERR_ARG on a handle without the histogram. */
#define RS_MAX_UE_RATE_BINS 65536
int rs_enable_ue_rate_hist(rs_handle* h, int32_t n_bins, int64_t bin_bytes);
int rs_close_ue_rate_window(rs_handle* h);
int32_t rs_ue_rate_hist_bins(const rs_handle* h);
int rs_ue_rate_hist_device(rs_handle* h, uint64_t* d_hist);
int rs_get_ue_rate_hist(rs_handle* h, uint64_t* hist);

/* ---- per-UE throughput over active time (UPT) histograms of a buffered handle ------------------------------------
 * The bytes a UE received over a window divided by the TTIs it had data waiting: the service a bursty bearer got,
 * where the throughput histogram above bins its offered load.  It rides on the throughput histogram's windows and
 * snapshot (rs_close_ue_rate_window closes both); integers throughout:
 *   active TTI      UE (b,u) is active at TTI t iff one of its slots showed q > 0 at step 2 of that TTI (what
 *                   queue_out receives: after the TTI's arrival, before its departure).  A backlogged slot shows
 *                   100 000 000, so a UE with one is active every TTI; a packet that arrives and leaves in the same TTI
 *                   makes one active TTI; the run calls' `active` flags play no part.
 *   active counts   n_a[b][u], uint32 [B][U] in device memory, the UE's active TTIs in the open window; a window must
 *                   be shorter than 2^32 TTIs (not checked).
 *   closing         d = c(b,u) - snap[b][u] (mod 2^64) as the throughput histogram takes it, before it moves snap;
 *                   a UE with n_a > 0 adds one sample, bin = min((d / n_a) / bin_bytes, n_bins - 1) (two integer
 *                   divisions, bin_bytes in bytes per TTI); a UE with n_a = 0 adds none; then n_a := 0.
 *   bytes           the booked bytes (cum_bytes), as in every throughput this library reports: id 1 books its TBS
 *                   uncapped, so with finite queues its bytes can exceed what left the FIFO, and so can its UPT.
 *   row, storage    as the throughput histogram: [profile at close][that profile's slice], uint64 [P][S][n_bins].
 *   restarts        rs_reset_state, rs_set_state with a non-NULL cum_bytes and rs_enable_ue_upt_hist zero n_a along
 *                   with the snapshot change they make.
 *   switching off   any rs_enable_ue_rate_hist call and rs_enable_buffers (again, or with 0); nothing else (run calls
 *                   and rs_set_cell_profiles leave it).
 * The counts come from a kernel launched after each TTI-kernel launch on the same stream; the schedules, state,
 * buffers and the other histograms are the same bits with UPT on and off.
 *
 * rs_enable_ue_upt_hist: n_bins 1..RS_MAX_UE_RATE_BINS, or 0 to switch UPT off and free it; bin_bytes >= 1.
 * RS_ERR_ARG on a handle without buffers, without the throughput histogram, or with a [P][S][n_bins] block over 2 GiB.
 * Synchronous: waits for the work in flight, zeroes the counts and n_a and retakes the snapshot, which restarts the
 * open window of both histograms (it adds no throughput samples and clears none).  rs_ue_upt_hist_bins: n_bins, 0 when
 * off.  rs_ue_upt_hist_device writes DEVICE memory (P x S x n_bins uint64; feed it to an NCCL reduce,
 * rs_reduce_ue_upt_hist); rs_get_ue_upt_hist copies to HOST; both ordered like rs_ue_rate_hist_device.  Every call but
 * rs_enable_ue_upt_hist returns RS_ERR_ARG when UPT is off. */
int rs_enable_ue_upt_hist(rs_handle* h, int32_t n_bins, int64_t bin_bytes);
int32_t rs_ue_upt_hist_bins(const rs_handle* h);
int rs_ue_upt_hist_device(rs_handle* h, uint64_t* d_hist);
int rs_get_ue_upt_hist(rs_handle* h, uint64_t* hist);

/* Synthetic arrivals into DEVICE int32 [n_ttis][B][U][nb] (bit-identical twin of radiosaber_b200/workload.py
 * synth_arrivals): pkt_bytes and pkts_q16 are HOST int32 [P][S] (P = rs_n_profiles; cell b reads the row of its
 * profile).  A bearer of slice s gets (q >> 16) + (draw16 < (q & 0xffff)) packets of pkt_bytes[s] bytes per TTI with
 * q = pkts_q16[s] (packets per TTI in 16.16 fixed point), draw16 the top 16 bits of splitmix64 of a counter over
 * (cell0 + b, tti0 + t, u, slot) built like rs_synth_cqi's.  pkt_bytes 0 = no arrivals.  Asynchronous on the handle's
 * stream. */
int rs_synth_arrivals(rs_handle* h, uint64_t seed, int64_t cell0, int64_t tti0, int32_t n_ttis, const int32_t* pkt_bytes,
                      const int32_t* pkts_q16, int32_t* d_out);
/* One slice's arrival spec for rs_synth_arrivals from a packet size and a mean rate in packets per TTI, as a traffic
 * file gives them (host only, no GPU needed; rs_batch and radiosaber_b200/sched.py load_traffic_config both use it).
 * *pkts_q16 = pkts_per_tti * 65536 rounded to the nearest integer (halves away from zero).  RS_ERR_ARG, with the
 * reason in rs_last_error, unless pkt_bytes is an integer 0..INT32_MAX, pkts_per_tti is finite and >= 0, a positive
 * rate is at least 1/65536 packet per TTI, and a TTI's most bytes, pkt_bytes x ((q >> 16) + 1), fit int32. */
int rs_arrival_spec(double pkt_bytes, double pkts_per_tti, int32_t* pkt_bytes_out, int32_t* pkts_q16);

/* ---- traffic sources drawn on the device -----------------------------------------------------------
 * Generic traffic models, parameters given by the caller: periodic frames (video-like) and on-off packet sources
 * (talk-spurt-like) next to rs_synth_arrivals' smooth rate.  They are NOT LTE-Sim's VoIP, TraceBased or InternetFlow
 * applications, and the slice config's traffic fields are not read.
 * A source is set per (profile, slice); every bearer of the slice (both slots with two bearers per UE) runs its own
 * copy.  Global TTI tau = tti0 + t and global cell = cell0 + b, as in rs_synth_arrivals, so N GPUs drawing their shards
 * of the cells draw exactly what one GPU draws.
 *   per-TTI draw     one 64-bit draw per (tau, cell, ue, slot): rs_synth_arrivals' counter and key.  RATE uses its top
 *                    16 bits, unchanged; ONOFF compares its low 32 bits with the leaving probability of its state.
 *   per-bearer draw  one 64-bit draw per (cell, ue, slot) under its own key ("SRC\0"), no tau in the counter.  It gives
 *                    the phase phi = (draw >> 32) % period_ttis (PERIODIC, ONOFF: the bearers of a cell do not all
 *                    burst in the same TTI), the start frame f0 = low32 % n_frames (PERIODIC) and the initial ONOFF
 *                    state: ON iff low32 < (uint64(leave_off_q32) << 32) / (leave_on_q32 + leave_off_q32), the
 *                    stationary distribution in integers.
 *   RATE             exactly rs_synth_arrivals: pkt_bytes x ((q >> 16) + (draw16 < (q & 0xffff))), q = pkts_q16.
 *   PERIODIC         a frame arrives at tau iff (tau + phi) % period_ttis == 0, of frame_bytes[((tau + phi) /
 *                    period_ttis + f0) % n_frames] bytes, pushed as one record (a buffer sends it in parts and keeps
 *                    its arrival time, so its head-of-line delay is the frame's own).
 *   ONOFF            at tau the chain steps first: it leaves its state iff low32 < leave_on_q32 (ON) / leave_off_q32
 *                    (OFF); then, if ON and (tau + phi) % period_ttis == 0, pkt_bytes arrive.
 * ONOFF is the only kind with state: one byte per bearer in HBM, owned by the handle.  rs_set_sources (again) resets
 * every chain to its initial draw; the first rs_synth_traffic call after it may start at any tti0 >= 0, each later call
 * must continue the chain: tti0 = the previous call's tti0 + n_ttis, with the same seed and cell0, else RS_ERR_ARG.
 * So one 64-TTI call draws exactly what four 16-TTI calls draw. */
#define RS_SRC_NONE 0      /* no arrivals (backlogged slices, or a silent slice) */
#define RS_SRC_RATE 1      /* exactly rs_synth_arrivals: pkt_bytes x ((q >> 16) + (draw16 < (q & 0xffff))) */
#define RS_SRC_PERIODIC 2  /* one frame every period_ttis TTIs; frame sizes cycle through frame_bytes[n_frames] */
#define RS_SRC_ONOFF 3     /* two-state Markov chain; while ON one pkt_bytes packet every period_ttis TTIs */
#define RS_MAX_FRAMES 1024
typedef struct rs_source {
  int32_t kind;
  int32_t pkt_bytes;            /* RATE: 0..INT32_MAX; ONOFF: 1..INT32_MAX */
  int32_t pkts_q16;             /* RATE: packets per TTI, 16.16 (rs_arrival_spec) */
  int32_t period_ttis;          /* PERIODIC, ONOFF: >= 1 */
  uint32_t leave_on_q32;        /* ONOFF: per-TTI probability of leaving ON, 0.32 fixed point (rs_onoff_spec), >= 1 */
  uint32_t leave_off_q32;       /* ONOFF: per-TTI probability of leaving OFF, >= 1 */
  int32_t n_frames;             /* PERIODIC: 1..RS_MAX_FRAMES */
  const int32_t* frame_bytes;   /* PERIODIC: HOST [n_frames], each 1..INT32_MAX; copied by rs_set_sources */
} rs_source;
/* The handle's sources, src HOST [P][S] (P = rs_n_profiles; cell b uses the row of its profile).  Every entry is
 * checked first (kind, sizes, period, frames, leaving probabilities, RATE's int32 rule of rs_synth_arrivals): RS_ERR_ARG
 * names the profile and slice of the first bad one and nothing changes.  Fields a kind does not use are ignored.
 * Ordered on the handle's stream like the generator; rs_synth_arrivals never touches these sources. */
int rs_set_sources(rs_handle* h, const rs_source* src);
/* Arrivals of the sources into DEVICE int32 [n_ttis][B][U][nb], exactly what rs_set_traffic takes.  Asynchronous on the
 * handle's stream.  RS_ERR_ARG without rs_set_sources, for tti0 < 0, or for a call that does not continue the chain. */
int rs_synth_traffic(rs_handle* h, uint64_t seed, int64_t cell0, int64_t tti0, int32_t n_ttis, int32_t* d_out);
/* ONOFF leaving probabilities from mean ON and OFF run lengths in TTIs (host only, no GPU needed; rs_batch and
 * radiosaber_b200/sched.py onoff_spec both use it): q = 2^32 / mean rounded to the nearest integer (halves away from
 * zero).  RS_ERR_ARG, with the reason in rs_last_error, unless each mean is finite and in [2, 2^32]. */
int rs_onoff_spec(double on_ttis, double off_ttis, uint32_t* leave_on_q32, uint32_t* leave_off_q32);

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

/* ---- synthetic channel drawn on the device ---------------------------------------------------------
 * CQI with the structure rs_synth_cqi lacks: a per-UE level (cell-centre or cell-edge UEs) and an offset that is
 * correlated across RBGs and across epochs.  A generic model with caller-given parameters, set per (profile, slice);
 * every UE of the slice runs its own realisation.  Global cell = cell0 + b and epoch e = epoch0 + j, as in
 * rs_synth_cqi: slab j holds epoch epoch0 + j, and the consumer's cqi_refresh maps TTIs to slabs.  Stateless in the
 * epoch: any (cell range, epoch range) can be drawn on its own, in any chunking, on any GPU.
 *   RS_CH_IID     exactly rs_synth_cqi's value for that (cell, epoch, UE, RBG): same key, counter and thresholds, so a
 *                 handle whose channels are all IID writes byte for byte what rs_synth_cqi writes.
 *   RS_CH_FADING  cqi = clamp(L + offset(g, e), 1, 15) at RBG g of epoch e, integers only:
 *     draws       per (cell, UE) 17 splitmix64 draws under the key ("CHN\0"), counter (cell << 20) ^ (ue << 8) ^ i ^
 *                 ((ue >> 12) * 0xD6E8FEB86659FD93), i = 0..16;  hi(i) / lo(i) = the draw's top / low 32 bits.
 *     level       L = 1 + #{k : hi(0) >= level_thr[k]}, fixed for the run.
 *     paths       K = 8; path k has phase theta_k = hi(1 + k), RBG slope omega_k = slope(lo(1 + k), W_f) and epoch
 *                 slope nu_k = slope(hi(9 + k), W_t), in phase units (2^32 = one turn), where slope(r, W) =
 *                 uint32((uint64(r) * (2W + 1)) >> 32) - W is uniform over [-W, W], W_f = floor(2^31 / coherence_rbgs),
 *                 W_t = floor(2^31 / coherence_epochs), and a coherence of 0 gives W = 0: flat across RBGs, or frozen.
 *     offset      x = sum_k cos_q14[(theta_k + g * omega_k + uint32(e) * nu_k) >> 22] (uint32 arithmetic; cos_q14 =
 *                 include/rs_cos_q14.inc, round(16384 cos(2 pi i / 1024))); offset = (x * depth_q8 + 2^22) >> 23
 *                 (arithmetic shift).  x has standard deviation 2^15, so the offset's is depth_q8 / 256 CQI steps.
 *     correlation Before rounding and clamping the offset's autocorrelation is sinc(pi dg / coherence_rbgs) x sinc(pi de /
 *                 coherence_epochs) (sinc(y) = sin(y) / y): offsets one coherence length apart are uncorrelated.
 * Not a 3GPP TDL/CDL model nor LTE-Sim's path-loss / shadowing / fast-fading tables; L does not move with mobility. */
#define RS_CH_IID 0
#define RS_CH_FADING 1
typedef struct rs_channel {
  int32_t kind;
  uint32_t level_thr[14];     /* FADING: non-decreasing thresholds on a 32-bit draw (rs_channel_spec) */
  int32_t depth_q8;           /* FADING: offset standard deviation in CQI steps, 8.8 fixed point, 0..15 x 256 */
  int32_t coherence_rbgs;     /* FADING: >= 0, 0 = flat across RBGs */
  int32_t coherence_epochs;   /* FADING: >= 0, 0 = frozen in time */
} rs_channel;
/* The handle's channels, ch HOST [P][S] (P = rs_n_profiles; cell b uses the row of its profile).  Every entry is checked
 * first (kind, thresholds, depth, coherences): RS_ERR_ARG names the profile and slice of the first bad one and nothing
 * changes.  Fields IID does not use are ignored.  Ordered on the handle's stream like rs_set_sources. */
int rs_set_channels(rs_handle* h, const rs_channel* ch);
/* n_slabs slabs [B][U][row] of the channels' CQI into DEVICE d_out, in the handle's CQI layout (0, or 2: 4-bit packed;
 * layout 1 is RS_ERR_UNSUPPORTED as in rs_synth_cqi).  Asynchronous on the handle's stream.  RS_ERR_ARG without
 * rs_set_channels. */
int rs_synth_channel(rs_handle* h, uint64_t seed, int64_t cell0, int64_t epoch0, int32_t n_slabs, uint8_t* d_out);
/* A FADING channel from a level histogram and the offset's spread and coherences (host only, no GPU needed; rs_batch and
 * radiosaber_b200/sched.py channel_spec both use it).  level_counts [15]: integer counts of levels 1..15, total 1..2^32-1;
 * level_thr[k] = min((cum_k << 32) / total, 2^32 - 1) with cum_k = the counts of levels 1..k+1 (so a level above the
 * last counted one has probability at most 2^-32).  depth_q8 = depth_cqi x 256 rounded to the nearest integer (halves
 * away from zero), depth_cqi in [0, 15]; each coherence 0 or in [1, INT32_MAX], rounded the same way.  RS_ERR_ARG, with
 * the reason in rs_last_error, otherwise (non-integer or negative counts, non-finite values). */
int rs_channel_spec(const double* level_counts, double depth_cqi, double coherence_rbgs, double coherence_epochs,
                    rs_channel* out);

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
