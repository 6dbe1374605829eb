/* oracle/rs_oracle.h -- CPU restatement of RadioSaber's per-TTI downlink RBG
 * allocation (TEST INFRASTRUCTURE ONLY).
 *
 * This is the checker, not the product: only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load it.  Nothing
 * under radiosaber_b200/ links, imports or calls it.
 *
 * Every function cites the reference file:line it restates (paths relative to
 * /root/reference/src).  Parity status: PINNED -- validated against the
 * reference's own classes compiled unmodified from /root/reference
 * (oracle/ref_harness.cpp -> oracle/_ref/ref_harness) and against the golden
 * vectors that harness produced (tests/golden/).
 */
#ifndef RS_ORACLE_H_
#define RS_ORACLE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rso_config {
  int32_t algo;             /* 1 PF, 7 NVS, 8 Sequential, 9 RadioSaber, 10 UpperBound, 11 NVS non-greedy; 101 SubOpt and 103 VogelApproximate = 100 + the
                               constructor argument of DownlinkTransportScheduler (no scenario id, ENodeB.cpp:363-379) (single-cell-with-interference.h:94-118) */
  int32_t n_slices;         /* S */
  int32_t n_ues;            /* U; user j == UE id j (Application.cpp:72-123) */
  int32_t n_rbs;            /* 512 for 100 MHz (bandwidth-manager.cpp:98-102) */
  int32_t rbg_size;         /* get_rbg_size(): 8 (eesm-effective-sinr.h:82-103) */
  int32_t cqi_per_rb;       /* 0: cqi[U][G] (one value per RBG); 1: cqi[U][n_rbs] */
  int32_t data_to_transmit; /* 100000000 for infinite buffer (transport.cpp:123-125) */
  int32_t dead_work;        /* 1: also do the reference's wideband-CQI EESM per user
                               (packet-scheduler.cpp:321-334); results never change */
  int32_t n_bearers;        /* bearers per UE: 0 / 1 = one; 2 = MAX_BEARERS (packet-scheduler.h:31): slot i of a UE = its bearer
                               of priority i; avg_rate / tx_bytes / cum_* / queue_bytes / hol_delay are then [B][U][2] */
  int32_t reserved;
  const double* weight;     /* [S] slice_weights_ */
  const int32_t* params;    /* [S][4] alpha,beta,epsilon,psi */
  const int32_t* ue_to_slice; /* [U] user_to_slice_ */
  const int32_t* tbs_row_m1;  /* [27] what TransportBlockSizeTable[-1][itbs] reads in the
                                 reference's -O0 build (AMCModule.cpp:312-316, SURVEY H2);
                                 NULL = values captured from oracle/_ref */
} rso_config;

/* All per-cell arrays are laid out [B][...] contiguous. NULL outputs are skipped. */
typedef struct rso_io {
  /* state, updated in place */
  double* avg_rate;      /* [B][U] m_averageTransmissionRate (radio-bearer.cpp:54) */
  int32_t* tx_bytes;     /* [B][U] m_transmittedBytes */
  uint64_t* cum_bytes;   /* [B][U] m_cumulativeBytes */
  uint64_t* cum_rbs;     /* [B][U] m_cumulativeRBs */
  double* slice_offset;  /* [B][S] slice_rbs_offset_ (ids 8/9) */
  double* nvs_ewma;      /* [B][S] slice_ewma_time_ (id 7) */
  /* inputs */
  const uint8_t* cqi;    /* [B][U][G] or [B][U][n_rbs] */
  const uint8_t* active; /* [B][U] 1 = bearer has packets; NULL = all active */
  const int32_t* rand2;  /* [B][2] the two rand() values of transport.cpp:490,511 */
  double dt;             /* Now - lastUpdate (radio-bearer.cpp:150); 0 = skip the EWMA */
  /* outputs */
  int16_t* rbg_to_ue;    /* [B][G] winner user index, -1 = RBG unallocated */
  int32_t* tbs_bits;     /* [B][U] UpdateAllocatedBits value, 0 if unscheduled */
  uint8_t* mcs;          /* [B][U] MCS on the PDCCH records, 0xff if unscheduled */
  uint8_t* final_cqi;    /* [B][U] "final_cqi" of transport.cpp:649, 0 if unscheduled */
  int32_t* slice_target; /* [B][S] slice_target_rbs (ids 8/9) */
  int32_t* slice_quota;  /* [B][S] slice_quota_rbgs (ids 8/9) */
  int32_t* nvs_slice;    /* [B] slice served (ids 7/11) */
  int32_t* alloc_n;      /* [B] id 10: number of (user, RBG) grants (an RBG can go to several slices) */
  int16_t* alloc_ue;     /* [B][L] id 10: user of grant e, slice-major, each slice's grants in its sorted order; -1 past n
                            (the first L of up to S*G grants; alloc_n counts them all) */
  int16_t* alloc_rbg;    /* [B][L] id 10: RBG of grant e */
  int32_t rand_stride;   /* int32 values per cell in rand2: 0 or 2 for ids 8/9; id 11: >= 300 x the users of a
                            slice, the rand() draws of nvs.cpp:437-446 in call order */
  /* queue state of the (single) bearer of each UE this TTI (SURVEY 8 f3); both optional */
  const int32_t* queue_bytes; /* [B][U] what SelectFlowsToSchedule takes as dataToTransmit (transport.cpp:119-128):
                                 0 = no packets (the bearer is not listed), 100000000 = infinite buffer, else the queue
                                 size; NULL = cfg.data_to_transmit for every UE */
  const double* hol_delay;    /* [B][U] RadioBearer::GetHeadOfLinePacketDelay; NULL = 0 */
  int32_t alloc_len;          /* L, entries per cell of alloc_ue / alloc_rbg; 0 = 2G */
} rso_io;

/* One TTI for n_cells cells, n_threads host threads (cells are independent). */
int rso_step(const rso_config* cfg, int32_t n_cells, rso_io* io, int32_t n_threads);

/* AMC / EESM helpers exposed for table checks. */
double rso_eesm_effective_sinr(const double* sinr_db, int32_t n);
int32_t rso_cqi_from_sinr(double sinr_db);
double rso_sinr_from_cqi(int32_t cqi);
int32_t rso_mcs_from_cqi(int32_t cqi);
int32_t rso_tbs_from_mcs(int32_t mcs, int32_t n_rbs, const int32_t* row_m1);
double rso_efficiency_from_cqi(int32_t cqi);
void rso_default_row_m1(int32_t* out27);

/* std::sort (the real libstdc++ one) on (index,key) pairs with the comparator
 * of transport.cpp:361 (key descending).  perm_out[i] = original index of the
 * element that ends at position i. */
void rso_std_sort_desc(const double* keys, int32_t n, int32_t* perm_out);
/* Independent emulation of libstdc++ introsort with an explicit depth limit
 * (depth_limit < 0 => 2*floor(log2 n), the library's own).  Used to cross-check
 * the device sort's heap-sort fallback. */
void rso_introsort_emul_desc(const double* keys, int32_t n, int32_t depth_limit, int32_t* perm_out);

#ifdef __cplusplus
}
#endif
#endif /* RS_ORACLE_H_ */
