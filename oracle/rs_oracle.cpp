/* oracle/rs_oracle.cpp -- CPU restatement of the reference's per-TTI downlink
 * RBG allocation.  TEST INFRASTRUCTURE ONLY (see rs_oracle.h).
 *
 * Parity status: PINNED against the unmodified reference classes
 * (oracle/ref_harness.cpp) and the golden vectors under tests/golden/.
 *
 * Deliberately written the way the reference computes: doubles, libm
 * pow/exp/log/log10 for EESM, the real libstdc++ std::sort for RadioSaber's
 * (rbg,slice) ordering.  Build with -ffp-contract=off so no a*b+c is fused.
 * Citations are file:line under /root/reference/src; "transport.cpp" is
 * protocolStack/mac/packet-scheduler/downlink-transport-scheduler.cpp,
 * "nvs.cpp" downlink-nvs-scheduler.cpp, "dlps.cpp" downlink-packet-scheduler.cpp,
 * "dl-pf.cpp" dl-pf-packet-scheduler.cpp, "ps.cpp" packet-scheduler.cpp.
 */
#include "rs_oracle.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <limits>
#include <thread>
#include <utility>
#include <unordered_map>
#include <vector>

namespace {

/* ---- AMC tables (protocolStack/mac/AMCModule.cpp) ---------------------- */
/* MapCQIToMCS, AMCModule.cpp:36-40 */
const int kCqiToMcs[15] = {0, 2, 4, 6, 8, 10, 12, 14, 16, 18, 20, 22, 24, 26, 28};
/* SINRForCQIIndex, AMCModule.cpp:96-100 */
const double kSinrForCqi[15] = {-4.63, -2.6, -0.12, 2.26, 4.73, 7.53, 8.67, 11.32,
                                14.24, 15.21, 18.63, 21.32, 23.47, 28.49, 34.6};
/* McsToItbs, AMCModule.cpp:114-117 */
const int kMcsToItbs[29] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 10, 11, 12, 13, 14, 15, 15, 16,
                            17, 18, 19, 20, 21, 22, 23, 24, 25, 26};
/* TransportBlockSizeTable, AMCModule.cpp:120-231 */
const int kTbs[110 * 27] = {
#include "../include/rs_tbs_36213.inc"
};

inline int Tbs(int row, int itbs, const int32_t* row_m1) {
  /* row == -1 is the reference's out-of-bounds read (SURVEY H2) */
  if (row < 0) return row_m1[itbs];
  return kTbs[row * 27 + itbs];
}

/* AMCModule::GetCQIFromSinr, AMCModule.cpp:252-261 */
int CqiFromSinr(double sinr) {
  int cqi = 1;
  while (cqi <= 14 && kSinrForCqi[cqi] <= sinr) cqi++;
  return cqi;
}
/* AMCModule::GetSinrFromCQI, AMCModule.cpp:263-268 */
double SinrFromCqi(int cqi) { return kSinrForCqi[cqi - 1]; }
/* AMCModule::GetMCSFromCQI, AMCModule.cpp:270-274 */
int McsFromCqi(int cqi) { return kCqiToMcs[cqi - 1]; }
/* AMCModule::GetTBSizeFromMCS(mcs), AMCModule.cpp:298-303 */
int Tbs1(int mcs) { return kTbs[kMcsToItbs[mcs]]; }
/* AMCModule::GetTBSizeFromMCS(mcs, nbRBs), AMCModule.cpp:305-317 */
int TbsN(int mcs, int nb_rbs, const int32_t* row_m1) {
  int itbs = kMcsToItbs[mcs];
  if (nb_rbs <= 110) return Tbs(nb_rbs - 1, itbs, row_m1);
  int sub = nb_rbs / 5;
  int rest = nb_rbs % 5;
  return 5 * Tbs(sub - 1, itbs, row_m1) + Tbs(rest - 1, itbs, row_m1);
}
/* AMCModule::GetEfficiencyFromCQI, AMCModule.cpp:319-327 */
double EffFromCqi(int cqi) {
  int bits = Tbs1(McsFromCqi(cqi));
  double eff = (bits / 0.001) / 180000.;
  return eff;
}
/* GetEesmEffectiveSinr, utility/eesm-effective-sinr.h:33-46 */
double Eesm(const std::vector<double>& sinr) {
  double sum_i = 0;
  double beta = 1;
  for (size_t i = 0; i < sinr.size(); ++i) {
    double s = pow(10, sinr[i] / 10);
    sum_i += exp(-s / beta);
  }
  double eff = -beta * log(sum_i / sinr.size());
  eff = 10 * log10(eff);
  return eff;
}

/* What TransportBlockSizeTable[-1][itbs] reads in the reference's own -O0 build:
 * the table sits 128 bytes after McsToItbs[29] (116 bytes + 12 of zero padding),
 * so row -1 (108 bytes back) aliases McsToItbs[5..28] followed by three zeros.
 * Confirmed with oracle/_ref/ref_harness --probe-row-m1. */
void DefaultRowM1(int32_t* out) {
  for (int i = 0; i < 27; ++i) out[i] = (i + 5 < 29) ? kMcsToItbs[i + 5] : 0;
}

struct User {          /* PacketScheduler::UserToSchedule, ps.h:88-123 */
  int id;
  int slice;
  std::vector<int> cqi;      /* per RB */
  std::vector<double> eff;   /* per RB */
  std::vector<int> rbs;      /* m_listOfAllocatedRBs */
  int wide_cqi = 0;
  int required_rbs = 0;
  int bits = 0;
  int data = 0;
  double hol = 0;   /* RadioBearer::GetHeadOfLinePacketDelay of the (single) bearer */
  /* two bearers per UE (m_bearers[MAX_BEARERS], m_dataToTransmit[MAX_BEARERS], ps.h:101-102): slot = bearer priority */
  int data2[2] = {0, 0};
  double hol2[2] = {0, 0};
};

struct CellView {
  const rso_config* cfg;
  double* avg;
  int32_t* tx;
  uint64_t* cum_bytes;
  uint64_t* cum_rbs;
  double* offset;
  double* ewma;
  const uint8_t* cqi;
  const uint8_t* active;
  const int32_t* rand2;
  double dt;
  int16_t* rbg_to_ue;
  int32_t* tbs_bits;
  uint8_t* mcs;
  uint8_t* final_cqi;
  int32_t* target;
  int32_t* quota;
  int32_t* nvs_slice;
  int32_t* alloc_n;
  int16_t* alloc_ue;
  int16_t* alloc_rbg;
  int alloc_len = 0;       /* entries of alloc_ue / alloc_rbg */
  const int32_t* queue;   /* [U] bytes queued per bearer this TTI, NULL = cfg->data_to_transmit for everyone */
  const double* hol;      /* [U] head-of-line delay, NULL = 0 */
  int nb = 1;             /* bearers per UE; per-bearer arrays are [U][nb] */
};

/* RadioBearer::UpdateAverageTransmissionRate, flows/radio-bearer.cpp:138-164,
 * looped over every bearer (transport.cpp:715-727, nvs.cpp:392-403, dlps.cpp:503-514). */
void UpdateAverages(const CellView& c) {
  if (c.dt == 0) return; /* Now == lastUpdate */
  for (int u = 0; u < c.cfg->n_ues * c.nb; ++u) {   /* every bearer */
    double rate = (c.tx[u] * 8) / c.dt;
    double beta = 0.02;
    c.avg[u] = ((1 - beta) * c.avg[u]) + (beta * rate);
    if (c.avg[u] < 1) c.avg[u] = 1;
    c.tx[u] = 0;
  }
}

/* SelectFlowsToSchedule (transport.cpp:105-150, nvs.cpp:144-194, dlps.cpp:48-94)
 * + InsertFlowToUser (ps.cpp:304-335). only_slice < 0 selects every slice. */
std::vector<User> SelectUsers(const CellView& c, int only_slice) {
  const rso_config* cfg = c.cfg;
  const int R = cfg->n_rbs, G = R / cfg->rbg_size;
  std::vector<User> users;
  for (int u = 0; u < cfg->n_ues; ++u) {
    if (c.active && !c.active[u]) continue;
    if (only_slice >= 0 && cfg->ue_to_slice[u] != only_slice) continue;
    User usr;
    usr.id = u;
    usr.slice = cfg->ue_to_slice[u];
    /* transport.cpp:119-128: only bearers with packets are listed; dataToTransmit = 100000000 for an
     * infinite buffer, else the queue size */
    if (c.nb == 2) {
      /* both bearers of the UE join one UserToSchedule (InsertFlowToUser, ps.cpp:304-318); the bearer that comes first
       * in the container (slot 0, then slot 1) creates the record and sets m_requiredRBs (:333) */
      for (int i = 0; i < 2; ++i) {
        usr.data2[i] = std::max(c.queue[2 * u + i], 0);
        usr.hol2[i] = c.hol ? c.hol[2 * u + i] : 0.0;
      }
      if (usr.data2[0] <= 0 && usr.data2[1] <= 0) continue;
      usr.data = usr.data2[0] > 0 ? usr.data2[0] : usr.data2[1];
    } else {
    usr.data = c.queue ? c.queue[u] : cfg->data_to_transmit;
    if (c.queue && usr.data <= 0) continue;
    usr.hol = c.hol ? c.hol[u] : 0.0;
    }
    usr.cqi.resize(R);
    usr.eff.resize(R);
    for (int r = 0; r < R; ++r) {
      int q = cfg->cqi_per_rb ? c.cqi[(size_t)u * R + r]
                              : c.cqi[(size_t)u * G + std::min(r / cfg->rbg_size, G - 1)];
      usr.cqi[r] = q;
      usr.eff[r] = EffFromCqi(q);
    }
    if (cfg->dead_work || cfg->algo == 7 || cfg->algo == 11) {
      std::vector<double> sinrs;
      for (int r = 0; r < R; ++r) sinrs.push_back(SinrFromCqi(usr.cqi[r]));
      usr.wide_cqi = CqiFromSinr(Eesm(sinrs));
      usr.required_rbs += (usr.data * 8 / Tbs1(McsFromCqi(usr.wide_cqi)));
    } else {
      usr.required_rbs = std::numeric_limits<int>::max();
    }
    users.push_back(std::move(usr));
  }
  return users;
}

/* ComputeSchedulingMetric, transport.cpp:677-713; nvs = the copy in nvs.cpp:360-390, which multiplies
 * the head-of-line delay in whenever alpha != 0 (the transport version only when beta != 0). */
/* 1 + the rates of the user's LISTED bearers in slot order (transport.cpp:680-687, ps.cpp:423-433) */
double RateSum(const CellView& c, const User& usr) {
  double sum_rate = 1;
  if (c.nb == 2) {
    for (int i = 0; i < 2; ++i)
      if (usr.data2[i] > 0) sum_rate += c.avg[2 * usr.id + i];
  } else {
    sum_rate += c.avg[usr.id];
  }
  return sum_rate;
}

/* slice_priority_ (transport.cpp:115, 143-146): the highest priority among the listed bearers of each slice */
std::vector<int> SlicePriority(const CellView& c, const std::vector<User>& users) {
  std::vector<int> prio(c.cfg->n_slices, 0);
  if (c.nb == 2)
    for (const User& u : users)
      if (u.data2[1] > 0) prio[u.slice] = 1;
  return prio;
}

double TransportMetric(const CellView& c, const User& usr, const std::vector<int>& slice_prio, double eff, bool nvs = false) {
  const rso_config* cfg = c.cfg;
  double metric = 0;
  double average_rate = RateSum(c, usr);
  eff = eff * 180000 / 1000;
  average_rate /= 1000.0;
  const int32_t* p = cfg->params + 4 * usr.slice;
  int alpha = p[0], beta = p[1], epsilon = p[2], psi = p[3];
  if (alpha == 0) {
    metric = pow(eff, epsilon) / pow(average_rate, psi);
  } else if (c.nb == 2) {
    /* the prioritized flow has no packet, set metric to 0 (:696-698); else its head-of-line delay (:700-706) */
    const int pr = slice_prio[usr.slice];
    if (usr.data2[pr] == 0) {
      metric = 0;
    } else if (beta || nvs) {
      metric = usr.hol2[pr] * pow(eff, epsilon) / pow(average_rate, psi);
    } else {
      metric = pow(eff, epsilon) / pow(average_rate, psi);
    }
  } else {
    /* one entry per UE: a caller that folds two bearers marks "the bearer of the slice's priority is empty" (:696-698)
     * with a head-of-line delay of 0 where the delay multiplies the metric anyway, and with a negative one where it does not */
    if (usr.data == 0 || (!(beta || nvs) && usr.hol < 0)) {
      metric = 0;
    } else {
      if (beta || nvs) {
        double HoL = usr.hol;
        metric = HoL * pow(eff, epsilon) / pow(average_rate, psi);
      } else {
        metric = pow(eff, epsilon) / pow(average_rate, psi);
      }
    }
  }
  return metric;
}

using coord_t = std::pair<int, int>;
using coord_cqi_t = std::pair<coord_t, double>;

/* GreedyByRow, transport.cpp:249-272 */
std::vector<int> GreedyByRow(const std::vector<std::vector<double>>& se, const std::vector<int>& quota,
                             int G, int S) {
  std::vector<int> used(S, 0), out(G, -1);
  for (int i = 0; i < G; ++i) {
    double best = -1;
    int pick = -1;
    for (int j = 0; j < S; ++j) {
      if (se[i][j] > best && used[j] < quota[j]) {
        best = se[i][j];
        pick = j;
      }
    }
    out[i] = pick; /* the reference asserts pick != -1 */
    if (pick >= 0) used[pick] += 1;
  }
  return out;
}

/* SubOpt, transport.cpp:274-349 (DLScheduler_SUBOPT, constructor argument 1): every RBG first goes to the
 * slice with the best efficiency, then RBGs move one at a time from slices above their quota to slices below
 * it, always the move that loses the least efficiency.  Ties are broken by the iteration order of the
 * reference's two std::unordered_map<int,int> (the same containers, filled in the same order, here). */
std::vector<int> SubOpt(const std::vector<std::vector<double>>& se, std::vector<int> quota, int G, int S) {
  std::vector<int> held(S, 0), out(G, -1);
  for (int& q : quota)
    if (q < 0) q = 0;
  for (int i = 0; i < G; ++i) {
    double best = -1;
    int pick = -1;
    for (int j = 0; j < S; ++j)
      if (se[i][j] > best) {
        best = se[i][j];
        pick = j;
      }
    out[i] = pick;
    held[pick] += 1;
  }
  std::unordered_map<int, int> over, under;
  for (int i = 0; i < S; ++i) {
    if (held[i] > quota[i]) over[i] = held[i] - quota[i];
    else if (held[i] < quota[i]) under[i] = quota[i] - held[i];
  }
  while (over.size() > 0 && under.size() > 0) {
    int from = -1, to = -1, rbg = -1;
    double least = std::numeric_limits<double>::max();
    for (int i = 0; i < G; ++i) {
      if (over.find(out[i]) == over.end()) continue;
      for (auto it = under.begin(); it != under.end(); ++it) {
        const double loss = se[i][out[i]] - se[i][it->first];
        if (loss < least) {
          least = loss;
          from = out[i];
          to = it->first;
          rbg = i;
        }
      }
    }
    if (from < 0) break; /* assert in the reference */
    held[from] -= 1;
    held[to] += 1;
    out[rbg] = to;
    over.at(from) -= 1;
    under.at(to) -= 1;
    if (over.at(from) <= 0 || held[from] <= 0) over.erase(from);
    if (under.at(to) <= 0) under.erase(to);
  }
  return out;
}

/* VogelApproximate, transport.cpp:378-451 (DLScheduler_VOGEL, constructor argument 3): G rounds; each round
 * looks at every free RBG (best and "second" efficiency among the slices with quota left) and at every such
 * slice (best and "second" among the free RBGs) and grants the best cell of the row / column with the
 * largest gap.  Reproduced with its quirks: the running largest gap is an int (the gap is truncated when it
 * is stored), and "second" is the best of the candidates seen AFTER the current best, not the runner-up. */
std::vector<int> VogelApproximate(const std::vector<std::vector<double>>& se, const std::vector<int>& quota, int G, int S) {
  std::vector<int> held(S, 0), out(G, -1);
  for (int round = 0; round < G; ++round) {
    int max_diff = -1;
    int grant_rbg = -1, grant_slice = -1;
    for (int j = 0; j < G; ++j) {
      if (out[j] != -1) continue;
      double e1 = -1, e2 = -1;
      int s1 = -1;
      for (int k = 0; k < S; ++k) {
        if (held[k] >= quota[k]) continue;
        if (e1 == -1 || se[j][k] > e1) { s1 = k; e1 = se[j][k]; continue; }
        if (e2 == -1 || se[j][k] > e2) { e2 = se[j][k]; continue; }
      }
      if (e1 - e2 > max_diff) {
        max_diff = e1 - e2;
        grant_rbg = j;
        grant_slice = s1;
      }
    }
    for (int k = 0; k < S; ++k) {
      if (held[k] >= quota[k]) continue;
      double e1 = -1, e2 = -1;
      int r1 = -1;
      for (int j = 0; j < G; ++j) {
        if (out[j] != -1) continue;
        if (e1 == -1 || se[j][k] > e1) { r1 = j; e1 = se[j][k]; continue; }
        if (e2 == -1 || se[j][k] > e2) { e2 = se[j][k]; continue; }
      }
      if (e1 - e2 > max_diff) {
        max_diff = e1 - e2;
        grant_rbg = r1;
        grant_slice = k;
      }
    }
    if (grant_rbg < 0 || grant_slice < 0) break; /* the reference would index with an uninitialised pair */
    out[grant_rbg] = grant_slice;
    held[grant_slice] += 1;
  }
  return out;
}

/* Diagnostic (rso_diag_*): histogram of the position of the last entry MaximizeCell's scan accepts, in 64ths of
 * the list length.  Off by default; results never depend on it. */
static std::atomic<int> g_diag_on{0};
static std::atomic<uint64_t> g_diag_stop[66];

/* MaximizeCell, transport.cpp:351-376 */
std::vector<int> MaximizeCell(const std::vector<std::vector<double>>& se, const std::vector<int>& quota,
                              int G, int S) {
  std::vector<coord_cqi_t> sorted;
  std::vector<int> used(S, 0), out(G, -1);
  for (int i = 0; i < G; ++i)
    for (int j = 0; j < S; ++j) sorted.emplace_back(coord_t(i, j), se[i][j]);
  std::sort(sorted.begin(), sorted.end(),
            [](coord_cqi_t a, coord_cqi_t b) { return a.second > b.second; });
  size_t last_take = 0;
  for (auto it = sorted.begin(); it != sorted.end(); ++it) {
    int rbg = it->first.first, sl = it->first.second;
    if (used[sl] < quota[sl] && out[rbg] == -1) {
      out[rbg] = sl;
      used[sl] += 1;
      last_take = (size_t)(it - sorted.begin()) + 1;
    }
  }
  if (g_diag_on.load(std::memory_order_relaxed)) {   /* diagnostic: how far into the sorted list the scan has to look */
    const size_t n = sorted.size();
    g_diag_stop[n ? (last_take * 64 + n - 1) / n : 0].fetch_add(1, std::memory_order_relaxed);
  }
  return out;
}

/* Link adaptation tail shared by all four schedulers:
 * transport.cpp:632-660, nvs.cpp:315-343, dlps.cpp:279-303. */
void FinalizeUser(const CellView& c, User& usr, const int32_t* row_m1) {
  if (usr.rbs.empty()) return;
  std::vector<double> sinrs;
  for (size_t i = 0; i < usr.rbs.size(); ++i) sinrs.push_back(SinrFromCqi(usr.cqi[usr.rbs[i]]));
  double eff_sinr = Eesm(sinrs);
  int fc = CqiFromSinr(eff_sinr);
  int mcs = McsFromCqi(fc);
  int tbs = TbsN(mcs, (int)usr.rbs.size(), row_m1);
  usr.bits += tbs;
  if (c.tbs_bits) c.tbs_bits[usr.id] = usr.bits;
  if (c.mcs) c.mcs[usr.id] = (uint8_t)mcs;
  if (c.final_cqi) c.final_cqi[usr.id] = (uint8_t)fc;
}

/* DoStopSchedule accounting, transport.cpp:170-199 / nvs.cpp:220-251 (user level) */
void AccountUser(const CellView& c, const User& usr) {
  int available = usr.bits / 8;
  if (available <= 0) return;
  if (c.nb == 2) {   /* priority 1 first, what is left to priority 0; every bearer that sends is booked the user's RBs */
    for (int i = 1; i >= 0 && available > 0; --i) {
      if (usr.data2[i] <= 0) continue;
      const int sent = std::min(available, usr.data2[i]);
      available -= sent;
      c.tx[2 * usr.id + i] += sent;
      c.cum_bytes[2 * usr.id + i] += sent;
      c.cum_rbs[2 * usr.id + i] += usr.rbs.size();
    }
    return;
  }
  if (usr.data > 0) {
    int sent = std::min(available, usr.data);
    c.tx[usr.id] += sent;        /* RadioBearer::UpdateTransmittedBytes, radio-bearer.cpp:118-123 */
    c.cum_bytes[usr.id] += sent;
    c.cum_rbs[usr.id] += usr.rbs.size(); /* UpdateCumulateRBs, radio-bearer.cpp:100-104 */
  }
}

/* DL_PF_PacketScheduler::DoStopSchedule accounting, dl-pf.cpp:64-96 (flow level) */
void AccountFlowPf(const CellView& c, const User& usr) {
  int available = usr.bits / 8;
  if (available > 0) {
    c.tx[usr.id] += available;
    c.cum_bytes[usr.id] += available;
    c.cum_rbs[usr.id] += usr.rbs.size();
  }
}

void ClearOutputs(const CellView& c) {
  const rso_config* cfg = c.cfg;
  const int G = cfg->n_rbs / cfg->rbg_size;
  if (c.rbg_to_ue) std::fill(c.rbg_to_ue, c.rbg_to_ue + G, (int16_t)-1);
  if (c.tbs_bits) std::fill(c.tbs_bits, c.tbs_bits + cfg->n_ues, 0);
  if (c.mcs) std::fill(c.mcs, c.mcs + cfg->n_ues, (uint8_t)0xff);
  if (c.final_cqi) std::fill(c.final_cqi, c.final_cqi + cfg->n_ues, (uint8_t)0);
  if (c.target) std::fill(c.target, c.target + cfg->n_slices, 0);
  if (c.quota) std::fill(c.quota, c.quota + cfg->n_slices, 0);
  if (c.nvs_slice) *c.nvs_slice = -1;
  if (c.alloc_n) *c.alloc_n = 0;
  if (c.alloc_ue) { std::fill(c.alloc_ue, c.alloc_ue + c.alloc_len, (int16_t)-1); std::fill(c.alloc_rbg, c.alloc_rbg + c.alloc_len, (int16_t)-1); }
}

/* DownlinkTransportScheduler::DoSchedule, transport.cpp:152-168, ids 8 and 9. */
void StepTransport(const CellView& c, const int32_t* row_m1) {
  const rso_config* cfg = c.cfg;
  const int S = cfg->n_slices, rbg_size = cfg->rbg_size;
  UpdateAverages(c);
  std::vector<User> users = SelectUsers(c, -1);
  if (users.empty()) return;
  const std::vector<int> slice_prio = SlicePriority(c, users);

  /* RBsAllocation, transport.cpp:453-675 */
  int nb_rbs = cfg->n_rbs;
  nb_rbs = nb_rbs - (nb_rbs % rbg_size);
  std::vector<bool> with_data(S, false);
  std::vector<int> target(S, 0);
  int nonempty = 0;
  int extra_rbs = nb_rbs;
  for (const User& usr : users) {           /* :468-477 */
    int sl = usr.slice;
    if (with_data[sl]) continue;
    nonempty += 1;
    with_data[sl] = true;
    target[sl] = (int)(nb_rbs * cfg->weight[sl] + c.offset[sl]);
    extra_rbs -= target[sl];
  }
  bool first = true;                        /* :489-500 */
  int begin = c.rand2[0];
  for (int i = 0; i < S; ++i) {
    int k = (i + begin) % S;
    if (with_data[k]) {
      target[k] += extra_rbs / nonempty;
      if (first) {
        target[k] += extra_rbs % nonempty;
        first = false;
      }
    }
  }
  int G = nb_rbs / rbg_size;                /* :501-521 */
  std::vector<int> quota(S, 0), final_rbgs(S, 0);
  int extra_rbgs = G;
  for (int i = 0; i < S; ++i) {
    quota[i] = (int)(target[i] / rbg_size);
    extra_rbgs -= quota[i];
  }
  first = true;
  begin = c.rand2[1];
  for (int i = 0; i < S; ++i) {
    int k = (begin + i) % S;
    if (with_data[k]) {
      quota[k] += extra_rbgs / nonempty;
      if (first) {
        quota[k] += extra_rbgs % nonempty;
        first = false;
      }
    }
  }
  if (c.target) std::copy(target.begin(), target.end(), c.target);
  if (c.quota) std::copy(quota.begin(), quota.end(), c.quota);

  const size_t n = users.size();            /* :530-539 */
  std::vector<std::vector<double>> metrics(G, std::vector<double>(n));
  for (int i = 0; i < G; ++i)
    for (size_t j = 0; j < n; ++j)
      metrics[i][j] = TransportMetric(c, users[j], slice_prio, users[j].eff[i * rbg_size]);

  std::vector<std::vector<int>> user_index(G, std::vector<int>(S, -1));   /* :543-567 */
  std::vector<std::vector<double>> se(G, std::vector<double>(S, 0));
  for (int i = 0; i < G; ++i) {
    std::vector<double> max_rank(S, -1);
    for (size_t j = 0; j < n; ++j) {
      int sl = users[j].slice;
      if (metrics[i][j] > max_rank[sl]) {
        max_rank[sl] = metrics[i][j];
        user_index[i][sl] = (int)j;
        se[i][sl] = users[j].eff[i * rbg_size];
      }
    }
  }

  if (cfg->algo == 10) {
    /* UpperBound, transport.cpp:223-246: every slice with a positive quota takes its own best quota RBGs
     * (the real std::sort of (rbg, eff) pairs), so an RBG can be granted to several slices; then
     * :603-616: the winners' RB lists are appended in that sorted order. */
    int n_alloc = 0;
    for (int j = 0; j < S; ++j) {
      if (quota[j] <= 0) continue;
      std::vector<std::pair<int, double>> sorted_cqi;
      for (int i = 0; i < G; ++i) sorted_cqi.emplace_back(i, se[i][j]);
      std::sort(sorted_cqi.begin(), sorted_cqi.end(),
                [](std::pair<int, double> a, std::pair<int, double> b) { return a.second > b.second; });
      for (int k = 0; k < quota[j] && k < G; ++k) {   /* k >= G would read past the vector in the reference */
        const int rbg = sorted_cqi[k].first;
        const int uindex = user_index[rbg][j];
        if (uindex < 0) continue;             /* assert in the reference */
        final_rbgs[j] += 1;
        for (int r = rbg * rbg_size; r < (rbg + 1) * rbg_size; ++r) users[uindex].rbs.push_back(r);
        if (c.alloc_ue && n_alloc < c.alloc_len) { c.alloc_ue[n_alloc] = (int16_t)users[uindex].id; c.alloc_rbg[n_alloc] = (int16_t)rbg; }
        n_alloc++;
      }
    }
    if (c.alloc_n) *c.alloc_n = n_alloc;
    if (c.rbg_to_ue)   /* what a single-valued map can say: the highest user id holding the RBG */
      for (const User& usr : users)
        for (int r : usr.rbs)
          if (r % rbg_size == 0) c.rbg_to_ue[r / rbg_size] = (int16_t)usr.id;
    for (int i = 0; i < S; ++i) c.offset[i] = target[i] - final_rbgs[i] * rbg_size;
    for (User& usr : users) FinalizeUser(c, usr, row_m1);
    for (const User& usr : users) AccountUser(c, usr);
    return;
  }

  std::vector<int> rbg_to_slice =           /* :569-586 */
      (cfg->algo == 8) ? GreedyByRow(se, quota, G, S)
      : (cfg->algo == 101) ? SubOpt(se, quota, G, S)
      : (cfg->algo == 103) ? VogelApproximate(se, quota, G, S)
                           : MaximizeCell(se, quota, G, S);

  for (int i = 0; i < G; ++i) {             /* :589-601 */
    if (rbg_to_slice[i] < 0) continue;      /* assert in the reference */
    int uindex = user_index[i][rbg_to_slice[i]];
    if (uindex < 0) continue;               /* assert in the reference */
    final_rbgs[rbg_to_slice[i]] += 1;
    for (int r = i * rbg_size; r < (i + 1) * rbg_size; ++r) users[uindex].rbs.push_back(r);
    if (c.rbg_to_ue) c.rbg_to_ue[i] = (int16_t)users[uindex].id;
  }
  for (int i = 0; i < S; ++i)               /* :618-620 */
    c.offset[i] = target[i] - final_rbgs[i] * rbg_size;

  for (User& usr : users) FinalizeUser(c, usr, row_m1);
  for (const User& usr : users) AccountUser(c, usr);
}

/* DownlinkNVSScheduler::AssignRBsGivenMCS, nvs.cpp:489-528: per RBG the first user with the strictly
 * largest metric, where a user counts only on RBGs whose CQI reaches its assigned MCS (the reference
 * calls the assigned CQI level "mcs"); returns the sum of the winning metrics. */
double AssignRbsGivenMcs(const CellView& c, const std::vector<User>& users, const std::vector<int>& assigned_mcs,
                         std::vector<int>& rbgs_assignment) {
  const int rbg_size = c.cfg->rbg_size;
  const int nb_rbgs = (int)rbgs_assignment.size();
  double pf_metric = 0;
  for (int i = 0; i < nb_rbgs; i++) {
    double highest_metric = -1;
    for (size_t index = 0; index < users.size(); ++index) {
      int cqi = users[index].cqi[i * rbg_size];
      double metric = 0;
      if (assigned_mcs[index] <= cqi) {
        double sEff = EffFromCqi(assigned_mcs[index]);
        /* UserToSchedule::GetAverageTransmissionRate, ps.cpp:423-433: 1 + sum of the bearers' rates */
        double sum_rate = RateSum(c, users[index]);
        metric = sEff * 180000 / sum_rate;
      }
      if (highest_metric < metric) {
        highest_metric = metric;
        rbgs_assignment[i] = (int)index;
      }
    }
    pf_metric += highest_metric;
  }
  return pf_metric;
}

/* DownlinkNVSScheduler::RBsAllocationNonGreedyPF, nvs.cpp:405-452 (id 11): 300 random per-user CQI
 * back-offs (rand() % 4 below the user's best RBG), keep the first sample with the largest metric sum.
 * draws = the rand() values in call order, 300 x users.size() of them. */
void AllocateNonGreedy(const CellView& c, std::vector<User>& users, const int32_t* draws) {
  const int rbg_size = c.cfg->rbg_size;
  int nb_rbs = c.cfg->n_rbs;
  nb_rbs = nb_rbs - (nb_rbs % rbg_size);
  const int nb_rbgs = nb_rbs / rbg_size;
  std::vector<int> user_highest_cqi;
  for (const User& usr : users) {
    int highest_cqi = 0;
    for (int i = 0; i < nb_rbgs; i++) {
      int cqi = usr.cqi[i * rbg_size];
      if (highest_cqi < cqi) highest_cqi = cqi;
    }
    user_highest_cqi.push_back(highest_cqi);
  }
  std::vector<int> best_rbgs_assignment;
  double highest_pf_metric = 0;
  const int cqi_search_range = 4;
  const int num_sample = 300;
  size_t pos = 0;
  for (int i = 0; i < num_sample; i++) {
    std::vector<int> assigned_mcs;
    std::vector<int> rbgs_assignment(nb_rbgs, -1);
    for (size_t k = 0; k < user_highest_cqi.size(); k++)
      assigned_mcs.push_back(std::max(user_highest_cqi[k] - draws[pos++] % cqi_search_range, 1));
    double pf_metric = AssignRbsGivenMcs(c, users, assigned_mcs, rbgs_assignment);
    if (highest_pf_metric < pf_metric) {
      highest_pf_metric = pf_metric;
      best_rbgs_assignment = rbgs_assignment;
    }
  }
  for (size_t rbg_id = 0; rbg_id < best_rbgs_assignment.size(); rbg_id++) {
    User& usr = users[best_rbgs_assignment[rbg_id]];
    for (int j = (int)rbg_id * rbg_size; j < (int)(rbg_id + 1) * rbg_size; ++j) usr.rbs.push_back(j);
    if (c.rbg_to_ue) c.rbg_to_ue[rbg_id] = (int16_t)usr.id;
  }
}

/* DownlinkNVSScheduler::DoSchedule, nvs.cpp:196-218 (id 7; id 11 = the non-greedy variant). */
void StepNvs(const CellView& c, const int32_t* row_m1) {
  const rso_config* cfg = c.cfg;
  const int S = cfg->n_slices, rbg_size = cfg->rbg_size;
  /* SelectSliceToServe, nvs.cpp:94-142 */
  int slice_id = 0;
  double max_score = 0;
  const double beta_ = 0.01; /* nvs.h:42 */
  std::vector<bool> with_queue(S, false);
  for (int u = 0; u < cfg->n_ues; ++u) {
    if (c.active && !c.active[u]) continue;
    const bool queued = c.nb == 2 ? (c.queue[2 * u] > 0 || c.queue[2 * u + 1] > 0) : ((c.queue ? c.queue[u] : cfg->data_to_transmit) > 0);
    if (queued) with_queue[cfg->ue_to_slice[u]] = true;
  }
  for (int i = 0; i < S; ++i) {
    if (!with_queue[i]) continue;
    if (c.ewma[i] == 0) {
      slice_id = i;
      break;
    } else {
      double score = cfg->weight[i] / c.ewma[i];
      if (score >= max_score) {
        max_score = score;
        slice_id = i;
      }
    }
  }
  for (int i = 0; i < S; ++i) {
    if (!with_queue[i]) continue;
    c.ewma[i] = (1 - beta_) * c.ewma[i];
    if (i == slice_id) c.ewma[i] += beta_ * 1;
  }
  if (c.nvs_slice) *c.nvs_slice = slice_id;

  UpdateAverages(c);
  std::vector<User> users = SelectUsers(c, slice_id);
  if (users.empty()) return;
  const std::vector<int> slice_prio = SlicePriority(c, users);

  if (cfg->algo == 11) {
    AllocateNonGreedy(c, users, c.rand2);
    for (User& usr : users) FinalizeUser(c, usr, row_m1);
    for (const User& usr : users) AccountUser(c, usr);
    return;
  }

  /* RBsAllocation, nvs.cpp:275-358 */
  int nb_rbs = cfg->n_rbs;
  nb_rbs = nb_rbs - (nb_rbs % rbg_size);
  int G = nb_rbs / rbg_size;
  const size_t n = users.size();
  std::vector<std::vector<double>> metrics(G, std::vector<double>(n));
  for (int i = 0; i < G; ++i)
    for (size_t j = 0; j < n; ++j)
      metrics[i][j] = TransportMetric(c, users[j], slice_prio, users[j].eff[i * rbg_size], true);
  for (int i = 0; i < G; ++i) {
    double target_metric = std::numeric_limits<double>::lowest();
    int pick = -1;
    for (size_t j = 0; j < n; ++j) {
      if (metrics[i][j] > target_metric && (long)users[j].rbs.size() < (long)users[j].required_rbs) {
        target_metric = metrics[i][j];
        pick = (int)j;
      }
    }
    if (pick >= 0) {
      for (int r = i * rbg_size; r < (i + 1) * rbg_size; ++r) users[pick].rbs.push_back(r);
      if (c.rbg_to_ue) c.rbg_to_ue[i] = (int16_t)users[pick].id;
    }
  }
  for (User& usr : users) FinalizeUser(c, usr, row_m1);
  for (const User& usr : users) AccountUser(c, usr);
}

/* DownlinkPacketScheduler::DoSchedule, dlps.cpp:96-115, with DL_PF metric (id 1). */
void StepPf(const CellView& c, const int32_t* row_m1) {
  const rso_config* cfg = c.cfg;
  const int rbg_size = cfg->rbg_size;
  UpdateAverages(c);
  std::vector<User> flows = SelectUsers(c, -1);
  if (flows.empty()) return;

  /* RBsAllocation, dlps.cpp:179-331 */
  int nb_rbs = cfg->n_rbs;
  int G = (nb_rbs + rbg_size - 1) / rbg_size;
  const size_t n = flows.size();
  std::vector<std::vector<double>> metrics(G, std::vector<double>(n));
  for (int i = 0; i < G; ++i)
    for (size_t j = 0; j < n; ++j) /* dl-pf.cpp:128-140 */
      metrics[i][j] = (flows[j].eff[i * rbg_size] * 180000.) / c.avg[flows[j].id];

  std::vector<bool> done(n, false);
  std::vector<std::vector<double>> flow_sinr(n);
  size_t n_done = 0;
  for (int s = 0; s < G; ++s) {
    if (n_done == n) break;
    double target_metric = 0;
    bool allocated = false;
    size_t pick = 0;
    for (size_t k = 0; k < n; ++k) {
      if (metrics[s][k] > target_metric && !done[k]) {
        target_metric = metrics[s][k];
        allocated = true;
        pick = k;
      }
    }
    if (allocated) {
      int l = s * rbg_size, r = (s + 1) * rbg_size;
      if (r > nb_rbs) r = nb_rbs;
      for (int i = l; i < r; ++i) {
        flows[pick].rbs.push_back(i);
        flow_sinr[pick].push_back(SinrFromCqi(flows[pick].cqi[i]));
      }
      if (c.rbg_to_ue) c.rbg_to_ue[s] = (int16_t)flows[pick].id;
      double eff_sinr = Eesm(flow_sinr[pick]);      /* dlps.cpp:259-269 */
      int mcs = McsFromCqi(CqiFromSinr(eff_sinr));
      int tbs = TbsN(mcs, (int)flows[pick].rbs.size(), row_m1);
      if (tbs >= flows[pick].data * 8) {
        done[pick] = true;
        n_done++;
      }
    }
  }
  for (User& f : flows) FinalizeUser(c, f, row_m1);
  for (const User& f : flows) AccountFlowPf(c, f);
}

void StepCell(const rso_config* cfg, rso_io* io, int b, const int32_t* row_m1) {
  const int U = cfg->n_ues, S = cfg->n_slices;
  const int G = (cfg->n_rbs + cfg->rbg_size - 1) / cfg->rbg_size;
  const size_t cqi_stride = (size_t)U * (cfg->cqi_per_rb ? cfg->n_rbs : G);
  CellView c;
  c.cfg = cfg;
  const int nb = cfg->n_bearers == 2 ? 2 : 1;
  c.nb = nb;
  c.avg = io->avg_rate + (size_t)b * U * nb;
  c.tx = io->tx_bytes + (size_t)b * U * nb;
  c.cum_bytes = io->cum_bytes + (size_t)b * U * nb;
  c.cum_rbs = io->cum_rbs + (size_t)b * U * nb;
  c.offset = io->slice_offset ? io->slice_offset + (size_t)b * S : nullptr;
  c.ewma = io->nvs_ewma ? io->nvs_ewma + (size_t)b * S : nullptr;
  c.cqi = io->cqi + (size_t)b * cqi_stride;
  c.active = io->active ? io->active + (size_t)b * U : nullptr;
  c.rand2 = io->rand2 ? io->rand2 + (size_t)b * (io->rand_stride > 0 ? io->rand_stride : 2) : nullptr;
  c.dt = io->dt;
  c.rbg_to_ue = io->rbg_to_ue ? io->rbg_to_ue + (size_t)b * G : nullptr;
  c.tbs_bits = io->tbs_bits ? io->tbs_bits + (size_t)b * U : nullptr;
  c.mcs = io->mcs ? io->mcs + (size_t)b * U : nullptr;
  c.final_cqi = io->final_cqi ? io->final_cqi + (size_t)b * U : nullptr;
  c.target = io->slice_target ? io->slice_target + (size_t)b * S : nullptr;
  c.quota = io->slice_quota ? io->slice_quota + (size_t)b * S : nullptr;
  c.nvs_slice = io->nvs_slice ? io->nvs_slice + b : nullptr;
  c.alloc_n = io->alloc_n ? io->alloc_n + b : nullptr;
  c.alloc_len = io->alloc_len > 0 ? io->alloc_len : 2 * G;
  c.alloc_ue = (io->alloc_ue && io->alloc_rbg) ? io->alloc_ue + (size_t)b * c.alloc_len : nullptr;
  c.alloc_rbg = (io->alloc_ue && io->alloc_rbg) ? io->alloc_rbg + (size_t)b * c.alloc_len : nullptr;
  c.queue = io->queue_bytes ? io->queue_bytes + (size_t)b * U * nb : nullptr;
  c.hol = io->hol_delay ? io->hol_delay + (size_t)b * U * nb : nullptr;
  ClearOutputs(c);
  switch (cfg->algo) {
    case 1: StepPf(c, row_m1); break;
    case 7: case 11: StepNvs(c, row_m1); break;
    default: StepTransport(c, row_m1); break;
  }
}

/* ---- independent introsort emulation (libstdc++ 13 bits/stl_algo.h:1848-1950,
 * bits/stl_heap.h:128-432), generic over a depth limit ----------------------- */
struct Item {
  double key;
  int idx;
};
inline bool Before(const Item& a, const Item& b) { return a.key > b.key; } /* transport.cpp:361 */

void EmulPushHeap(Item* f, long hole, long top, Item v) {
  long parent = (hole - 1) / 2;
  while (hole > top && Before(f[parent], v)) {
    f[hole] = f[parent];
    hole = parent;
    parent = (hole - 1) / 2;
  }
  f[hole] = v;
}
void EmulAdjustHeap(Item* f, long hole, long len, Item v) {
  const long top = hole;
  long child = hole;
  while (child < (len - 1) / 2) {
    child = 2 * (child + 1);
    if (Before(f[child], f[child - 1])) child--;
    f[hole] = f[child];
    hole = child;
  }
  if ((len & 1) == 0 && child == (len - 2) / 2) {
    child = 2 * (child + 1);
    f[hole] = f[child - 1];
    hole = child - 1;
  }
  EmulPushHeap(f, hole, top, v);
}
void EmulHeapSort(Item* f, long len) {
  if (len >= 2) {
    long parent = (len - 2) / 2;
    while (true) {
      Item v = f[parent];
      EmulAdjustHeap(f, parent, len, v);
      if (parent == 0) break;
      parent--;
    }
  }
  long last = len;
  while (last > 1) {
    --last;
    Item v = f[last];
    f[last] = f[0];
    EmulAdjustHeap(f, 0, last, v);
  }
}
void EmulIntroLoop(Item* a, long first, long last, long depth) {
  while (last - first > 16) {
    if (depth == 0) {
      EmulHeapSort(a + first, last - first);
      return;
    }
    --depth;
    long mid = first + (last - first) / 2;
    long pa = first + 1, pb = mid, pc = last - 1;
    if (Before(a[pa], a[pb])) {
      if (Before(a[pb], a[pc])) std::swap(a[first], a[pb]);
      else if (Before(a[pa], a[pc])) std::swap(a[first], a[pc]);
      else std::swap(a[first], a[pa]);
    } else if (Before(a[pa], a[pc])) std::swap(a[first], a[pa]);
    else if (Before(a[pb], a[pc])) std::swap(a[first], a[pc]);
    else std::swap(a[first], a[pb]);
    long lo = first + 1, hi = last;
    while (true) {
      while (Before(a[lo], a[first])) ++lo;
      --hi;
      while (Before(a[first], a[hi])) --hi;
      if (!(lo < hi)) break;
      std::swap(a[lo], a[hi]);
      ++lo;
    }
    EmulIntroLoop(a, lo, last, depth);
    last = lo;
  }
}

}  // namespace

extern "C" {

int rso_step(const rso_config* cfg, int32_t n_cells, rso_io* io, int32_t n_threads) {
  if (!cfg || !io || n_cells < 0) return 1;
  const bool transport = cfg->algo == 8 || cfg->algo == 9 || cfg->algo == 10 || cfg->algo == 101 || cfg->algo == 103;
  if (cfg->algo != 1 && cfg->algo != 7 && cfg->algo != 11 && !transport) return 2;
  if (transport && (!io->rand2 || !io->slice_offset)) return 3;
  if ((cfg->algo == 7 || cfg->algo == 11) && !io->nvs_ewma) return 3;
  if (cfg->algo == 11 && (!io->rand2 || io->rand_stride < 300)) return 3;
  if (cfg->n_bearers == 2 && (cfg->algo == 1 || !io->queue_bytes)) return 4;   /* id 1 schedules flows: one user per bearer */
  int32_t row_m1[27];
  if (cfg->tbs_row_m1) std::memcpy(row_m1, cfg->tbs_row_m1, sizeof(row_m1));
  else DefaultRowM1(row_m1);
  if (n_threads <= 1) {
    for (int b = 0; b < n_cells; ++b) StepCell(cfg, io, b, row_m1);
    return 0;
  }
  std::vector<std::thread> pool;
  for (int t = 0; t < n_threads; ++t) {
    pool.emplace_back([=]() {
      for (int b = t; b < n_cells; b += n_threads) StepCell(cfg, io, b, row_m1);
    });
  }
  for (auto& th : pool) th.join();
  return 0;
}

double rso_eesm_effective_sinr(const double* sinr_db, int32_t n) {
  std::vector<double> v(sinr_db, sinr_db + n);
  return Eesm(v);
}
int32_t rso_cqi_from_sinr(double sinr_db) { return CqiFromSinr(sinr_db); }
double rso_sinr_from_cqi(int32_t cqi) { return SinrFromCqi(cqi); }
int32_t rso_mcs_from_cqi(int32_t cqi) { return McsFromCqi(cqi); }
int32_t rso_tbs_from_mcs(int32_t mcs, int32_t n_rbs, const int32_t* row_m1) {
  int32_t def[27];
  if (!row_m1) {
    DefaultRowM1(def);
    row_m1 = def;
  }
  return TbsN(mcs, n_rbs, row_m1);
}
double rso_efficiency_from_cqi(int32_t cqi) { return EffFromCqi(cqi); }
void rso_default_row_m1(int32_t* out27) { DefaultRowM1(out27); }

void rso_std_sort_desc(const double* keys, int32_t n, int32_t* perm_out) {
  std::vector<coord_cqi_t> v;
  for (int i = 0; i < n; ++i) v.emplace_back(coord_t(i, 0), keys[i]);
  std::sort(v.begin(), v.end(), [](coord_cqi_t a, coord_cqi_t b) { return a.second > b.second; });
  for (int i = 0; i < n; ++i) perm_out[i] = v[i].first.first;
}

void rso_introsort_emul_desc(const double* keys, int32_t n, int32_t depth_limit, int32_t* perm_out) {
  std::vector<Item> a(n);
  for (int i = 0; i < n; ++i) a[i] = Item{keys[i], i};
  if (n > 0) {
    long depth = depth_limit;
    if (depth < 0) {
      long lg = 0;
      for (long m = n; m > 1; m >>= 1) lg++;
      depth = 2 * lg;
    }
    EmulIntroLoop(a.data(), 0, n, depth);
    /* __final_insertion_sort == a stable insertion sort of what is there now */
    for (long i = 1; i < n; ++i) {
      Item v = a[i];
      long j = i;
      while (j > 0 && Before(v, a[j - 1])) {
        a[j] = a[j - 1];
        --j;
      }
      a[j] = v;
    }
  }
  for (int i = 0; i < n; ++i) perm_out[i] = a[i].idx;
}

}  /* extern "C" */

extern "C" void rso_diag_enable(int on) {
  g_diag_on.store(on);
  if (on) for (auto& x : g_diag_stop) x.store(0);
}
extern "C" void rso_diag_stop_hist(uint64_t* out66) {
  for (int i = 0; i < 66; ++i) out66[i] = g_diag_stop[i].load();
}
