/* oracle/dropin/dropin_replay.cpp -- the product's LTE-Sim plug-in (radiosaber_b200/host/rs_gpu_scheduler.h -> C ABI ->
 * CUDA), compiled unchanged against the stand-in classes of oracle/dropin/ltesim.h and driven through a golden record of
 * the unmodified reference.  TEST INFRASTRUCTURE ONLY (tests/test_dropin_gpu.py).
 *
 * Each TTI the replay sets what the simulator would hand the scheduler -- Simulator::Now(), the CQI in the eNB's UE
 * records, which bearers have packets, their queue sizes and head-of-line delays, and the rand() values the process
 * would return -- calls RsGpuScheduler::DoSchedule() and records what came out exactly like oracle/ref_harness.cpp
 * records the reference classes (same RSGOLD1 stream; targets, quotas and final CQI parsed from the scheduler's own
 * stdout lines; the bearers' EWMA rates, byte and RB counters chained on their own state from the first TTI on).
 *
 *   dropin_replay --algo ID --config cfg.json --replay inputs.bin --out rec.bin [--alloc-log f] [--rand-log f]
 *                 [--bearer-out f] [--log-out PREFIX]
 *
 * inputs.bin (little endian): int32 T, U, S, G, NB (bearers per UE slot: 1, or 2 = slot i holds the bearer of priority
 * i), first_ts (PacketScheduler's TTI count at the first TTI); uint8 exists[U][NB]; int32 app_id[U][NB] (the eNB's
 * bearer container is in application order); double avg_rate0[U][NB]; int32 tx_bytes0[U][NB]; double last_update0;
 * double slice_state0[S]; uint8 cqi[T][U][G]; then per TTI: double now, uint8 has_packets[U][NB], int32 queue[U][NB]
 * (what SelectFlowsToSchedule takes as dataToTransmit: 100000000 = infinite buffer), double hol[U][NB], int32 n,
 * int32 rand[n].
 * --bearer-out: per TTI and bearer slot [U][NB] double avg_rate, int32 tx_bytes, int32 pad, uint64 cum_bytes, cum_rbs
 * after the TTI (zeros where no bearer).  --log-out: what the plug-in printed, PREFIX.stdout / PREFIX.stderr.  The
 * per-UE fields of the record hold the last bearer of each UE in container order, like oracle/ref_harness.cpp.  */
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>

#include "ltesim.h"
#include "../../radiosaber_b200/host/rs_gpu_scheduler.h"

static double g_now = 0;
double SimulatorNow() { return g_now; }

/* rand() of the whole binary: inside DoSchedule it returns the TTI's recorded values, in order; running past them is an
 * error (the plug-in drew more values than the reference did) */
static std::vector<int32_t> g_script;
static size_t g_script_pos = 0;
static std::vector<int32_t> g_drawn;
static bool g_overrun = false;
extern "C" int rand(void) {
  int32_t v = 0;
  if (g_script_pos < g_script.size()) v = g_script[g_script_pos++];
  else g_overrun = true;
  g_drawn.push_back(v);
  return v;
}
extern "C" void srand(unsigned) {}

struct Reader {
  std::vector<uint8_t> raw;
  size_t pos = 0;
  template <typename T>
  void Get(T* out, size_t n) {
    if (pos + sizeof(T) * n > raw.size()) throw std::runtime_error("short --replay file");
    memcpy(out, raw.data() + pos, sizeof(T) * n);
    pos += sizeof(T) * n;
  }
  template <typename T>
  T Get1() { T v; Get(&v, 1); return v; }
};

/* std::cout / std::cerr (the plug-in's per-bearer lines) into the TTI's texts; restored on any exit */
struct CaptureStreams {
  std::streambuf* out;
  std::streambuf* err;
  CaptureStreams(std::stringstream& text, std::stringstream& etext)
      : out(std::cout.rdbuf(text.rdbuf())), err(std::cerr.rdbuf(etext.rdbuf())) {}
  ~CaptureStreams() { std::cout.rdbuf(out); std::cerr.rdbuf(err); }
};

static FILE* g_out = nullptr;
template <typename T>
static void Put(const T* p, size_t n) { fwrite(p, sizeof(T), n, g_out); }
template <typename T>
static void Put1(T v) { Put(&v, 1); }

int main(int argc, char** argv) {
  std::string config, replay, out, alloc_log, rand_log, bearer_out, log_out;
  int algo = 9;
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    if (i + 1 >= argc) { fprintf(stderr, "missing value for %s\n", a.c_str()); return 2; }
    std::string v = argv[++i];
    if (a == "--algo") algo = atoi(v.c_str());
    else if (a == "--config") config = v;
    else if (a == "--replay") replay = v;
    else if (a == "--out") out = v;
    else if (a == "--alloc-log") alloc_log = v;
    else if (a == "--rand-log") rand_log = v;
    else if (a == "--bearer-out") bearer_out = v;
    else if (a == "--log-out") log_out = v;
    else { fprintf(stderr, "unknown arg %s\n", a.c_str()); return 2; }
  }
  if (config.empty() || replay.empty() || out.empty()) {
    fprintf(stderr, "usage: dropin_replay --algo ID --config cfg.json --replay inputs.bin --out rec.bin [--alloc-log f] [--rand-log f]\n");
    return 2;
  }
  Reader in;
  {
    FILE* f = fopen(replay.c_str(), "rb");
    if (!f) { fprintf(stderr, "cannot open %s\n", replay.c_str()); return 2; }
    fseek(f, 0, SEEK_END);
    in.raw.resize(ftell(f));
    fseek(f, 0, SEEK_SET);
    if (fread(in.raw.data(), 1, in.raw.size(), f) != in.raw.size()) { fprintf(stderr, "short read %s\n", replay.c_str()); return 2; }
    fclose(f);
  }
  g_out = fopen(out.c_str(), "wb");
  FILE* falloc = alloc_log.empty() ? nullptr : fopen(alloc_log.c_str(), "wb");
  FILE* frand = rand_log.empty() ? nullptr : fopen(rand_log.c_str(), "wb");
  FILE* fbearer = bearer_out.empty() ? nullptr : fopen(bearer_out.c_str(), "wb");
  FILE* flog_out = log_out.empty() ? nullptr : fopen((log_out + ".stdout").c_str(), "w");
  FILE* flog_err = log_out.empty() ? nullptr : fopen((log_out + ".stderr").c_str(), "w");
  if (!g_out || (!alloc_log.empty() && !falloc) || (!rand_log.empty() && !frand) || (!bearer_out.empty() && !fbearer) ||
      (!log_out.empty() && (!flog_out || !flog_err))) {
    fprintf(stderr, "cannot write outputs\n");
    return 2;
  }

  int rc = 0;
  try {
    const int T = in.Get1<int32_t>(), U = in.Get1<int32_t>(), S = in.Get1<int32_t>(), G = in.Get1<int32_t>();
    const int NB = in.Get1<int32_t>(), first_ts = in.Get1<int32_t>();
    const int R = 512, rbg = get_rbg_size(R);
    if (G * rbg != R) throw std::runtime_error("the record's RBG count does not match the 512-RB band");
    if (NB < 1 || NB > MAX_BEARERS) throw std::runtime_error("bearers per UE outside 1..MAX_BEARERS");

    /* the cell: one eNB, U UEs (node id = user id), NB bearer slots each; slot i is the bearer of priority i */
    ENodeB enb;
    enb.ues.resize(U);
    std::vector<NetworkNode> ue_nodes(U);
    std::vector<RadioBearer> bearers((size_t)U * NB);
    std::vector<uint8_t> exists((size_t)U * NB);
    std::vector<int32_t> app_id((size_t)U * NB), tx0((size_t)U * NB);
    std::vector<double> avg0((size_t)U * NB), state0(S);
    in.Get(exists.data(), exists.size());
    in.Get(app_id.data(), app_id.size());
    in.Get(avg0.data(), avg0.size());
    in.Get(tx0.data(), tx0.size());
    const double last0 = in.Get1<double>();
    in.Get(state0.data(), S);
    std::vector<int> order;   /* bearer slots in container order: by application id */
    for (int k = 0; k < U * NB; ++k)
      if (exists[k]) order.push_back(k);
    std::sort(order.begin(), order.end(), [&](int a, int b) { return app_id[a] < app_id[b]; });
    RrcEntity::RadioBearersContainer* container = enb.GetProtocolStack()->GetRrcEntity()->GetRadioBearerContainer();
    for (int u = 0; u < U; ++u) ue_nodes[u].id = u;
    for (int k : order) {
      RadioBearer& b = bearers[k];
      b.user_id = k / NB;
      b.priority = k % NB;
      b.destination = &ue_nodes[k / NB];
      b.application.id = app_id[k];
      b.m_averageTransmissionRate = avg0[k];
      b.m_transmittedBytes = tx0[k];
      b.m_lastUpdate = last0;
      container->push_back(&b);
    }
    std::vector<uint8_t> cqi_all((size_t)T * U * G);
    in.Get(cqi_all.data(), cqi_all.size());

    MacEntity mac;
    mac.device = &enb;
    RsGpuScheduler sched(config, algo);
    sched.SetMacEntity(&mac);
    if ((int)sched.user_to_slice_.size() != U || sched.num_slices_ != S) throw std::runtime_error("config does not match the record");
    sched.slice_state_ = state0;
    sched.SetTimeStamp(first_ts);

    const char magic[8] = {'R', 'S', 'G', 'O', 'L', 'D', '1', 0};
    Put(magic, 8);
    Put1<int32_t>(algo); Put1<int32_t>(S); Put1<int32_t>(U); Put1<int32_t>(R); Put1<int32_t>(rbg);
    for (int s = 0; s < S; ++s) Put1<double>(sched.slice_weights_[s]);
    for (int s = 0; s < S; ++s) {
      const SchedulerAlgoParam& p = sched.slice_algo_params_[s];
      const int32_t v[4] = {p.alpha, p.beta, p.epsilon, p.psi};
      Put(v, 4);
    }
    for (int u = 0; u < U; ++u) Put1<int32_t>(sched.user_to_slice_[u]);

    std::vector<uint8_t> has((size_t)U * NB);
    std::vector<int32_t> queue((size_t)U * NB);
    std::vector<double> hol((size_t)U * NB);
    for (int t = 0; t < T; ++t) {
      g_now = in.Get1<double>();
      in.Get(has.data(), has.size());
      in.Get(queue.data(), queue.size());
      in.Get(hol.data(), hol.size());
      g_script.resize(in.Get1<int32_t>());
      in.Get(g_script.data(), g_script.size());
      for (int k : order) {
        RadioBearer& b = bearers[k];
        b.has_packets = has[k] != 0;
        b.queue_size = queue[k];
        b.application.type = queue[k] == 100000000 ? Application::APPLICATION_TYPE_INFINITE_BUFFER
                                                   : Application::APPLICATION_TYPE_INTERNET_FLOW;
        b.hol_delay = hol[k];
      }
      for (int u = 0; u < U; ++u) {
        std::vector<int>& v = enb.ues[u].cqi;
        v.resize(R);
        for (int r = 0; r < R; ++r) v[r] = cqi_all[((size_t)t * U + u) * G + r / rbg];
      }

      std::vector<double> avg_before(U), last_update(U), state_before = sched.slice_state_;
      std::vector<int32_t> tx_before(U);
      for (int k : order) {
        const RadioBearer& b = bearers[k];
        avg_before[b.user_id] = b.m_averageTransmissionRate;
        tx_before[b.user_id] = b.m_transmittedBytes;
        last_update[b.user_id] = b.m_lastUpdate;
      }

      g_script_pos = 0;
      g_drawn.clear();
      std::stringstream text, etext;
      {
        CaptureStreams capture(text, etext);
        sched.DoSchedule();
      }
      if (flog_out) {
        fputs(text.str().c_str(), flog_out);
        fputs(etext.str().c_str(), flog_err);
      }
      if (g_overrun) throw std::runtime_error("the plug-in drew more rand() values than the reference did");

      const int32_t rand2[2] = {g_drawn.size() > 0 ? g_drawn[0] : 0, g_drawn.size() > 1 ? g_drawn[1] : 0};
      if (frand) {
        const int32_t n = (int32_t)g_drawn.size();
        fwrite(&n, 4, 1, frand);
        fwrite(g_drawn.data(), 4, g_drawn.size(), frand);
      }

      /* CollectUsers and the NVS fill of oracle/ref_harness.cpp */
      std::vector<uint8_t> active(U, 0), final_cqi(U, 0);
      std::vector<int16_t> rbg_to_ue(G, -1), grants;
      std::vector<int32_t> bits(U, 0), target(S, 0), quota(S, 0);
      int32_t nvs_slice = -1;
      for (auto* usr : *sched.GetUsersToSchedule()) {
        const int id = usr->GetUserID();
        active[id] = 1;
        bits[id] = usr->GetAllocatedBits();
        for (int rb : *usr->GetListOfAllocatedRBs())
          if (rb % rbg == 0) {
            rbg_to_ue[rb / rbg] = (int16_t)id;
            grants.push_back((int16_t)id);
            grants.push_back((int16_t)(rb / rbg));
          }
      }
      if (falloc) {
        const int32_t n = (int32_t)(grants.size() / 2);
        fwrite(&n, 4, 1, falloc);
        fwrite(grants.data(), 2, grants.size(), falloc);
      }
      if (algo == 7 || algo == 11) {
        std::fill(active.begin(), active.end(), (uint8_t)1);
        if (!sched.GetUsersToSchedule()->empty()) nvs_slice = sched.user_to_slice_[sched.GetUsersToSchedule()->at(0)->GetUserID()];
      }
      /* targets / quotas and final CQI from what the scheduler printed (downlink-transport-scheduler.cpp:523-527, 637-649) */
      std::string line;
      while (std::getline(text, line)) {
        if (line.compare(0, 9, "slice_id,") == 0) {
          const char* p = line.c_str();
          while ((p = strchr(p, '(')) != nullptr) {
            int i, tg, q;
            if (sscanf(p, "(%d, %d, %d)", &i, &tg, &q) == 3 && i >= 0 && i < S) { target[i] = tg; quota[i] = q; }
            ++p;
          }
        } else if (line.compare(0, 5, "User(") == 0) {
          const int uid = atoi(line.c_str() + 5);
          const size_t k = line.rfind("final_cqi: ");
          if (k != std::string::npos && uid >= 0 && uid < U) final_cqi[uid] = (uint8_t)atoi(line.c_str() + k + 11);
        }
      }

      std::vector<uint8_t> cqi((size_t)U * R);
      for (int u = 0; u < U; ++u)
        for (int r = 0; r < R; ++r) cqi[(size_t)u * R + r] = (uint8_t)enb.ues[u].cqi[r];
      Put1<int32_t>(0x54544921); Put1<int32_t>(t); Put1<double>(g_now);
      Put(avg_before.data(), U); Put(tx_before.data(), U); Put(last_update.data(), U);
      Put(state_before.data(), S);
      Put(cqi.data(), cqi.size()); Put(active.data(), U); Put(rand2, 2);
      Put(rbg_to_ue.data(), G); Put(bits.data(), U); Put(final_cqi.data(), U);
      Put(target.data(), S); Put(quota.data(), S); Put1<int32_t>(nvs_slice);
      std::vector<double> avg_after(U);
      std::vector<int32_t> tx_after(U);
      std::vector<uint64_t> cum_bytes(U), cum_rbs(U);
      for (int k : order) {
        const RadioBearer& b = bearers[k];
        avg_after[b.user_id] = b.m_averageTransmissionRate;
        tx_after[b.user_id] = b.m_transmittedBytes;
        cum_bytes[b.user_id] = b.m_cumulativeBytes;
        cum_rbs[b.user_id] = b.m_cumulativeRBs;
      }
      Put(avg_after.data(), U); Put(tx_after.data(), U); Put(cum_bytes.data(), U); Put(cum_rbs.data(), U);
      Put(sched.slice_state_.data(), S);
      if (fbearer)
        for (int k = 0; k < U * NB; ++k) {
          const RadioBearer& b = bearers[k];
          const bool e = exists[k] != 0;
          const double av = e ? b.m_averageTransmissionRate : 0.0;
          const int32_t tx[2] = {e ? b.m_transmittedBytes : 0, 0};
          const uint64_t cu[2] = {e ? b.m_cumulativeBytes : 0, e ? b.m_cumulativeRBs : 0};
          fwrite(&av, 8, 1, fbearer);
          fwrite(tx, 4, 2, fbearer);
          fwrite(cu, 8, 2, fbearer);
        }
    }
  } catch (const std::exception& e) {
    fprintf(stderr, "dropin_replay: %s\n", e.what());
    rc = 3;
  }
  fclose(g_out);
  if (falloc) fclose(falloc);
  if (frand) fclose(frand);
  if (fbearer) fclose(fbearer);
  if (flog_out) fclose(flog_out);
  if (flog_err) fclose(flog_err);
  return rc;
}
