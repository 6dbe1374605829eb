/* rs_batch -- C++ host program for batch runs: thousands of independent cells of one slice configuration (or of
 * several of the same shape, one per cell) on one or several GPUs of a box through the C ABI of include/rs_sched.h (+ include/rs_sched_nccl.h for --gpus N).
 *
 * It takes what the reference's SingleCellWithI scenario takes -- the scheduler id and the JSON slice config
 * (src/scenarios/single-cell-with-interference.h:94-123, 214-248; the scheduler constructors parse the same file,
 * downlink-transport-scheduler.cpp:55-97) -- plus a batch size, and either replays the cqi-traces-noise0 files
 * through per-cell UE->trace mappings (enb-mac-entity.cc:42-56, 160-193) or draws synthetic CQI on the device.
 * Output: one JSON line with the per-slice totals the reference's plotters compute from its logs
 * (plot_throughput.py:26-98) and, with --log-cell, the reference's own log text for one cell of the batch.
 *
 *   rs_batch --algo 9 --config cfg.json --cells 4096 --ttis 1000 [--seed 1]
 *            [--config cfg2.json ...]           more slice configs (rs_create_profiles): cell b uses config b % P; every
 *                                               config must expand to the same slices and UEs; one output line per
 *                                               config, over that config's cells
 *            [--traces DIR --mapping FILE]      replay DIR/ue<id>.log; cell b, UE u replays map[(u + 7 b) % n]
 *            [--trace-rows N]                   lines per trace file (475 in cqi-traces-noise0)
 *            [--log-cell B --log-prefix P]      P.stdout / P.stderr as the reference prints them for cell B
 *            [--gpus N]                         cells block-partitioned over N GPUs, one host thread per GPU, no traffic
 *                                               between GPUs inside a TTI; ONE ncclReduce of the per-slice totals at the
 *                                               end (SURVEY 8e; reference analogue: one process per seed + a sum in
 *                                               plot_throughput.py:26-56)
 *
 * Host logic only; every scheduling decision is made by the CUDA kernels behind the ABI (no CPU fallback).
 */
#include <cctype>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <sstream>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "rs_sched.h"
#include "rs_sched_nccl.h"

namespace {

/* ---- the little JSON the slice configs use: objects, arrays, numbers (strings are skipped over) ---------- */
struct Json {
  enum Kind { Null, Num, Arr, Obj, Str } kind = Null;
  double num = 0;
  std::vector<Json> arr;
  std::map<std::string, Json> obj;
  const Json& operator[](const char* k) const {
    static const Json none;
    auto it = obj.find(k);
    return it == obj.end() ? none : it->second;
  }
  int as_int() const { return (int)num; }
};

struct Parser {
  const std::string& s;
  size_t i = 0;
  explicit Parser(const std::string& text) : s(text) {}
  void ws() { while (i < s.size() && isspace((unsigned char)s[i])) ++i; }
  std::string str() {
    std::string out;
    ++i;
    while (i < s.size() && s[i] != '"') { if (s[i] == '\\') ++i; out += s[i++]; }
    ++i;
    return out;
  }
  Json value() {
    ws();
    Json v;
    if (i >= s.size()) throw std::runtime_error("config: unexpected end");
    if (s[i] == '{') {
      v.kind = Json::Obj;
      ++i;
      for (ws(); s[i] != '}'; ws()) {
        if (s[i] == ',') { ++i; continue; }
        std::string k = str();
        ws();
        if (s[i] != ':') throw std::runtime_error("config: ':' expected");
        ++i;
        v.obj[k] = value();
      }
      ++i;
    } else if (s[i] == '[') {
      v.kind = Json::Arr;
      ++i;
      for (ws(); s[i] != ']'; ws()) {
        if (s[i] == ',') { ++i; continue; }
        v.arr.push_back(value());
      }
      ++i;
    } else if (s[i] == '"') {
      v.kind = Json::Str;
      str();
    } else {
      char* end = nullptr;
      v.kind = Json::Num;
      v.num = strtod(s.c_str() + i, &end);
      if (end == s.c_str() + i) throw std::runtime_error("config: value expected");
      i = (size_t)(end - s.c_str());
    }
    return v;
  }
};

void check(int rc, const char* what) {
  if (rc != RS_OK) throw std::runtime_error(std::string(what) + ": " + rs_last_error());
}
void cu(cudaError_t e, const char* what) {
  if (e != cudaSuccess) throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}

struct Args {
  int algo = 9, cells = 4096, ttis = 1000, log_cell = -1, trace_rows = 475;   /* 475 lines: enb-mac-entity.cc:181 */
  int gpus = 1;
  uint64_t seed = 1;
  std::vector<std::string> configs;
  std::string traces, mapping, log_prefix;
};

struct Profile {   /* one slice config, expanded like the scheduler constructors do */
  std::vector<double> weight;
  std::vector<int32_t> params, u2s;
};

struct Setup {   /* what every shard shares */
  Args a;
  int S = 0, U = 0;
  std::vector<Profile> prof;     /* [P]; cell b of the batch uses prof[b % P] */
  bool replay = false;
  int n_traces = 0;
  std::vector<uint8_t> traces;   /* [n_traces][rows][R] */
  std::vector<int32_t> map;
  std::vector<double> now, dt;
};

struct ShardResult {
  double ms = 0;                 /* host clock around the synchronised scheduling calls */
  std::vector<uint64_t> stats;   /* [P][4][S] of this shard's cells (single GPU) or of ALL cells (root after the reduce) */
  std::string log_out, log_err, error;
};

constexpr int R = 512, RBG = 8, G = R / RBG;   /* 100 MHz: bandwidth-manager.cpp:98-102, eesm-effective-sinr.h:82-103 */

/* Cells [cell0, cell0 + nb) of the batch on GPU `gpu`.  comm != NULL: join the end-of-run reduce (root = rank 0). */
void run_shard(const Setup& su, int gpu, int rank, int cell0, int nb, void* comm, ShardResult* res) {
  const Args& a = su.a;
  const int S = su.S, U = su.U, B = nb, T = a.ttis, P = (int)su.prof.size();
  std::vector<rs_config> cfgs((size_t)P);
  for (int p = 0; p < P; ++p) {
    rs_config& cfg = cfgs[(size_t)p];
    memset(&cfg, 0, sizeof cfg);
    cfg.algo = a.algo;
    cfg.n_slices = S;
    cfg.n_ues = U;
    cfg.n_rbs = R;
    cfg.rbg_size = RBG;
    cfg.cqi_per_rb = 2;   /* 4 bits per RBG: what a CQI is on the air */
    cfg.data_to_transmit = 100000000;
    cfg.weight = su.prof[(size_t)p].weight.data();
    cfg.params = su.prof[(size_t)p].params.data();
    cfg.ue_to_slice = su.prof[(size_t)p].u2s.data();
  }
  rs_handle* h = nullptr;
  if (P == 1) {
    check(rs_create(cfgs.data(), B, gpu, &h), "rs_create");
  } else {
    /* this shard's slice of the assignment: cell cell0 + b of the batch uses config (cell0 + b) % P */
    std::vector<int32_t> cell_profile((size_t)B);
    for (int b = 0; b < B; ++b) cell_profile[(size_t)b] = (int32_t)((cell0 + b) % P);
    check(rs_create_profiles(cfgs.data(), P, cell_profile.data(), B, gpu, &h), "rs_create_profiles");
  }
  cu(cudaSetDevice(gpu), "cudaSetDevice");   /* this thread's own allocations below */
  const int n_draws = rs_rand_draws_per_cell_tti(h);
  const int n_rows = a.trace_rows;
  const bool replay = su.replay;
  std::vector<int32_t> ue_trace;
  if (replay) {
    const size_t n_map = su.map.size();
    ue_trace.resize((size_t)B * U);
    for (int b = 0; b < B; ++b)   /* every cell its own mapping (the reference: map[u % n] for its one cell) */
      for (int u = 0; u < U; ++u) ue_trace[(size_t)b * U + u] = su.map[(size_t)(u + 7 * (int64_t)(cell0 + b)) % n_map];
    check(rs_set_traces(h, su.traces.data(), su.n_traces, n_rows, ue_trace.data()), "rs_set_traces");
  }

  /* ---- run in blocks of TB TTIs with everything resident on the device ------------------------------- */
  const int TB = 16;
  uint8_t* d_cqi = nullptr;
  int32_t* d_draws = nullptr;
  int16_t *d_rbg = nullptr, *d_gue = nullptr, *d_grbg = nullptr;   /* d_g*: id 10's grant list */
  int32_t* d_gn = nullptr;
  size_t n_list = 0;   /* entries per cell of the grant list */
  int32_t *d_bits = nullptr, *d_tgt = nullptr, *d_quo = nullptr;
  uint8_t* d_fc = nullptr;
  const size_t row = G / 2;
  if (!replay) cu(cudaMalloc(&d_cqi, (size_t)TB * B * U * row), "cudaMalloc");
  if (n_draws > 0) cu(cudaMalloc(&d_draws, sizeof(int32_t) * (size_t)TB * B * n_draws), "cudaMalloc");
  const int lc = a.log_cell - cell0;   /* the logged cell, if it lives in this shard */
  const bool want_log = lc >= 0 && lc < B && !a.log_prefix.empty();
  rs_log* lg = nullptr;
  std::vector<int16_t> h_rbg, h_gue, h_grbg;
  std::vector<int32_t> h_bits, h_tgt, h_quo;
  std::vector<uint8_t> h_fc, h_cqi;
  rs_outputs out;
  memset(&out, 0, sizeof out);
  if (want_log) {
    check(rs_log_create(&cfgs[(size_t)(a.log_cell % P)], &lg), "rs_log_create");   /* the logged cell's own slices */
    cu(cudaMalloc(&d_rbg, sizeof(int16_t) * (size_t)TB * B * G), "cudaMalloc");
    cu(cudaMalloc(&d_bits, sizeof(int32_t) * (size_t)TB * B * U), "cudaMalloc");
    cu(cudaMalloc(&d_fc, (size_t)TB * B * U), "cudaMalloc");
    cu(cudaMalloc(&d_tgt, sizeof(int32_t) * (size_t)TB * B * S), "cudaMalloc");
    cu(cudaMalloc(&d_quo, sizeof(int32_t) * (size_t)TB * B * S), "cudaMalloc");
    out.rbg_to_ue = d_rbg; out.tbs_bits = d_bits; out.final_cqi = d_fc; out.slice_target = d_tgt; out.slice_quota = d_quo;
    if (a.algo == 10) {   /* the logged cell's every grant: up to S*G */
      check(rs_set_grant_list_len(h, std::max(S * G, 2 * G)), "rs_set_grant_list_len");
      n_list = rs_grant_list_len(h);
      cu(cudaMalloc(&d_gn, sizeof(int32_t) * (size_t)TB * B), "cudaMalloc");
      cu(cudaMalloc(&d_gue, sizeof(int16_t) * (size_t)TB * B * n_list), "cudaMalloc");
      cu(cudaMalloc(&d_grbg, sizeof(int16_t) * (size_t)TB * B * n_list), "cudaMalloc");
      out.alloc_n = d_gn; out.alloc_ue = d_gue; out.alloc_rbg = d_grbg;
      h_gue.resize(n_list); h_grbg.resize(n_list);
    }
    h_rbg.resize(G); h_bits.resize(U); h_fc.resize(U); h_tgt.resize(S); h_quo.resize(S); h_cqi.resize((size_t)U * row);
  }
  std::vector<int32_t> trow(TB);
  for (int t0 = 0; t0 < T; t0 += TB) {
    const int n = std::min(TB, T - t0);
    if (!replay) check(rs_synth_cqi(h, a.seed, cell0, t0, n, d_cqi), "rs_synth_cqi");
    if (n_draws > 0) check(rs_synth_rand2(h, a.seed, cell0, t0, n, d_draws), "rs_synth_rand2");
    check(rs_sync(h), "rs_sync");
    const auto w0 = std::chrono::steady_clock::now();
    if (replay) {
      /* all UEs report in the same TTI, every 40 TTIs from the first (phy/ue-lte-phy.cpp:215-232) */
      for (int k = 0; k < n; ++k) trow[k] = rs_trace_row(su.now[(t0 + k) - (t0 + k) % 40], n_rows);
      check(rs_run_traces_device(h, n, trow.data(), d_draws, nullptr, 0, su.dt.data() + t0, want_log ? &out : nullptr, TB), "rs_run_traces_device");
    } else {
      check(rs_run_device(h, n, d_cqi, (int64_t)B * U * row, 1, d_draws, nullptr, 0, su.dt.data() + t0, want_log ? &out : nullptr, TB), "rs_run_device");
    }
    check(rs_sync(h), "rs_sync");
    res->ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - w0).count();
    if (want_log) {
      for (int k = 0; k < n; ++k) {
        const size_t tb = (size_t)k * B + lc;
        if (replay) {
          /* the CQI vectors the cell's UEs hold this TTI, rebuilt from the traces in the 4-bit layout */
          for (int u = 0; u < U; ++u) {
            const int tid = ue_trace[(size_t)lc * U + u];
            const uint8_t* src = su.traces.data() + ((size_t)tid * n_rows + (trow[k] < 0 ? 0 : trow[k])) * R;
            for (int g = 0; g < G; g += 2) {
              const int lo = trow[k] < 0 ? 10 : src[(size_t)g * RBG], hi = trow[k] < 0 ? 10 : src[(size_t)(g + 1) * RBG];
              h_cqi[(size_t)u * row + g / 2] = (uint8_t)(lo | (hi << 4));
            }
          }
        } else {
          cu(cudaMemcpy(h_cqi.data(), d_cqi + tb * U * row, (size_t)U * row, cudaMemcpyDeviceToHost), "copy");
        }
        cu(cudaMemcpy(h_rbg.data(), d_rbg + tb * G, sizeof(int16_t) * G, cudaMemcpyDeviceToHost), "copy");
        cu(cudaMemcpy(h_bits.data(), d_bits + tb * U, sizeof(int32_t) * U, cudaMemcpyDeviceToHost), "copy");
        cu(cudaMemcpy(h_fc.data(), d_fc + tb * U, U, cudaMemcpyDeviceToHost), "copy");
        cu(cudaMemcpy(h_tgt.data(), d_tgt + tb * S, sizeof(int32_t) * S, cudaMemcpyDeviceToHost), "copy");
        cu(cudaMemcpy(h_quo.data(), d_quo + tb * S, sizeof(int32_t) * S, cudaMemcpyDeviceToHost), "copy");
        /* PacketScheduler::m_ts counts TTIs since the eNB was created: 100 at the first TTI with bearers */
        const uint64_t ts = 100 + (uint64_t)(t0 + k);
        if (a.algo == 10) {
          int32_t n_grants = 0;
          cu(cudaMemcpy(&n_grants, d_gn + tb, sizeof n_grants, cudaMemcpyDeviceToHost), "copy");
          cu(cudaMemcpy(h_gue.data(), d_gue + tb * n_list, sizeof(int16_t) * n_list, cudaMemcpyDeviceToHost), "copy");
          cu(cudaMemcpy(h_grbg.data(), d_grbg + tb * n_list, sizeof(int16_t) * n_list, cudaMemcpyDeviceToHost), "copy");
          check(rs_log_tti_grants(lg, ts, h_cqi.data(), n_grants, h_gue.data(), h_grbg.data(), h_bits.data(), h_fc.data(),
                                  h_tgt.data(), h_quo.data()), "rs_log_tti_grants");
        } else {
          check(rs_log_tti(lg, ts, h_cqi.data(), h_rbg.data(), h_bits.data(), h_fc.data(), h_tgt.data(), h_quo.data()), "rs_log_tti");
        }
      }
    }
  }
  res->stats.assign((size_t)4 * S * P, 0);
  if (comm) {
    if (rs_reduce_stats(h, comm, 0, res->stats.data()) != RS_OK)
      throw std::runtime_error(std::string("rs_reduce_stats: ") + rs_nccl_last_error());
  } else {
    check(rs_get_stats(h, res->stats.data()), "rs_get_stats");
  }
  (void)rank;
  if (lg) {
    res->log_out = rs_log_stdout(lg, nullptr);
    res->log_err = rs_log_stderr(lg, nullptr);
    rs_log_destroy(lg);
  }
  rs_destroy(h);
  cudaFree(d_cqi); cudaFree(d_draws); cudaFree(d_rbg); cudaFree(d_bits); cudaFree(d_fc); cudaFree(d_tgt); cudaFree(d_quo); cudaFree(d_gn); cudaFree(d_gue); cudaFree(d_grbg);
}

}  // namespace

int main(int argc, char** argv) {
  try {
    Setup su;
    Args& a = su.a;
    for (int i = 1; i < argc; ++i) {
      const std::string k = argv[i];
      auto next = [&]() -> std::string { if (i + 1 >= argc) throw std::runtime_error("missing value for " + k); return argv[++i]; };
      if (k == "--algo") a.algo = atoi(next().c_str());
      else if (k == "--config") a.configs.push_back(next());
      else if (k == "--cells") a.cells = atoi(next().c_str());
      else if (k == "--ttis") a.ttis = atoi(next().c_str());
      else if (k == "--seed") a.seed = strtoull(next().c_str(), nullptr, 10);
      else if (k == "--traces") a.traces = next();
      else if (k == "--mapping") a.mapping = next();
      else if (k == "--trace-rows") a.trace_rows = atoi(next().c_str());
      else if (k == "--log-cell") a.log_cell = atoi(next().c_str());
      else if (k == "--log-prefix") a.log_prefix = next();
      else if (k == "--gpus") a.gpus = atoi(next().c_str());
      else throw std::runtime_error("unknown argument " + k);
    }
    if (a.configs.empty() || a.cells < 1 || a.ttis < 1 || a.trace_rows < 1 || a.gpus < 1 || a.gpus > a.cells) {
      fprintf(stderr, "usage: rs_batch --algo ID --config cfg.json [--config cfg2.json ...] --cells B --ttis T [--seed s] [--gpus N] "
                      "[--traces DIR --mapping FILE [--trace-rows N]] [--log-cell b --log-prefix P]\n");
      return 2;
    }
    /* ---- the slice configs, expanded like the scheduler constructors do -------------------------------- */
    for (const std::string& path : a.configs) {
      std::ifstream ifs(path);
      if (!ifs.is_open()) throw std::runtime_error("Fail to open configuration file.");   /* transport.cpp:58-60 */
      std::stringstream ss;
      ss << ifs.rdbuf();
      const std::string text = ss.str();
      const Json cfgj = Parser(text).value();
      Profile pr;
      for (const Json& grp : cfgj["slices"].arr)
        for (int j = 0; j < grp["n_slices"].as_int(); ++j) {
          pr.weight.push_back(grp["weight"].num);
          pr.params.push_back(grp["algo_alpha"].as_int());
          pr.params.push_back(grp["algo_beta"].as_int());
          pr.params.push_back(grp["algo_epsilon"].as_int());
          pr.params.push_back(grp["algo_psi"].as_int());
        }
      const std::vector<Json>& ups = cfgj["ues_per_slice"].arr;
      for (size_t s = 0; s < ups.size(); ++s)
        for (int j = 0; j < ups[s].as_int(); ++j) pr.u2s.push_back((int32_t)s);
      const int ps = (int)ups.size(), pu = (int)pr.u2s.size();
      if ((int)pr.weight.size() != ps || pu < 1) throw std::runtime_error(path + ": slices and ues_per_slice do not match");
      if (!su.prof.empty() && (ps != su.S || pu != su.U))
        throw std::runtime_error(path + ": " + std::to_string(ps) + " slices and " + std::to_string(pu) + " UEs, the first config " +
                                 std::to_string(su.S) + " and " + std::to_string(su.U) + " (every config must have the same)");
      su.S = ps;
      su.U = pu;
      su.prof.push_back(std::move(pr));
    }
    const int S = su.S, B = a.cells, T = a.ttis, P = (int)su.prof.size();

    /* ---- CQI source ------------------------------------------------------------------------------------ */
    su.replay = !a.traces.empty();
    if (su.replay) {
      if (a.mapping.empty()) throw std::runtime_error("--traces needs --mapping");
      int32_t n_map = 0;
      check(rs_parse_mapping_file(a.mapping.c_str(), nullptr, 0, &n_map), "mapping");
      if (n_map < 1) throw std::runtime_error("empty mapping file");
      su.map.resize(n_map);
      check(rs_parse_mapping_file(a.mapping.c_str(), su.map.data(), n_map, &n_map), "mapping");
      const int kMaxTraceId = 65535;   /* ue<id>.log: the shipped set has 158 files */
      for (int t : su.map) {
        if (t < 0 || t > kMaxTraceId) throw std::runtime_error("mapping: trace id " + std::to_string(t) + " outside 0.." + std::to_string(kMaxTraceId));
        su.n_traces = std::max(su.n_traces, t + 1);
      }
      su.traces.assign((size_t)su.n_traces * a.trace_rows * R, 10);
      std::vector<char> have(su.n_traces, 0);
      for (int t : su.map) {
        if (have[t]) continue;
        have[t] = 1;
        const std::string path = a.traces + "/ue" + std::to_string(t) + ".log";
        check(rs_parse_trace_file(path.c_str(), a.trace_rows, R, su.traces.data() + (size_t)t * a.trace_rows * R), path.c_str());
      }
    }

    /* ---- the TTI clock of the reference (simulator.cc:116-126): t += 0.001 in double from the first TTI >= 0.1 s */
    su.now.resize(T);
    su.dt.resize(T);
    {
      double t = 0.0;
      while (t < 0.1) t = t + 0.001;
      double last = 0.1;
      for (int k = 0; k < T; ++k) { su.now[k] = t; su.dt[k] = t - last; last = t; t = t + 0.001; }
    }

    /* ---- shards: contiguous blocks of cells, one host thread per GPU ----------------------------------- */
    const int N = a.gpus;
    std::vector<ShardResult> res(N);
    std::vector<void*> comms(N, nullptr);
    if (N > 1) {
      int n_dev = 0;
      cu(cudaGetDeviceCount(&n_dev), "cudaGetDeviceCount");
      if (n_dev < N) throw std::runtime_error("--gpus " + std::to_string(N) + ": only " + std::to_string(n_dev) + " CUDA devices");
      std::vector<int32_t> devs(N);
      for (int i = 0; i < N; ++i) devs[i] = i;
      if (rs_comm_init_all(N, devs.data(), comms.data()) != RS_OK)
        throw std::runtime_error(std::string("rs_comm_init_all: ") + rs_nccl_last_error());
    }
    auto shard_of = [&](int r, int* c0) { const int base = B / N, rem = B % N; *c0 = r * base + std::min(r, rem); return base + (r < rem ? 1 : 0); };
    if (P > 1 && B / N < P)
      throw std::runtime_error(std::to_string(P) + " configs need at least as many cells per GPU (" + std::to_string(B / N) + ")");
    std::vector<std::thread> th;
    for (int r = 0; r < N; ++r)
      th.emplace_back([&, r]() {
        try {
          int c0 = 0;
          const int nb = shard_of(r, &c0);
          run_shard(su, r, r, c0, nb, comms[r], &res[r]);
        } catch (const std::exception& e) { res[r].error = e.what(); }
      });
    for (auto& t : th) t.join();
    for (void* c : comms) rs_comm_destroy(c);
    double ms_max = 0;
    for (int r = 0; r < N; ++r) {
      if (!res[r].error.empty()) throw std::runtime_error("gpu " + std::to_string(r) + ": " + res[r].error);
      ms_max = std::max(ms_max, res[r].ms);
    }
    /* rank 0 holds the totals over every GPU's cells; one line per config over the cells that use it (with one config:
     * the whole batch, as before configs could repeat) */
    for (int p = 0; p < P; ++p) {
      const uint64_t* stats = res[0].stats.data() + (size_t)p * 4 * S;
      const int Bp = B / P + (p < B % P ? 1 : 0);   /* cells b with b % P == p */
      printf("{\"algo\": %d, \"cells\": %d, \"ttis\": %d, \"slices\": %d, \"ues\": %d, \"gpus\": %d, \"cqi\": \"%s\", ",
             a.algo, Bp, T, S, su.U, N, su.replay ? "trace replay" : "synthetic");
      if (P > 1) printf("\"config\": %d, \"config_file\": \"%s\", \"batch_cells\": %d, ", p, a.configs[(size_t)p].c_str(), B);
      printf("\"tbs_row_m1\": \"stock -O0 build (McsToItbs alias, SURVEY H2)\", \"cell_ttis_per_s\": %.1f, \"slice_bytes\": [",
             (double)B * T / (ms_max * 1e-3));
      for (int s = 0; s < S; ++s) printf("%s%llu", s ? ", " : "", (unsigned long long)stats[s]);
      printf("], \"slice_rbs\": [");
      for (int s = 0; s < S; ++s) printf("%s%llu", s ? ", " : "", (unsigned long long)stats[S + s]);
      printf("], \"slice_mbps_per_cell\": [");
      for (int s = 0; s < S; ++s) printf("%s%.3f", s ? ", " : "", (double)stats[s] * 8 / 1e6 / (T * 1e-3) / Bp);
      printf("]}\n");
    }
    for (int r = 0; r < N; ++r) {
      if (res[r].log_out.empty() && res[r].log_err.empty()) continue;
      FILE* fo = fopen((a.log_prefix + ".stdout").c_str(), "w");
      FILE* fe = fopen((a.log_prefix + ".stderr").c_str(), "w");
      if (!fo || !fe) throw std::runtime_error("cannot write the log files");
      fputs(res[r].log_out.c_str(), fo);
      fputs(res[r].log_err.c_str(), fe);
      fclose(fo);
      fclose(fe);
    }
    return 0;
  } catch (const std::exception& e) {
    fprintf(stderr, "rs_batch: %s\n", e.what());
    return 1;
  }
}
