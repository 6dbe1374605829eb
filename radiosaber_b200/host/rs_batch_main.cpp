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
 *            [--buffers K --traffic FILE ...]   closed loop: a byte FIFO of K records per bearer on the device
 *                                               (rs_enable_buffers); arrivals drawn on the device by the traffic file's
 *                                               sources (rs_set_sources, rs_synth_traffic), the file named by --traffic
 *                                               once for every config or once per --config
 *                                               (file p with config p); every line gains the per-slice queued_bytes,
 *                                               dropped_bytes and records left at the end
 *            [--hol-bins N]                     with --buffers: head-of-line delay histograms of N 1-TTI bins counted on
 *                                               the device (rs_enable_hol_hist, one rs_reduce_hol_hist with --gpus N);
 *                                               every line gains per slice the samples of the bearers that sent
 *                                               (hol_served) and of those with bytes queued (hol_waiting), and their
 *                                               50th, 95th and 99th percentiles as bin indices (null without samples)
 *            [--rate-window W --rate-bins N     per-UE throughput histograms counted on the device (rs_enable_ue_rate_hist;
 *             --rate-bin-bytes X]               one rs_reduce_ue_rate_hist with --gpus N): every W TTIs (W divides T)
 *                                               each UE adds the bytes it received in those W TTIs, in N bins of X bytes
 *                                               (the last holds the rest); every line gains per slice the samples
 *                                               (ue_rate_samples) and their 5th, 50th and 95th percentiles as bin
 *                                               indices (ue_rate_p5 / p50 / p95, null without samples).  The three go
 *                                               together
 *            [--upt-bin-bytes X]                with --buffers and the three --rate-* flags: per-UE throughput over
 *                                               active time histograms (rs_enable_ue_upt_hist; one rs_reduce_ue_upt_hist
 *                                               with --gpus N): at each window's end every UE that had data queued in
 *                                               k of its TTIs adds its bytes / k in --rate-bins bins of X bytes per TTI;
 *                                               every line gains per slice the samples (upt_samples) and their 5th,
 *                                               50th and 95th percentiles as bin indices (upt_p5 / p50 / p95, null
 *                                               without samples)
 *            [--channel FILE ...]               synthetic channel CQI drawn on the device (rs_set_channels,
 *                                               rs_synth_channel) in place of rs_synth_cqi's i.i.d. draws, the file named
 *                                               once for every config or once per --config; not with --traces
 *
 * A traffic file, read with the slice config it goes with:
 *     {"bearers": 2, "slices": [{"backlogged": 1}, {"pkt_bytes": 1500, "pkts_per_tti": 0.6}, ...]}
 * "bearers" (1 or 2) becomes rs_config.n_bearers; "slices" has one entry per entry of the config's "slices", in the same
 * order, and applies to each of its n_slices slices.  Every bearer of those slices
 *   {"backlogged": 1}                                   is backlogged (no FIFO);
 *   {"pkt_bytes": n, "pkts_per_tti": x}                 receives packets of n bytes at a mean of x per TTI (RS_SRC_RATE;
 *                                                       rs_arrival_spec converts the rate to 16.16 fixed point);
 *   {"period_ttis": n, "frame_bytes": [f0, f1, ...]}    receives one frame every n TTIs, sizes cycling through the list
 *                                                       (RS_SRC_PERIODIC);
 *   {"pkt_bytes": n, "period_ttis": p,                  runs an on-off chain with mean ON / OFF runs of x / y TTIs
 *    "on_ttis": x, "off_ttis": y}                       (rs_onoff_spec) and receives n bytes every p TTIs while ON
 *                                                       (RS_SRC_ONOFF).
 * These are generic traffic models, not LTE-Sim's VoIP, TraceBased or InternetFlow applications.  The config's own
 * traffic fields (internet_flow, if_bitrate, video_*) are not read: LTE-Sim's application models and
 * RLC header bytes behind them are not modelled here (DESIGN.md), and turning them into packet sizes and rates would
 * pass an approximation off as the reference's traffic.
 *
 * A channel file, read with the slice config it goes with:
 *     {"report_ttis": 40, "slices": [{"iid": 1}, {"level_counts": [15 counts], "depth_cqi": 1.5, "coherence_rbgs": 8,
 *                                                 "coherence_reports": 4}, ...]}
 * CQI reports fall on the global TTIs that are multiples of "report_ttis" (default 1; 40 is the reference's
 * CQI_INTERVAL), as in the trace replay path, and report e is epoch e of the channel.  "slices" has one entry per entry
 * of the config's "slices", applying to each of its n_slices slices:
 *   {"iid": 1}                                          rs_synth_cqi's i.i.d. draws (RS_CH_IID);
 *   {"level_counts": [...], "depth_cqi": d,             a per-UE level drawn from the 15 counts and an offset of standard
 *    "coherence_rbgs": f, "coherence_reports": t}       deviation d CQI steps, coherent over f RBGs and t reports
 *                                                       (RS_CH_FADING, rs_channel_spec).
 * Other keys (a "note") are not read.  A file of {"iid": 1} entries with report_ttis 1 gives the output of a run
 * without --channel, byte for byte.
 *
 * Host logic only; every scheduling decision is made by the CUDA kernels behind the ABI (no CPU fallback).
 */
#include <algorithm>
#include <cctype>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <initializer_list>
#include <map>
#include <sstream>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "rs_sched.h"
#include "rs_sched_nccl.h"
#include "rs_sched_nccl_ue_upt.h"

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
    } else if (s.compare(i, 4, "null") == 0) {   /* read like an absent key, as Python's dict.get reads None */
      i += 4;
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
  int buffers = -1;                  /* --buffers K; -1 = backlogged bearers only, as without the flag */
  int hol_bins = 0;                  /* --hol-bins N; 0 = no delay histograms */
  int rate_window = 0, rate_bins = 0;   /* --rate-window W --rate-bins N; 0 = no throughput histograms */
  long long rate_bin_bytes = 0;         /* --rate-bin-bytes X */
  int rate_given = 0;                   /* bits 1, 2, 4: which of the three flags were given */
  long long upt_bin_bytes = 0;          /* --upt-bin-bytes X; 0 = no UPT histograms */
  bool upt_given = false;
  uint64_t seed = 1;
  std::vector<std::string> configs, traffic, channel;
  std::string traces, mapping, log_prefix;
};

struct Profile {   /* one slice config, expanded like the scheduler constructors do */
  std::vector<double> weight;
  std::vector<int32_t> params, u2s;
  std::vector<int> groups;         /* n_slices of each entry of the config's "slices" */
  /* from the traffic file (--buffers): src and backlogged [S]; frames [groups], a PERIODIC entry's frame sizes */
  std::vector<rs_source> src;
  std::vector<uint8_t> backlogged;
  std::vector<std::vector<int32_t>> frames;
  std::vector<rs_channel> chn;     /* [S], from the channel file (--channel) */
};

struct Setup {   /* what every shard shares */
  Args a;
  int S = 0, U = 0;
  int nb = 1;                    /* bearers per UE (the traffic file's "bearers") */
  int report = 1;                /* TTIs per CQI report: the channel file's "report_ttis" (1 without --channel) */
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
  std::vector<uint64_t> buf_stats;   /* [P][3][S] (--buffers), the same way */
  std::vector<uint64_t> hol_hist;    /* [P][2][S][hol_bins] (--hol-bins), the same way */
  std::vector<uint64_t> rate_hist;   /* [P][S][rate_bins] (--rate-window), the same way */
  std::vector<uint64_t> upt_hist;    /* [P][S][rate_bins] (--upt-bin-bytes), the same way */
  std::string log_out, log_err, error;
};

std::string read_file(const std::string& path, const char* what) {
  std::ifstream ifs(path);
  if (!ifs.is_open()) throw std::runtime_error(std::string("Fail to open ") + what + " file " + path + ".");
  std::stringstream ss;
  ss << ifs.rdbuf();
  return ss.str();
}

/* x as an integer lo..INT32_MAX, else the reason (the words of sched.py's load_traffic) */
int32_t int_in(double x, double lo, const char* name) {
  if (!(x >= lo && x <= 2147483647.0) || x != std::floor(x)) {
    char buf[128];
    snprintf(buf, sizeof buf, "%s %g is not an integer %g..2147483647", name, x, lo);
    throw std::invalid_argument(buf);
  }
  return (int32_t)x;
}

/* One entry of "slices" -> its source (kind RS_SRC_NONE = backlogged); frames receives a PERIODIC entry's sizes. */
rs_source parse_source(const Json& e, std::vector<int32_t>* frames) {
  rs_source src;
  memset(&src, 0, sizeof src);
  const size_t nk = e.kind == Json::Obj ? e.obj.size() : 0;
  auto num = [&](const char* k) { return e[k].kind == Json::Num; };
  if (nk == 1 && num("backlogged")) {
    if (e["backlogged"].num != 1) throw std::invalid_argument("\"backlogged\" must be 1");
    src.kind = RS_SRC_NONE;
  } else if (nk == 2 && num("pkt_bytes") && num("pkts_per_tti")) {
    src.kind = RS_SRC_RATE;
    if (rs_arrival_spec(e["pkt_bytes"].num, e["pkts_per_tti"].num, &src.pkt_bytes, &src.pkts_q16) != RS_OK)
      throw std::invalid_argument(rs_last_error());
  } else if (nk == 2 && num("period_ttis") && e["frame_bytes"].kind == Json::Arr &&
             std::all_of(e["frame_bytes"].arr.begin(), e["frame_bytes"].arr.end(), [](const Json& v) { return v.kind == Json::Num; })) {
    src.kind = RS_SRC_PERIODIC;
    src.period_ttis = int_in(e["period_ttis"].num, 1, "period_ttis");
    const std::vector<Json>& f = e["frame_bytes"].arr;
    if (f.empty() || f.size() > RS_MAX_FRAMES)
      throw std::invalid_argument(std::to_string(f.size()) + " frame_bytes, expected 1.." + std::to_string(RS_MAX_FRAMES));
    for (const Json& v : f) frames->push_back(int_in(v.num, 1, "frame_bytes"));
    src.n_frames = (int32_t)f.size();
  } else if (nk == 4 && num("pkt_bytes") && num("period_ttis") && num("on_ttis") && num("off_ttis")) {
    src.kind = RS_SRC_ONOFF;
    src.pkt_bytes = int_in(e["pkt_bytes"].num, 1, "pkt_bytes");
    src.period_ttis = int_in(e["period_ttis"].num, 1, "period_ttis");
    if (rs_onoff_spec(e["on_ttis"].num, e["off_ttis"].num, &src.leave_on_q32, &src.leave_off_q32) != RS_OK)
      throw std::invalid_argument(rs_last_error());
  } else {
    throw std::invalid_argument("expected {\"backlogged\": 1}, {\"pkt_bytes\": n, \"pkts_per_tti\": x}, {\"period_ttis\": n, "
                                "\"frame_bytes\": [n, ...]} or {\"pkt_bytes\": n, \"period_ttis\": n, \"on_ttis\": x, \"off_ttis\": x}");
  }
  return src;
}

/* The traffic file `path` (format: header comment) for the slice config of `pr`; returns its "bearers". */
int load_traffic(const std::string& path, Profile* pr) {
  const std::string text = read_file(path, "traffic");
  const Json t = Parser(text).value();
  const std::string where = "traffic file " + path + ": ";
  const Json& bearers = t["bearers"];
  if (bearers.kind != Json::Num || (bearers.num != 1 && bearers.num != 2)) throw std::runtime_error(where + "\"bearers\" must be 1 or 2");
  const Json& groups = t["slices"];
  if (groups.kind != Json::Arr) throw std::runtime_error(where + "\"slices\" must be a list");
  if (groups.arr.size() != pr->groups.size())
    throw std::runtime_error(where + std::to_string(groups.arr.size()) + " entries in \"slices\", the slice config has " +
                             std::to_string(pr->groups.size()) + " slice groups");
  pr->frames.resize(groups.arr.size());
  for (size_t g = 0; g < groups.arr.size(); ++g) {
    rs_source src;
    try {
      src = parse_source(groups.arr[g], &pr->frames[g]);
    } catch (const std::invalid_argument& e) {
      throw std::runtime_error(where + "slices[" + std::to_string(g) + "]: " + e.what());
    }
    for (int j = 0; j < pr->groups[g]; ++j) {
      pr->src.push_back(src);
      pr->backlogged.push_back(src.kind == RS_SRC_NONE ? 1 : 0);
    }
  }
  return bearers.as_int();
}

/* One entry of a channel file's "slices" -> its channel. */
rs_channel parse_channel(const Json& e) {
  rs_channel ch;
  memset(&ch, 0, sizeof ch);
  const size_t nk = e.kind == Json::Obj ? e.obj.size() : 0;
  auto num = [&](const char* k) { return e[k].kind == Json::Num; };
  const Json& lc = e["level_counts"];
  if (nk == 1 && num("iid")) {
    if (e["iid"].num != 1) throw std::invalid_argument("\"iid\" must be 1");
    ch.kind = RS_CH_IID;
  } else if (nk == 4 && lc.kind == Json::Arr && lc.arr.size() == 15 &&
             std::all_of(lc.arr.begin(), lc.arr.end(), [](const Json& v) { return v.kind == Json::Num; }) &&
             num("depth_cqi") && num("coherence_rbgs") && num("coherence_reports")) {
    double counts[15];
    for (int k = 0; k < 15; ++k) counts[k] = lc.arr[(size_t)k].num;
    if (rs_channel_spec(counts, e["depth_cqi"].num, e["coherence_rbgs"].num, e["coherence_reports"].num, &ch) != RS_OK)
      throw std::invalid_argument(rs_last_error());
  } else {
    throw std::invalid_argument("expected {\"iid\": 1} or {\"level_counts\": [15 counts], \"depth_cqi\": x, "
                                "\"coherence_rbgs\": x, \"coherence_reports\": x}");
  }
  return ch;
}

/* The channel file `path` (format: header comment) for the slice config of `pr`; returns its "report_ttis". */
int load_channel(const std::string& path, Profile* pr) {
  const std::string text = read_file(path, "channel");
  const Json t = Parser(text).value();
  const std::string where = "channel file " + path + ": ";
  const Json& groups = t["slices"];
  if (groups.kind != Json::Arr) throw std::runtime_error(where + "\"slices\" must be a list");
  const Json& rep = t["report_ttis"];
  int report = 1;
  if (rep.kind != Json::Null) {
    if (rep.kind != Json::Num || !(rep.num >= 1 && rep.num <= 2147483647.0) || rep.num != std::floor(rep.num))
      throw std::runtime_error(where + "\"report_ttis\" must be an integer 1..2147483647");
    report = (int)rep.num;
  }
  if (groups.arr.size() != pr->groups.size())
    throw std::runtime_error(where + std::to_string(groups.arr.size()) + " entries in \"slices\", the slice config has " +
                             std::to_string(pr->groups.size()) + " slice groups");
  for (size_t g = 0; g < groups.arr.size(); ++g) {
    rs_channel ch;
    try {
      ch = parse_channel(groups.arr[g]);
    } catch (const std::invalid_argument& e) {
      throw std::runtime_error(where + "slices[" + std::to_string(g) + "]: " + e.what());
    }
    pr->chn.insert(pr->chn.end(), (size_t)pr->groups[g], ch);
  }
  return report;
}

/* The S histograms of nbins bins at hist, as lists of an output line (each opened by "], " like the line's others):
 * "<samples>" the samples per slice, and "<prefix>_p<q>" for each q the q-th percentile per slice as a bin index, by
 * sched.hist_percentile's rule (the smallest bin d with 100 x samples in 0..d >= q x samples; null without samples). */
void print_hist(const char* samples, const char* prefix, const uint64_t* hist, int S, size_t nbins,
                std::initializer_list<int> qs) {
  printf("], \"%s\": [", samples);
  for (int s = 0; s < S; ++s) {
    uint64_t n = 0;
    for (size_t d = 0; d < nbins; ++d) n += hist[(size_t)s * nbins + d];
    printf("%s%llu", s ? ", " : "", (unsigned long long)n);
  }
  for (int q : qs) {
    printf("], \"%s_p%d\": [", prefix, q);
    for (int s = 0; s < S; ++s) {
      const uint64_t* hs = hist + (size_t)s * nbins;
      uint64_t n = 0, cum = 0;
      for (size_t d = 0; d < nbins; ++d) n += hs[d];
      size_t d = 0;
      for (; n > 0 && d < nbins; ++d) {   /* the smallest bin with 100 x cum >= q x n */
        cum += hs[d];
        if (100 * cum >= (uint64_t)q * n) break;
      }
      if (n == 0) printf("%snull", s ? ", " : "");
      else printf("%s%zu", s ? ", " : "", d);
    }
  }
}

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
    if (a.buffers > 0) cfg.n_bearers = su.nb;
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
  const bool buffered = a.buffers > 0;
  const int slots = su.nb;   /* bearers per UE */
  if (buffered) {
    std::vector<uint8_t> backlogged((size_t)B * U * slots);   /* cell cell0 + b: its config's slices */
    for (int b = 0; b < B; ++b) {
      const Profile& pr = su.prof[(size_t)((cell0 + b) % P)];
      for (int u = 0; u < U; ++u)
        for (int i = 0; i < slots; ++i) backlogged[((size_t)b * U + u) * slots + i] = pr.backlogged[(size_t)pr.u2s[(size_t)u]];
    }
    check(rs_enable_buffers(h, a.buffers, backlogged.data()), "rs_enable_buffers");
    std::vector<rs_source> src;   /* [P][S]: profile p of the handle is config p */
    for (const Profile& pr : su.prof)
      for (size_t g = 0, s = 0; g < pr.groups.size(); ++g)
        for (int j = 0; j < pr.groups[g]; ++j, ++s) {
          src.push_back(pr.src[s]);
          if (src.back().kind == RS_SRC_PERIODIC) src.back().frame_bytes = pr.frames[g].data();
        }
    check(rs_set_sources(h, src.data()), "rs_set_sources");
    if (a.hol_bins > 0) check(rs_enable_hol_hist(h, a.hol_bins, 1000.0), "rs_enable_hol_hist");   /* the clock is in s */
  }
  const bool channel = !a.channel.empty();
  if (channel) {
    std::vector<rs_channel> chn;   /* [P][S]: profile p of the handle is config p */
    for (const Profile& pr : su.prof) chn.insert(chn.end(), pr.chn.begin(), pr.chn.end());
    check(rs_set_channels(h, chn.data()), "rs_set_channels");
  }
  const int rep = su.report;
  const int W = a.rate_window;   /* 0 = no throughput histograms */
  if (W > 0) check(rs_enable_ue_rate_hist(h, a.rate_bins, a.rate_bin_bytes), "rs_enable_ue_rate_hist");
  if (a.upt_given) check(rs_enable_ue_upt_hist(h, a.rate_bins, a.upt_bin_bytes), "rs_enable_ue_upt_hist");

  /* ---- run in blocks of TB TTIs with everything resident on the device ------------------------------- */
  const int TB = 16;
  uint8_t* d_cqi = nullptr;
  int32_t* d_draws = nullptr;
  int16_t *d_rbg = nullptr, *d_gue = nullptr, *d_grbg = nullptr;   /* d_g*: id 10's grant list */
  int32_t* d_gn = nullptr;
  size_t n_list = 0;   /* entries per cell of the grant list */
  int32_t *d_bits = nullptr, *d_tgt = nullptr, *d_quo = nullptr;
  uint8_t* d_fc = nullptr;
  int32_t *d_arr = nullptr, *d_qo = nullptr;   /* [TB][B][U][nb]: arrivals; the queues the TTIs showed (logged cell) */
  double* d_ho = nullptr;                      /* [TB][B][U][nb]: the head-of-line delays they showed */
  const size_t row = G / 2, per_tti = (size_t)B * U * slots;
  if (!replay) cu(cudaMalloc(&d_cqi, (size_t)TB * B * U * row), "cudaMalloc");
  if (buffered) cu(cudaMalloc(&d_arr, sizeof(int32_t) * TB * per_tti), "cudaMalloc");
  if (n_draws > 0) cu(cudaMalloc(&d_draws, sizeof(int32_t) * (size_t)TB * B * n_draws), "cudaMalloc");
  const int lc = a.log_cell - cell0;   /* the logged cell, if it lives in this shard */
  const bool want_log = lc >= 0 && lc < B && !a.log_prefix.empty();
  rs_log* lg = nullptr;
  std::vector<int16_t> h_rbg, h_gue, h_grbg;
  std::vector<int32_t> h_bits, h_tgt, h_quo, h_q;
  std::vector<uint8_t> h_fc, h_cqi;
  std::vector<double> h_hol;
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
    if (buffered) {
      cu(cudaMalloc(&d_qo, sizeof(int32_t) * TB * per_tti), "cudaMalloc");
      cu(cudaMalloc(&d_ho, sizeof(double) * TB * per_tti), "cudaMalloc");
      h_q.resize((size_t)U * slots); h_hol.resize((size_t)U * slots);
    }
  }
  std::vector<int32_t> trow(TB);
  for (int t0 = 0, n = 0; t0 < T; t0 += n) {
    n = std::min(TB, T - t0);
    /* rs_run_device reads slab t / rep from the start of the call: a chunk that starts between two reports ends at the
     * next one, so every chunk starts on a report or lies within one */
    if (t0 % rep) n = std::min(n, rep - t0 % rep);
    if (W > 0) n = std::min(n, W - t0 % W);   /* and a chunk that would cross a window's end ends there */
    if (channel) {
      /* the reports of TTIs t0 .. t0 + n - 1, one slab each */
      check(rs_synth_channel(h, a.seed, cell0, t0 / rep, (t0 + n - 1) / rep - t0 / rep + 1, d_cqi), "rs_synth_channel");
    } else if (!replay) {
      check(rs_synth_cqi(h, a.seed, cell0, t0, n, d_cqi), "rs_synth_cqi");
    }
    if (n_draws > 0) check(rs_synth_rand2(h, a.seed, cell0, t0, n, d_draws), "rs_synth_rand2");
    if (buffered) {
      /* counter-based draws over global cells: N GPUs draw exactly the arrivals one GPU would */
      check(rs_synth_traffic(h, a.seed, cell0, t0, n, d_arr), "rs_synth_traffic");
      const rs_traffic tr = {d_arr, su.now.data() + t0, su.now.data() + t0, d_qo, d_ho};
      check(rs_set_traffic(h, &tr), "rs_set_traffic");
    }
    check(rs_sync(h), "rs_sync");
    const auto w0 = std::chrono::steady_clock::now();
    if (replay) {
      /* all UEs report in the same TTI, every 40 TTIs from the first (phy/ue-lte-phy.cpp:215-232) */
      for (int k = 0; k < n; ++k) trow[k] = rs_trace_row(su.now[(t0 + k) - (t0 + k) % 40], n_rows);
      check(rs_run_traces_device(h, n, trow.data(), d_draws, nullptr, 0, su.dt.data() + t0, want_log ? &out : nullptr, TB), "rs_run_traces_device");
    } else {
      check(rs_run_device(h, n, d_cqi, (int64_t)B * U * row, rep, d_draws, nullptr, 0, su.dt.data() + t0, want_log ? &out : nullptr, TB), "rs_run_device");
    }
    check(rs_sync(h), "rs_sync");
    res->ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - w0).count();
    if (W > 0 && (t0 + n) % W == 0) check(rs_close_ue_rate_window(h), "rs_close_ue_rate_window");
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
          /* the slab TTI t0 + k read */
          const size_t sb = (size_t)((t0 + k) / rep - t0 / rep) * B + lc;
          cu(cudaMemcpy(h_cqi.data(), d_cqi + sb * U * row, (size_t)U * row, cudaMemcpyDeviceToHost), "copy");
        }
        cu(cudaMemcpy(h_rbg.data(), d_rbg + tb * G, sizeof(int16_t) * G, cudaMemcpyDeviceToHost), "copy");
        cu(cudaMemcpy(h_bits.data(), d_bits + tb * U, sizeof(int32_t) * U, cudaMemcpyDeviceToHost), "copy");
        cu(cudaMemcpy(h_fc.data(), d_fc + tb * U, U, cudaMemcpyDeviceToHost), "copy");
        cu(cudaMemcpy(h_tgt.data(), d_tgt + tb * S, sizeof(int32_t) * S, cudaMemcpyDeviceToHost), "copy");
        cu(cudaMemcpy(h_quo.data(), d_quo + tb * S, sizeof(int32_t) * S, cudaMemcpyDeviceToHost), "copy");
        if (buffered) {   /* what the TTI showed the scheduler: the logged dataToTransmit and hol_delay */
          cu(cudaMemcpy(h_q.data(), d_qo + tb * U * slots, sizeof(int32_t) * U * slots, cudaMemcpyDeviceToHost), "copy");
          cu(cudaMemcpy(h_hol.data(), d_ho + tb * U * slots, sizeof(double) * U * slots, cudaMemcpyDeviceToHost), "copy");
          check(rs_log_set_queues(lg, h_q.data(), h_hol.data()), "rs_log_set_queues");
        }
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
  if (buffered) {
    res->buf_stats.assign((size_t)3 * S * P, 0);
    if (comm) {
      if (rs_reduce_buffer_stats(h, comm, 0, res->buf_stats.data()) != RS_OK)
        throw std::runtime_error(std::string("rs_reduce_buffer_stats: ") + rs_nccl_last_error());
    } else {
      check(rs_get_buffer_stats(h, res->buf_stats.data()), "rs_get_buffer_stats");
    }
  }
  if (a.hol_bins > 0) {
    res->hol_hist.assign((size_t)2 * S * P * a.hol_bins, 0);
    if (comm) {
      if (rs_reduce_hol_hist(h, comm, 0, res->hol_hist.data()) != RS_OK)
        throw std::runtime_error(std::string("rs_reduce_hol_hist: ") + rs_nccl_last_error());
    } else {
      check(rs_get_hol_hist(h, res->hol_hist.data()), "rs_get_hol_hist");
    }
  }
  if (W > 0) {
    res->rate_hist.assign((size_t)S * P * a.rate_bins, 0);
    if (comm) {
      if (rs_reduce_ue_rate_hist(h, comm, 0, res->rate_hist.data()) != RS_OK)
        throw std::runtime_error(std::string("rs_reduce_ue_rate_hist: ") + rs_nccl_last_error());
    } else {
      check(rs_get_ue_rate_hist(h, res->rate_hist.data()), "rs_get_ue_rate_hist");
    }
  }
  if (a.upt_given) {
    res->upt_hist.assign((size_t)S * P * a.rate_bins, 0);
    if (comm) {
      if (rs_reduce_ue_upt_hist(h, comm, 0, res->upt_hist.data()) != RS_OK)
        throw std::runtime_error(std::string("rs_reduce_ue_upt_hist: ") + rs_nccl_last_error());
    } else {
      check(rs_get_ue_upt_hist(h, res->upt_hist.data()), "rs_get_ue_upt_hist");
    }
  }
  (void)rank;
  if (lg) {
    res->log_out = rs_log_stdout(lg, nullptr);
    res->log_err = rs_log_stderr(lg, nullptr);
    rs_log_destroy(lg);
  }
  rs_destroy(h);
  cudaFree(d_cqi); cudaFree(d_draws); cudaFree(d_rbg); cudaFree(d_bits); cudaFree(d_fc); cudaFree(d_tgt); cudaFree(d_quo); cudaFree(d_gn); cudaFree(d_gue); cudaFree(d_grbg);
  cudaFree(d_arr); cudaFree(d_qo); cudaFree(d_ho);
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
      else if (k == "--buffers") a.buffers = atoi(next().c_str());
      else if (k == "--traffic") a.traffic.push_back(next());
      else if (k == "--channel") a.channel.push_back(next());
      else if (k == "--hol-bins") a.hol_bins = atoi(next().c_str());
      else if (k == "--rate-window") { a.rate_window = atoi(next().c_str()); a.rate_given |= 1; }
      else if (k == "--rate-bins") { a.rate_bins = atoi(next().c_str()); a.rate_given |= 2; }
      else if (k == "--rate-bin-bytes") { a.rate_bin_bytes = strtoll(next().c_str(), nullptr, 10); a.rate_given |= 4; }
      else if (k == "--upt-bin-bytes") { a.upt_bin_bytes = strtoll(next().c_str(), nullptr, 10); a.upt_given = true; }
      else throw std::runtime_error("unknown argument " + k);
    }
    if (a.configs.empty() || a.cells < 1 || a.ttis < 1 || a.trace_rows < 1 || a.gpus < 1 || a.gpus > a.cells) {
      fprintf(stderr, "usage: rs_batch --algo ID --config cfg.json [--config cfg2.json ...] --cells B --ttis T [--seed s] [--gpus N] "
                      "[--traces DIR --mapping FILE [--trace-rows N]] [--log-cell b --log-prefix P] [--buffers K --traffic FILE ...] "
                      "[--channel FILE ...] [--hol-bins N] [--rate-window W --rate-bins N --rate-bin-bytes X] "
                      "[--upt-bin-bytes X]\n");
      return 2;
    }
    if (a.buffers != -1 && (a.buffers < 1 || a.buffers > RS_MAX_BUFFER_RECORDS))
      throw std::runtime_error("--buffers K: K records per bearer, 1.." + std::to_string(RS_MAX_BUFFER_RECORDS));
    if (a.buffers > 0 && a.traffic.empty()) throw std::runtime_error("--buffers needs --traffic FILE");
    if (a.buffers < 0 && !a.traffic.empty()) throw std::runtime_error("--traffic needs --buffers K");
    if (a.hol_bins != 0 && (a.hol_bins < 1 || a.hol_bins > RS_MAX_HOL_BINS))
      throw std::runtime_error("--hol-bins N: N bins of one TTI, 1.." + std::to_string(RS_MAX_HOL_BINS));
    if (a.hol_bins > 0 && a.buffers < 0) throw std::runtime_error("--hol-bins needs --buffers K");
    if (a.rate_given != 0 && a.rate_given != 7)
      throw std::runtime_error("--rate-window W, --rate-bins N and --rate-bin-bytes X go together");
    if (a.rate_given && (a.rate_window < 1 || a.ttis % a.rate_window))
      throw std::runtime_error("--rate-window W: W TTIs per window, >= 1 and dividing --ttis " + std::to_string(a.ttis));
    if (a.rate_given && (a.rate_bins < 1 || a.rate_bins > RS_MAX_UE_RATE_BINS))
      throw std::runtime_error("--rate-bins N: N bins, 1.." + std::to_string(RS_MAX_UE_RATE_BINS));
    if (a.rate_given && a.rate_bin_bytes < 1) throw std::runtime_error("--rate-bin-bytes X: X bytes per bin, >= 1");
    if (a.upt_given && (a.buffers < 0 || a.rate_given != 7))
      throw std::runtime_error("--upt-bin-bytes needs --buffers K and --rate-window W --rate-bins N --rate-bin-bytes X");
    if (a.upt_given && a.upt_bin_bytes < 1) throw std::runtime_error("--upt-bin-bytes X: X bytes per TTI per bin, >= 1");
    if (!a.traffic.empty() && a.traffic.size() != 1 && a.traffic.size() != a.configs.size())
      throw std::runtime_error(std::to_string(a.traffic.size()) + " --traffic files for " + std::to_string(a.configs.size()) +
                               " --config files: give one for all or one per config");
    if (!a.channel.empty() && !a.traces.empty()) throw std::runtime_error("--channel and --traces both give the CQI: use one");
    if (!a.channel.empty() && a.channel.size() != 1 && a.channel.size() != a.configs.size())
      throw std::runtime_error(std::to_string(a.channel.size()) + " --channel files for " + std::to_string(a.configs.size()) +
                               " --config files: give one for all or one per config");
    /* ---- the slice configs, expanded like the scheduler constructors do -------------------------------- */
    for (const std::string& path : a.configs) {
      std::ifstream ifs(path);
      if (!ifs.is_open()) throw std::runtime_error("Fail to open configuration file.");   /* transport.cpp:58-60 */
      std::stringstream ss;
      ss << ifs.rdbuf();
      const std::string text = ss.str();
      const Json cfgj = Parser(text).value();
      Profile pr;
      for (const Json& grp : cfgj["slices"].arr) {
        pr.groups.push_back(grp["n_slices"].as_int());
        for (int j = 0; j < grp["n_slices"].as_int(); ++j) {
          pr.weight.push_back(grp["weight"].num);
          pr.params.push_back(grp["algo_alpha"].as_int());
          pr.params.push_back(grp["algo_beta"].as_int());
          pr.params.push_back(grp["algo_epsilon"].as_int());
          pr.params.push_back(grp["algo_psi"].as_int());
        }
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
      if (a.buffers > 0) {
        const int nb = load_traffic(a.traffic[a.traffic.size() == 1 ? 0 : su.prof.size()], &pr);
        if (!su.prof.empty() && nb != su.nb)
          throw std::runtime_error("traffic files with \"bearers\" " + std::to_string(su.nb) + " and " + std::to_string(nb) +
                                   " (every config of a batch must have the same)");
        su.nb = nb;
      }
      if (!a.channel.empty()) {
        const int report = load_channel(a.channel[a.channel.size() == 1 ? 0 : su.prof.size()], &pr);
        if (!su.prof.empty() && report != su.report)
          throw std::runtime_error("channel files with \"report_ttis\" " + std::to_string(su.report) + " and " +
                                   std::to_string(report) + " (every config of a batch must have the same)");
        su.report = report;
      }
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
      if (a.buffers > 0) {   /* what the config's cells left in their buffers at the end */
        const uint64_t* bs = res[0].buf_stats.data() + (size_t)p * 3 * S;
        const char* names[3] = {"queued_bytes", "dropped_bytes", "records"};
        for (int k = 0; k < 3; ++k) {
          printf("], \"%s\": [", names[k]);
          for (int s = 0; s < S; ++s) printf("%s%llu", s ? ", " : "", (unsigned long long)bs[(size_t)k * S + s]);
        }
      }
      if (a.hol_bins > 0) {   /* per slice: samples, and percentiles as bin indices */
        const size_t nbins = (size_t)a.hol_bins;
        const char* rows[2] = {"hol_served", "hol_waiting"};
        for (int r = 0; r < 2; ++r)
          print_hist(rows[r], rows[r], res[0].hol_hist.data() + ((size_t)p * 2 + r) * S * nbins, S, nbins, {50, 95, 99});
      }
      if (a.rate_window > 0)
        print_hist("ue_rate_samples", "ue_rate", res[0].rate_hist.data() + (size_t)p * S * a.rate_bins, S,
                   (size_t)a.rate_bins, {5, 50, 95});
      if (a.upt_given)
        print_hist("upt_samples", "upt", res[0].upt_hist.data() + (size_t)p * S * a.rate_bins, S, (size_t)a.rate_bins,
                   {5, 50, 95});
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
