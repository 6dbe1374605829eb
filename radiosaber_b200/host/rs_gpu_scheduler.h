/* rs_gpu_scheduler.h -- the host-side plug-in: a PacketScheduler subclass that drops into LTE-Sim.
 *
 * Compiled INSIDE the reference tree (it includes the reference's own headers), constructed with
 * the arguments the reference's schedulers take, installed by ENodeB::SetDLScheduler
 * (src/device/ENodeB.cpp:302-391; the three-line change is in INTEGRATION.md):
 *
 *     case ENodeB::DLScheduler_TYPE_PROPORTIONAL_FAIR:   // id 1
 *       scheduler = new RsGpuScheduler(config_fname, 1);   // was DL_PF_PacketScheduler(config_fname)
 *     case ENodeB::DLScheduler_MAXCELL:      // id 9
 *       scheduler = new RsGpuScheduler(config_fname, 9);   // was DownlinkTransportScheduler(config_fname, 2)
 *   (likewise 7 NVS, 8 Sequential, 10 UpperBound, 11 NVS non-greedy, 101 SubOpt, 103 VogelApproximate)
 *
 * What stays on the host, done by the reference's own objects exactly as before:
 *   - RadioBearer::UpdateAverageTransmissionRate / UpdateTransmittedBytes / UpdateCumulateRBs
 *     (flows/radio-bearer.cpp:100-164) -- bearers are LTE-Sim objects other code reads;
 *   - the UserToSchedule list, PDCCH map message, RLC TransmissionProcedure, packet burst
 *     (downlink-transport-scheduler.cpp:170-221, 661-674).
 * What the GPU does through the C ABI (one cell, B = 1): slice targets/quotas, the UE x RBG metric,
 * the per-slice enterprise argmax, the inter-slice assignment (RadioSaber / Sequential / NVS), and
 * EESM -> CQI -> MCS -> TBS per served UE, i.e. RBsAllocation() (downlink-transport-scheduler.cpp:
 * 453-675, downlink-nvs-scheduler.cpp:94-142 + 275-358).
 *
 * Errors: like the reference (std::runtime_error on a bad config); a non-zero status from the C ABI
 * becomes std::runtime_error.  No CPU fallback: without a GPU the constructor throws.
 */
#ifndef RS_GPU_SCHEDULER_H_
#define RS_GPU_SCHEDULER_H_

#include <jsoncpp/json/json.h>

#include <cstdint>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <list>
#include <stdexcept>
#include <algorithm>
#include <chrono>
#include <string>
#include <vector>

#include "rs_sched.h" /* include/rs_sched.h */

/* reference headers, relative to the reference's src/ directory (compile with -I<LTE-Sim>/src) */
#include "core/spectrum/bandwidth-manager.h"
#include "device/ENodeB.h"
#include "device/NetworkNode.h"
#include "flows/application/Application.h"
#include "flows/radio-bearer.h"
#include "phy/lte-phy.h"
#include "protocolStack/mac/AMCModule.h"
#include "protocolStack/mac/mac-entity.h"
#include "protocolStack/mac/packet-scheduler/packet-scheduler.h"
#include "protocolStack/packet/Packet.h"
#include "protocolStack/packet/packet-burst.h"
#include "protocolStack/protocol-stack.h"
#include "protocolStack/rlc/rlc-entity.h"
#include "protocolStack/rrc/rrc-entity.h"
#include "utility/eesm-effective-sinr.h"

class RsGpuScheduler : public PacketScheduler {
 public:
  /* public like the fields the test harness reads from the reference classes */
  int num_slices_ = 1;
  std::vector<int> user_to_slice_;
  std::vector<double> slice_weights_;
  std::vector<SchedulerAlgoParam> slice_algo_params_;
  std::vector<double> slice_state_; /* slice_rbs_offset_ (ids 8/9) or slice_ewma_time_ (id 7) */
  double step_seconds_ = 0;         /* wall time spent inside rs_step_cell (copy up, launch, copy down, sync) */
  long step_calls_ = 0;

  /* scheduler_id: 1 No-Slicing PF, 7 NVS, 8 Sequential, 9 RadioSaber, 10 UpperBound (single-cell-with-interference.h:95-110),
   * and 101 SubOpt / 103 VogelApproximate, the two inter-slice algorithms ENodeB.cpp:363-379 can install.
   * Id 1 replaces DL_PF_PacketScheduler(config_fname) (ENodeB.cpp:309-313); that class schedules flows
   * (FlowToSchedule, one per bearer), which with one bearer per UE is the same list as the users kept here.
   * Bearers may be backlogged or have finite queues (internet flows, video); two bearers on one UE are folded into one
   * user like InsertFlowToUser does (ids 1 and 11 throw). */
  RsGpuScheduler(std::string config_fname, int scheduler_id) : id_(scheduler_id) {
    if (id_ != 1 && !Nvs() && !Transport())
      throw std::runtime_error("RsGpuScheduler: scheduler id must be 1, 7, 8, 9, 10, 11, 101 or 103");
    std::ifstream ifs(config_fname);
    if (!ifs.is_open()) throw std::runtime_error("Fail to open configuration file.");
    Json::Reader reader;
    Json::Value obj;
    reader.parse(ifs, obj);
    ifs.close();
    const Json::Value& ues_per_slice = obj["ues_per_slice"];
    num_slices_ = ues_per_slice.size();
    for (int i = 0; i < num_slices_; i++)
      for (int j = 0, n = ues_per_slice[i].asInt(); j < n; j++) user_to_slice_.push_back(i);
    const Json::Value& schemes = obj["slices"];
    for (int i = 0; i < (int)schemes.size(); i++)
      for (int j = 0, n = schemes[i]["n_slices"].asInt(); j < n; j++) {
        slice_weights_.push_back(schemes[i]["weight"].asDouble());
        slice_algo_params_.emplace_back(schemes[i]["algo_alpha"].asInt(), schemes[i]["algo_beta"].asInt(),
                                        schemes[i]["algo_epsilon"].asInt(), schemes[i]["algo_psi"].asInt());
      }
    slice_state_.assign(num_slices_, 0.0);
    SetMacEntity(0);
    CreateUsersToSchedule();
  }

  virtual ~RsGpuScheduler() {
    if (h_) rs_destroy(h_);
    Destroy();
  }

  virtual void DoSchedule(void) {
    RrcEntity* rrc = GetMacEntity()->GetDevice()->GetProtocolStack()->GetRrcEntity();
    RrcEntity::RadioBearersContainer* bearers = rrc->GetRadioBearerContainer();
    /* UpdateAverageTransmissionRate (downlink-transport-scheduler.cpp:715-727): the bearers' own method */
    for (auto it = bearers->begin(); it != bearers->end(); ++it) (*it)->UpdateAverageTransmissionRate();
    SelectUsers(bearers);
    if (n_users_total_ != 0) RBsAllocation();
    StopSchedule();
  }

  virtual void DoStopSchedule(void) {
    /* byte accounting + RLC, as downlink-transport-scheduler.cpp:170-221 */
    PacketBurst* burst = new PacketBurst();
    UsersToSchedule* users = GetUsersToSchedule();
    for (auto it = users->begin(); it != users->end(); ++it) {
      UserToSchedule* user = *it;
      int available = user->GetAllocatedBits() / 8;
      for (int i = MAX_BEARERS - 1; i >= 0 && available > 0; i--) {
        if (user->m_dataToTransmit[i] <= 0) continue;
        RadioBearer* bearer = user->m_bearers[i];
        /* DL_PF_PacketScheduler::DoStopSchedule hands the RLC all allocated bytes (dl-pf-packet-scheduler.cpp:80-82);
         * the user-level schedulers cap them by the queue (downlink-transport-scheduler.cpp:183-186) */
        const int sent = (id_ == 1 || available < user->m_dataToTransmit[i]) ? available : user->m_dataToTransmit[i];
        available -= sent;
        bearer->UpdateTransmittedBytes(sent);
        bearer->UpdateCumulateRBs(user->GetListOfAllocatedRBs()->size());
        std::cerr << GetTimeStamp() << " app: " << bearer->GetApplication()->GetApplicationID()
                  << " cumu_bytes: " << bearer->GetCumulateBytes() << " cumu_rbs: " << bearer->GetCumulateRBs()
                  << " hol_delay: " << bearer->GetHeadOfLinePacketDelay() << " user: " << user->GetUserID()
                  << " slice: " << user_to_slice_[user->GetUserID()] << std::endl;
        PacketBurst* part = bearer->GetRlcEntity()->TransmissionProcedure(sent);
        if (part->GetNPackets() > 0) {
          std::list<Packet*> packets = part->GetPackets();
          for (auto p = packets.begin(); p != packets.end(); ++p) burst->AddPacket((*p)->Copy());
        }
        delete part;
      }
    }
    UpdateTimeStamp();
    GetMacEntity()->GetDevice()->SendPacketBurst(burst);
  }

 private:
  int id_;
  rs_handle* h_ = nullptr;
  int n_rbs_ = 0, rbg_size_ = 0, n_rbgs_ = 0;
  int n_users_total_ = 0;
  std::vector<uint8_t> cqi_, active_, mcs_, final_cqi_;
  std::vector<double> avg_, hol_;   /* hol_: head-of-line delay of each listed bearer */
  std::vector<int32_t> queue_;      /* dataToTransmit of each listed bearer, 0 = not listed */
  std::vector<int16_t> rbg_to_ue_, grant_ue_, grant_rbg_;
  std::vector<int> slice_priority_;   /* highest priority among the listed bearers of each slice */
  std::vector<int32_t> bits_, target_, quota_, draws_;

  /* DownlinkTransportScheduler with one of its inter-slice algorithms (ENodeB.cpp:357-385): 8 Sequential,
   * 9 MaximizeCell (RadioSaber), 10 UpperBound, 101 SubOpt, 103 VogelApproximate */
  bool Nvs() const { return id_ == 7 || id_ == 11; }   /* DownlinkNVSScheduler(config, non_greedy), ENodeB.cpp:345-355 */
  bool Transport() const { return id_ == 8 || id_ == 9 || id_ == 10 || id_ == 101 || id_ == 103; }

  static void Check(int rc, const char* what) {
    if (rc != RS_OK) throw std::runtime_error(std::string("RsGpuScheduler: ") + what + ": " + rs_last_error());
  }

  void EnsureHandle() {
    if (h_) return;
    n_rbs_ = (int)GetMacEntity()->GetDevice()->GetPhy()->GetBandwidthManager()->GetDlSubChannels().size();
    rbg_size_ = get_rbg_size(n_rbs_);
    /* nb_rbs = nb_rbs - (nb_rbs % rbg_size), downlink-transport-scheduler.cpp:460 / downlink-nvs-scheduler.cpp:281;
     * DownlinkPacketScheduler rounds up instead (a short last RBG, downlink-packet-scheduler.cpp:190): id 1 keeps
     * the full count and rs_create refuses a band that is not whole RBGs */
    if (id_ != 1) n_rbs_ -= n_rbs_ % rbg_size_;
    n_rbgs_ = n_rbs_ / rbg_size_;
    const int U = (int)user_to_slice_.size(), S = num_slices_;
    std::vector<int32_t> params(4 * S), u2s(user_to_slice_.begin(), user_to_slice_.end());
    for (int s = 0; s < S; ++s) {
      params[4 * s + 0] = slice_algo_params_[s].alpha;
      params[4 * s + 1] = slice_algo_params_[s].beta;
      params[4 * s + 2] = slice_algo_params_[s].epsilon;
      params[4 * s + 3] = slice_algo_params_[s].psi;
    }
    /* TransportBlockSizeTable[-1][itbs] as THIS build's AMCModule reads it (AMCModule.cpp:312-316):
     * TBS(mcs,120) = 5*T[23][itbs] + T[-1][itbs] and TBS(mcs,24) = T[23][itbs]. */
    AMCModule* amc = GetMacEntity()->GetAmcModule();
    static const int kMcsOfItbs[27] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 11, 12, 13, 14, 15, 16, 18,
                                       19, 20, 21, 22, 23, 24, 25, 26, 27, 28};
    int32_t row_m1[27];
    for (int itbs = 0; itbs < 27; ++itbs)
      row_m1[itbs] = amc->GetTBSizeFromMCS(kMcsOfItbs[itbs], 120) - 5 * amc->GetTBSizeFromMCS(kMcsOfItbs[itbs], 24);
    rs_config cfg;
    cfg.algo = id_;
    cfg.n_slices = S;
    cfg.n_ues = U;
    cfg.n_rbs = n_rbs_;
    cfg.rbg_size = rbg_size_;
    cfg.cqi_per_rb = 1; /* ENodeB::UserEquipmentRecord::GetCQI() is one value per RB */
    cfg.data_to_transmit = 100000000;
    cfg.n_bearers = 1; /* two bearers of a UE are folded into one user here, like InsertFlowToUser does */
    cfg.weight = slice_weights_.data();
    cfg.params = params.data();
    cfg.ue_to_slice = u2s.data();
    cfg.tbs_row_m1 = row_m1;
    const char* dev = getenv("RS_DEVICE");
    Check(rs_create(&cfg, 1, dev ? atoi(dev) : 0, &h_), "rs_create");
    /* UpperBound: every slice may take its own best RBGs, up to S * G grants; list them all */
    if (id_ == 10) Check(rs_set_grant_list_len(h_, std::max(S * n_rbgs_, 2 * n_rbgs_)), "rs_set_grant_list_len");
    cqi_.assign((size_t)U * n_rbs_, 10); /* UserEquipmentRecord's initial CQI, ENodeB.cpp:207-217 */
    active_.assign(U, 0);
    queue_.assign(U, 0);
    hol_.assign(U, 0.0);
    avg_.assign(U, 100000.0);
    mcs_.assign(U, 0xff);
    final_cqi_.assign(U, 0);
    bits_.assign(U, 0);
    rbg_to_ue_.assign(n_rbgs_, -1);
    target_.assign(S, 0);
    quota_.assign(S, 0);
  }

  /* SelectFlowsToSchedule (downlink-transport-scheduler.cpp:105-150; for id 7 every slice is listed
   * here and the GPU picks the slice, downlink-nvs-scheduler.cpp:144-194).  Builds the
   * UserToSchedule objects the rest of LTE-Sim expects, without the per-RB efficiency vector and
   * the wideband-CQI EESM (dead work for backlogged bearers). */
  void SelectUsers(RrcEntity::RadioBearersContainer* bearers) {
    ClearUsersToSchedule();
    n_users_total_ = 0;
    if (bearers->empty()) return;
    EnsureHandle();
    std::fill(active_.begin(), active_.end(), (uint8_t)0);
    std::fill(queue_.begin(), queue_.end(), 0);
    std::fill(hol_.begin(), hol_.end(), 0.0);
    slice_priority_.assign(num_slices_, 0);   /* :115 */
    ENodeB* enb = (ENodeB*)GetMacEntity()->GetDevice();
    UsersToSchedule* users = GetUsersToSchedule();
    for (auto it = bearers->begin(); it != bearers->end(); ++it) {
      RadioBearer* bearer = *it;
      if (!(bearer->HasPackets() && bearer->GetDestination()->GetNodeState() == NetworkNode::STATE_ACTIVE)) continue;
      /* dataToTransmit as downlink-transport-scheduler.cpp:121-128 */
      const int data = (bearer->GetApplication()->GetApplicationType() == Application::APPLICATION_TYPE_INFINITE_BUFFER)
                           ? 100000000 : bearer->GetQueueSize();
      const int uid = bearer->GetUserID();
      if (uid < 0 || uid >= (int)user_to_slice_.size()) throw std::runtime_error("RsGpuScheduler: user id outside the slice config");
      UserToSchedule* user = nullptr;
      for (auto u = users->begin(); u != users->end(); ++u)
        if ((*u)->GetUserID() == uid) user = *u;
      /* A second bearer of a UE joins the same UserToSchedule (InsertFlowToUser, packet-scheduler.cpp:304-318).  Id 1
       * schedules flows, and id 11's 300-sample search has no gate for an empty prioritised bearer: not covered. */
      if (user && (id_ == 1 || id_ == 11)) throw std::runtime_error("RsGpuScheduler: two bearers on one UE are not covered for ids 1 and 11");
      const int prio = bearer->GetPriority();
      if (prio < 0 || prio >= MAX_BEARERS) throw std::runtime_error("RsGpuScheduler: bearer priority outside MAX_BEARERS");
      const int slice = user_to_slice_[uid];
      if (prio > slice_priority_[slice]) slice_priority_[slice] = prio;   /* :144-146 */
      if (!user) {
        user = new UserToSchedule(uid, bearer->GetDestination());
        std::vector<int> cqi = enb->GetUserEquipmentRecord(bearer->GetDestination()->GetIDNetworkNode())->GetCQI();
        user->SetCqiFeedbacks(cqi);
        for (int r = 0; r < n_rbs_ && r < (int)cqi.size(); ++r) cqi_[(size_t)uid * n_rbs_ + r] = (uint8_t)cqi[r];
        avg_[uid] = 0.0;
        users->push_back(user);
        queue_[uid] = data;   /* m_requiredRBs counts the bearer that created the user (packet-scheduler.cpp:333) */
      }
      user->m_bearers[prio] = bearer;
      user->m_dataToTransmit[prio] = data;
      avg_[uid] += bearer->GetAverageTransmissionRate();   /* :683-687: the sum over the listed bearers */
      active_[uid] = 1;
      n_users_total_++;
    }
    /* the head-of-line delay in the metric is the one of the bearer with the slice's priority; a user whose bearer of
     * that priority is empty has metric 0 (:696-706, nvs :379-386) -- see rs_set_queues for how that is passed */
    for (auto u = users->begin(); u != users->end(); ++u) {
      const int uid = (*u)->GetUserID(), slice = user_to_slice_[uid], pr = slice_priority_[slice];
      if (id_ == 1 || slice_algo_params_[slice].alpha == 0) { hol_[uid] = 0.0; continue; }
      if ((*u)->m_dataToTransmit[pr] == 0)
        hol_[uid] = (Nvs() || slice_algo_params_[slice].beta) ? 0.0 : -1.0;
      else
        hol_[uid] = (*u)->m_bearers[pr]->GetHeadOfLinePacketDelay();
    }
  }

  /* RBsAllocation (downlink-transport-scheduler.cpp:453-675) through the C ABI */
  void RBsAllocation() {
    const int U = (int)user_to_slice_.size(), S = num_slices_;
    int32_t rand2[2] = {0, 0};
    const int32_t* draws = rand2;
    int host_slice = -1;
    if (Transport()) { /* the two draws of :490 and :511, in the reference's order */
      rand2[0] = rand();
      rand2[1] = rand();
    } else if (id_ == 11) {
      /* The non-greedy search draws 300 x (listed users of the served slice) libc rand() values
       * (downlink-nvs-scheduler.cpp:437-446).  To take exactly that many from the process's stream the host must
       * know the slice first: the choice of SelectSliceToServe (:94-127) from the credits it already holds.  The
       * device makes the same choice from the same numbers; a disagreement throws below. */
      std::vector<char> with_queue(S, 0);
      for (int u = 0; u < U; ++u)
        if (active_[u] && queue_[u] > 0) with_queue[user_to_slice_[u]] = 1;
      double max_score = 0;
      host_slice = 0;
      for (int i = 0; i < S; ++i) {
        if (!with_queue[i]) continue;
        if (slice_state_[i] == 0) { host_slice = i; break; }
        const double score = slice_weights_[i] / slice_state_[i];
        if (score >= max_score) { max_score = score; host_slice = i; }
      }
      int listed = 0;
      for (int u = 0; u < U; ++u)
        if (active_[u] && queue_[u] > 0 && user_to_slice_[u] == host_slice) listed++;
      const int stride = rs_rand_draws_per_cell_tti(h_);
      if (300 * listed > stride) throw std::runtime_error("RsGpuScheduler: more rand() draws than the ABI takes");
      draws_.assign((size_t)(stride > 2 ? stride : 2), 0);
      for (int k = 0; k < 300 * listed; ++k) draws_[k] = rand();
      draws = draws_.data();
    }
    /* One call per TTI (rs_step_cell): the bearers' rates, the slice offsets / NVS credits and the queue state go up
     * with the CQI in one copy, the results and the updated per-slice state come back in one copy.  Finite queues cap
     * the bytes, bind id 7's required-RBs guard and id 1's flow-satisfied cut-off, and the head-of-line delay enters
     * the metric of alpha/beta slices.  dt = 0: the EWMA was applied by the bearers themselves a few lines up. */
    rs_cell_io io = {};
    int32_t nvs_slice = -1;
    int32_t n_grants = 0;
    io.avg_rate = avg_.data();
    io.slice_state = (Transport() || Nvs()) ? slice_state_.data() : nullptr;
    io.cqi = cqi_.data();
    io.rand2 = draws;
    io.active = active_.data();
    io.queue_bytes = queue_.data();
    io.hol_delay = hol_.data();
    io.dt = 0.0;
    io.out.rbg_to_ue = rbg_to_ue_.data();
    io.out.tbs_bits = bits_.data();
    io.out.mcs = mcs_.data();
    io.out.final_cqi = final_cqi_.data();
    io.out.slice_target = target_.data();
    io.out.slice_quota = quota_.data();
    io.out.nvs_slice = &nvs_slice;
    if (id_ == 10) { /* UpperBound books an RBG to several slices: the grants come back as a list */
      grant_ue_.assign((size_t)rs_grant_list_len(h_), -1);
      grant_rbg_.assign((size_t)rs_grant_list_len(h_), -1);
      io.out.alloc_n = &n_grants;
      io.out.alloc_ue = grant_ue_.data();
      io.out.alloc_rbg = grant_rbg_.data();
    }
    const auto c0 = std::chrono::steady_clock::now();
    Check(rs_step_cell(h_, &io), "rs_step_cell");
    step_seconds_ += std::chrono::duration<double>(std::chrono::steady_clock::now() - c0).count();
    step_calls_++;
    if (id_ == 11 && nvs_slice != host_slice) throw std::runtime_error("RsGpuScheduler: host and device disagree on the NVS slice");

    UsersToSchedule* users = GetUsersToSchedule();
    if (Nvs()) { /* only the served slice's users are "users to schedule" (downlink-nvs-scheduler.cpp:161-162) */
      for (auto it = users->begin(); it != users->end();) {
        if (user_to_slice_[(*it)->GetUserID()] != nvs_slice) { delete *it; it = users->erase(it); } else ++it;
      }
    } else if (id_ != 1) { /* the reference's log line, :523-527 */
      std::cout << "slice_id, target_rbs, quota_rbgs: ";
      for (int i = 0; i < S; ++i) std::cout << "(" << i << ", " << target_[i] << ", " << quota_[i] << ") ";
      std::cout << std::endl;
    }
    std::vector<UserToSchedule*> by_id(U, nullptr);
    for (auto it = users->begin(); it != users->end(); ++it) by_id[(*it)->GetUserID()] = *it;
    if (id_ == 10) {
      for (int k = 0; k < n_grants; ++k) {   /* per user in grant order, like the reference fills the RB lists */
        const int ue = grant_ue_[k], g = grant_rbg_[k];
        if (ue < 0 || ue >= U || !by_id[ue]) continue;
        for (int r = g * rbg_size_; r < (g + 1) * rbg_size_; ++r) by_id[ue]->GetListOfAllocatedRBs()->push_back(r);
      }
    } else {
      for (int g = 0; g < n_rbgs_; ++g) {
        const int ue = rbg_to_ue_[g];
        if (ue < 0 || !by_id[ue]) continue;
        for (int r = g * rbg_size_; r < (g + 1) * rbg_size_; ++r) by_id[ue]->GetListOfAllocatedRBs()->push_back(r);
      }
    }
    PdcchMapIdealControlMessage* pdcch = new PdcchMapIdealControlMessage();
    if (id_ != 1) std::cout << GetTimeStamp() << std::endl;   /* DownlinkPacketScheduler::RBsAllocation prints nothing */
    for (auto it = users->begin(); it != users->end(); ++it) {
      UserToSchedule* ue = *it;
      std::vector<int>* rbs = ue->GetListOfAllocatedRBs();
      if (rbs->empty()) continue;
      if (id_ != 1) {
        std::cout << "User(" << ue->GetUserID() << ") allocated RBGS:";
        for (size_t i = 0; i < rbs->size(); i++)
          if (rbs->at(i) % rbg_size_ == 0)
            std::cout << " " << rbs->at(i) / rbg_size_ << "(" << ue->GetCqiFeedbacks().at(rbs->at(i)) << ")";
        std::cout << " final_cqi: " << (int)final_cqi_[ue->GetUserID()] << std::endl;
      }
      ue->UpdateAllocatedBits(bits_[ue->GetUserID()]);
      for (size_t i = 0; i < rbs->size(); i++)
        pdcch->AddNewRecord(PdcchMapIdealControlMessage::DOWNLINK, rbs->at(i), ue->GetUserNode(), mcs_[ue->GetUserID()]);
    }
    if (pdcch->GetMessage()->size() > 0) GetMacEntity()->GetDevice()->GetPhy()->SendIdealControlMessage(pdcch);
    delete pdcch;
  }
};

#endif /* RS_GPU_SCHEDULER_H_ */
