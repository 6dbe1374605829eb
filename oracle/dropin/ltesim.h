/* oracle/dropin/ltesim.h -- the few LTE-Sim classes radiosaber_b200/host/rs_gpu_scheduler.h uses, reduced to what the
 * plug-in calls.  TEST INFRASTRUCTURE ONLY (oracle/dropin/dropin_replay.cpp).
 *
 * The plug-in includes the simulator's headers by their paths under LTE-Sim's src/ (device/ENodeB.h, ...); the Makefile
 * target `dropin` generates one forwarding header per path that includes this file, so the plug-in compiles unchanged.
 * The bearers carry what the simulator's applications and RLC would hand the scheduler each TTI (packets or not, queue
 * size, head-of-line delay); dropin_replay.cpp sets those from a golden record of the reference.  What the scheduler
 * does to the bearers -- the EWMA of RadioBearer::UpdateAverageTransmissionRate, UpdateTransmittedBytes,
 * UpdateCumulateRBs (flows/radio-bearer.cpp:100-164, restated as in oracle/rs_oracle.cpp) -- is chained here. */
#ifndef RS_DROPIN_LTESIM_H_
#define RS_DROPIN_LTESIM_H_

#include <cstdint>
#include <list>
#include <stdexcept>
#include <string>
#include <vector>

#define MAX_BEARERS 2   /* packet-scheduler.h:31 */

double SimulatorNow();   /* the replayed Simulator::Now(), dropin_replay.cpp */

struct SchedulerAlgoParam {
  int alpha, beta, epsilon, psi;
  SchedulerAlgoParam(int a, int b, int e, int p) : alpha(a), beta(b), epsilon(e), psi(p) {}
};

/* RBG size of a downlink band; every recorded cell is 100 MHz = 512 RBs in RBGs of 8 */
inline int get_rbg_size(int n_rbs) {
  if (n_rbs != 512) throw std::runtime_error("dropin replay: only the 512-RB band of the golden records");
  return 8;
}

class Packet {
 public:
  Packet* Copy() { return new Packet(*this); }
};

class PacketBurst {
 public:
  ~PacketBurst() { for (Packet* p : packets_) delete p; }
  int GetNPackets() const { return (int)packets_.size(); }
  std::list<Packet*> GetPackets() { return packets_; }
  void AddPacket(Packet* p) { packets_.push_back(p); }
 private:
  std::list<Packet*> packets_;
};

/* the replay has no packet objects: queues come from the record, so the RLC hands back an empty burst */
class RlcEntity {
 public:
  PacketBurst* TransmissionProcedure(int) { return new PacketBurst(); }
};

class Application {
 public:
  enum ApplicationType { APPLICATION_TYPE_INFINITE_BUFFER, APPLICATION_TYPE_INTERNET_FLOW };
  ApplicationType type = APPLICATION_TYPE_INFINITE_BUFFER;
  int id = 0;
  ApplicationType GetApplicationType() const { return type; }
  int GetApplicationID() const { return id; }
};

class BandwidthManager {
 public:
  std::vector<double> GetDlSubChannels() const { return std::vector<double>(512, 0.0); }
};

class IdealControlMessage {};
class NetworkNode;
class PdcchMapIdealControlMessage : public IdealControlMessage {
 public:
  enum ChannelDirection { DOWNLINK, UPLINK };
  struct Record { ChannelDirection dir; int rb; NetworkNode* node; int mcs; };
  void AddNewRecord(ChannelDirection d, int rb, NetworkNode* n, int mcs) { records_.push_back({d, rb, n, mcs}); }
  std::vector<Record>* GetMessage() { return &records_; }
 private:
  std::vector<Record> records_;
};

class LtePhy {
 public:
  BandwidthManager* GetBandwidthManager() { return &bw_; }
  void SendIdealControlMessage(IdealControlMessage*) {}
 private:
  BandwidthManager bw_;
};

class RadioBearer;
class RrcEntity {
 public:
  typedef std::vector<RadioBearer*> RadioBearersContainer;
  RadioBearersContainer* GetRadioBearerContainer() { return &bearers_; }
 private:
  RadioBearersContainer bearers_;
};

class ProtocolStack {
 public:
  RrcEntity* GetRrcEntity() { return &rrc_; }
 private:
  RrcEntity rrc_;
};

class NetworkNode {
 public:
  enum NodeState { STATE_ACTIVE, STATE_IDLE };
  int id = 0;
  virtual ~NetworkNode() {}
  NodeState GetNodeState() const { return STATE_ACTIVE; }
  int GetIDNetworkNode() const { return id; }
  LtePhy* GetPhy() { return &phy_; }
  ProtocolStack* GetProtocolStack() { return &stack_; }
  void SendPacketBurst(PacketBurst* b) { delete b; }
 private:
  LtePhy phy_;
  ProtocolStack stack_;
};

class ENodeB : public NetworkNode {
 public:
  struct UserEquipmentRecord {
    std::vector<int> cqi;
    std::vector<int> GetCQI() const { return cqi; }
  };
  std::vector<UserEquipmentRecord> ues;   /* indexed by the UE's node id */
  UserEquipmentRecord* GetUserEquipmentRecord(int id) { return &ues.at(id); }
};

class RadioBearer {
 public:
  /* the reference's member names, which the recording reads */
  double m_averageTransmissionRate = 0;
  int m_transmittedBytes = 0;
  double m_lastUpdate = 0;
  uint64_t m_cumulativeBytes = 0, m_cumulativeRBs = 0;
  /* set each TTI from the record: what the applications and the RLC queue hold */
  bool has_packets = true;
  int queue_size = 100000000;
  double hol_delay = 0;
  int user_id = 0, priority = 0;
  NetworkNode* destination = nullptr;
  Application application;
  RlcEntity rlc;

  void UpdateAverageTransmissionRate() {
    const double dt = SimulatorNow() - m_lastUpdate;
    if (dt != 0) {
      double rate = (m_transmittedBytes * 8) / dt;
      double beta = 0.02;
      m_averageTransmissionRate = ((1 - beta) * m_averageTransmissionRate) + (beta * rate);
      if (m_averageTransmissionRate < 1) m_averageTransmissionRate = 1;
      m_transmittedBytes = 0;
    }
    m_lastUpdate = SimulatorNow();
  }
  void UpdateTransmittedBytes(int bytes) { m_transmittedBytes += bytes; m_cumulativeBytes += bytes; }
  void UpdateCumulateRBs(int rbs) { m_cumulativeRBs += rbs; }
  uint64_t GetCumulateBytes() const { return m_cumulativeBytes; }
  uint64_t GetCumulateRBs() const { return m_cumulativeRBs; }
  double GetAverageTransmissionRate() const { return m_averageTransmissionRate; }
  double GetHeadOfLinePacketDelay() const { return hol_delay; }
  int GetQueueSize() const { return queue_size; }
  bool HasPackets() const { return has_packets; }
  NetworkNode* GetDestination() { return destination; }
  Application* GetApplication() { return &application; }
  RlcEntity* GetRlcEntity() { return &rlc; }
  int GetUserID() const { return user_id; }
  int GetPriority() const { return priority; }
};

/* AMCModule::GetTBSizeFromMCS is read by the plug-in only as TBS(mcs,120) - 5 TBS(mcs,24) = TransportBlockSizeTable[-1]
 * (AMCModule.cpp:312-316).  The stock -O0 build reads McsToItbs[itbs + 5] there (0 past its end), which is what this
 * difference returns. */
class AMCModule {
 public:
  int GetTBSizeFromMCS(int mcs, int nrb) const {
    static const int kMcsToItbs[29] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 10, 11, 12, 13, 14, 15, 15, 16,
                                       17, 18, 19, 20, 21, 22, 23, 24, 25, 26};
    if (mcs < 0 || mcs > 28 || (nrb != 120 && nrb != 24))
      throw std::runtime_error("AMCModule stand-in: only TBS(mcs, 120) - 5 TBS(mcs, 24) is modelled");
    const int itbs = kMcsToItbs[mcs];
    return nrb == 120 ? (itbs + 5 < 29 ? kMcsToItbs[itbs + 5] : 0) : 0;
  }
};

class MacEntity {
 public:
  NetworkNode* device = nullptr;
  NetworkNode* GetDevice() { return device; }
  AMCModule* GetAmcModule() { return &amc_; }
 private:
  AMCModule amc_;
};

class PacketScheduler {
 public:
  class UserToSchedule {
   public:
    RadioBearer* m_bearers[MAX_BEARERS] = {nullptr, nullptr};
    int m_dataToTransmit[MAX_BEARERS] = {0, 0};
    UserToSchedule(int id, NetworkNode* node) : id_(id), node_(node) {}
    int GetUserID() const { return id_; }
    NetworkNode* GetUserNode() { return node_; }
    void SetCqiFeedbacks(std::vector<int> cqi) { cqi_ = cqi; }
    std::vector<int> GetCqiFeedbacks() { return cqi_; }
    std::vector<int>* GetListOfAllocatedRBs() { return &rbs_; }
    int GetAllocatedBits() const { return bits_; }
    void UpdateAllocatedBits(int bits) { bits_ += bits; }
   private:
    int id_;
    NetworkNode* node_;
    std::vector<int> cqi_, rbs_;
    int bits_ = 0;
  };
  typedef std::vector<UserToSchedule*> UsersToSchedule;

  virtual ~PacketScheduler() {}
  virtual void DoSchedule() = 0;
  virtual void DoStopSchedule() = 0;
  void SetMacEntity(MacEntity* mac) { mac_ = mac; }
  MacEntity* GetMacEntity() { return mac_; }
  void CreateUsersToSchedule() { users_ = new UsersToSchedule(); }
  UsersToSchedule* GetUsersToSchedule() { return users_; }
  void ClearUsersToSchedule() {
    for (UserToSchedule* u : *users_) delete u;
    users_->clear();
  }
  void Destroy() {
    if (!users_) return;
    ClearUsersToSchedule();
    delete users_;
    users_ = nullptr;
  }
  void StopSchedule() { DoStopSchedule(); }
  int GetTimeStamp() const { return timestamp_; }
  void SetTimeStamp(int ts) { timestamp_ = ts; }   /* the replay starts at the recorded TTI's count */
  void UpdateTimeStamp() { timestamp_++; }

 private:
  MacEntity* mac_ = nullptr;
  UsersToSchedule* users_ = nullptr;
  int timestamp_ = 0;
};

#endif /* RS_DROPIN_LTESIM_H_ */
