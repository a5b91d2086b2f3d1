// rpk_host.hpp -- C++ mirror of the reference's Provider surface for the hot path.
//
// The reference is Go and no Go toolchain exists in the build image, so the host side above the C-ABI is
// written in C++ (the Go binding a maintainer would add is in go/rpk and INTEGRATION.md).  Names, argument
// meaning and error behaviour follow pkg/virtual_kubelet:
//
//   Provider::CreatePod/UpdatePod/DeletePod/GetPod/GetPodStatus/GetPods/NotifyPods   kubelet.go:384-731
//   Provider::ProcessPendingPods     kubelet.go:747-814   (now ONE rpk_select per tick instead of one
//                                                           GraphQL fetch + filter + sort per pod)
//   Provider::UpdateAllPodStatuses   kubelet.go:816-974   (now ONE rpk_status_diff per tick)
//   PrepareColumns / column producers runpod_client.go:1102-1134, 1181-1191, 1261-1281
//   CheckPortsExposed                kubelet.go:566-605
//   TranslateRunPodStatus            kubelet.go:1848-2024 (the phase / readiness / container-state table)
//
// Everything network-facing (GraphQL/REST transport, k8s API server) is behind the RunPodAPI interface and
// stays out of scope; tests plug a scripted fake in.
#pragma once
#include <condition_variable>
#include <cstdint>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "rpk.h"

namespace rpkhost {

// ---- annotation schema (runpod_client.go:37-52) --------------------------------------------------------
constexpr const char* PodIDAnnotation = "runpod.io/pod-id";
constexpr const char* CostAnnotation = "runpod.io/cost-per-hr";
constexpr const char* CloudTypeAnnotation = "runpod.io/cloud-type";
constexpr const char* TemplateIdAnnotation = "runpod.io/templateId";
constexpr const char* GpuMemoryAnnotation = "runpod.io/required-gpu-memory";
constexpr const char* ContainerRegistryAuthAnnotation = "runpod.io/container-registry-auth-id";
constexpr const char* DatacenterAnnotation = "runpod.io/datacenter-ids";
constexpr const char* PortsAnnotation = "runpod.io/ports";
// extension annotations of this build (absent = reference behaviour)
constexpr const char* MaxPriceAnnotation = "runpod.io/max-price-per-hr";
constexpr const char* VcpuAnnotation = "runpod.io/required-vcpu";
constexpr const char* RamAnnotation = "runpod.io/required-ram-gb";
// comma-separated GPU type ids the pod may run on (parsed like DatacenterAnnotation, runpod_client.go:1354-1362)
constexpr const char* GpuTypeIdsAnnotation = "runpod.io/gpu-type-ids";
constexpr double DefaultMaxPrice = 0.5;  // runpod_client.go:48

// PodStatus enum strings (runpod_client.go:55-64)
constexpr const char* PodRunning = "RUNNING";
constexpr const char* PodStarting = "STARTING";
constexpr const char* PodTerminating = "TERMINATING";
constexpr const char* PodTerminated = "TERMINATED";
constexpr const char* PodNotFound = "NOT_FOUND";
constexpr const char* PodExited = "EXITED";

using Annotations = std::map<std::string, std::string>;

// the slice of v1.Pod this path reads and writes
struct PodStatusView {  // what translateRunPodStatus decides (kubelet.go:1848-2024)
    std::string phase = "Unknown";       // v1.PodPhase
    bool ready = false;                  // containerStatus.Ready and the Ready/ContainersReady conditions
    bool started = false;                // containerStatus.Started
    std::string state = "Waiting";       // Running | Waiting | Terminated
    std::string reason;                  // Waiting/Terminated reason
    std::string message;                 // podStatus.Message = statusMessage (kubelet.go:2013)
    std::string container_message;       // State.Waiting / State.Terminated Message (kubelet.go:1885,1899,1923,1950,1963,1975)
    int exit_code = 0;
    bool operator==(const PodStatusView& o) const {
        return phase == o.phase && ready == o.ready && started == o.started && state == o.state && reason == o.reason &&
               message == o.message && container_message == o.container_message && exit_code == o.exit_code;
    }
};

struct Pod {
    std::string ns, name;
    Annotations annotations;
    std::vector<std::string> container_ports;  // "8080/http", "5432/tcp" (extractPortsFromPod's result)
    PodStatusView status;
    std::shared_ptr<Annotations> owner_job;    // annotations of the owning Job, if any (getOwnerJob)
};
using PodPtr = std::shared_ptr<Pod>;

struct InstanceInfo {  // runpod_client.go:98-109
    std::string ID;
    double CostPerHr = 0;
    std::string PodName, Namespace, Status, StatusMessage;
    int ExitCode = 0;
    double CreationTime = 0;  // seconds, from the provider's clock
    std::vector<std::string> RequestedPorts;
    bool PortsExposed = false;
};

struct GPUType {  // runpod_client.go:83-95 (+ the two extension columns)
    std::string ID, DisplayName;
    int MemoryInGb = 0;
    bool SecureCloud = false;
    double SecurePrice = 0;
    bool CommunityCloud = false;
    double CommunityPrice = 0;
    int VCPU = 0, RAMGb = 0;
};

struct DetailedStatus {  // GetDetailedPodStatus's result (runpod_client.go:773)
    std::string DesiredStatus;
    std::map<std::string, int> PortMappings;
};

// The out-of-scope transport (runpod_client.go:160-843): RunPod GraphQL/REST.
class RunPodAPI {
public:
    virtual ~RunPodAPI() = default;
    virtual bool FetchGPUTypes(std::vector<GPUType>* out, std::string* err) = 0;                  // :431-455
    virtual bool DeployPod(const Pod& pod, const std::vector<std::string>& gpu_type_ids, int min_ram_per_gpu,
                           const std::string& cloud_type, std::string* id, double* cost_per_hr, std::string* err) = 0;  // :522
    virtual bool GetDetailedPodStatus(const std::string& id, DetailedStatus* out, std::string* err) = 0;  // :773
    virtual bool TerminatePod(const std::string& id, std::string* err) = 0;                        // :712
};

// ---- column producers ------------------------------------------------------------------------------------
std::string GetAnnotationWithFallback(const Pod& pod, const std::string& key, const std::string& def);  // :1102-1112
std::string ValidateCloudType(const std::string& v);                                                    // :1115-1134
long long ExtractGPUMemory(const std::string& v);                                                       // :1181-1191
std::vector<std::string> GetRequestedPorts(const Pod& pod);                                             // :1381-1393
bool CheckPortsExposed(const std::map<std::string, int>& port_mappings, const std::vector<std::string>& requested);  // kubelet.go:566-605
PodStatusView TranslateRunPodStatus(const std::string& status, const std::string& message, bool has_exposed_ports);  // kubelet.go:1848-2024
// canonical slot [len | flag << 7][status][0x00][ports][zero pad] (include/rpk.h); false if the status does not fit the stride
bool EncodeStatusRecord(uint8_t* slot, uint32_t stride, const std::string& status, bool ports_exposed, bool message_has_error = false);
bool MessageHasError(const std::string& message);  // strings.Contains(strings.ToLower(m), "error") || ... "fail" (kubelet.go:1907-1908)
// the same decision from the 16-bit code the sweep kernel emits next to a changed slot (RPK_CODE_*): no string work
PodStatusView StatusFromCode(uint16_t code, const std::string& status, const std::string& message);

// runpod.io/gpu-type-ids value -> ids: strings.Split(v, ",") then strings.TrimSpace on each element, exactly like the
// datacenter list (runpod_client.go:1354-1362); "" (annotation absent) -> no restriction (empty vector)
std::vector<std::string> ParseGpuTypeIds(const std::string& v);

struct PodColumns {  // one row of the P x G grid
    int32_t req_mem_gb;
    int32_t req_vcpu, req_ram_gb;
    double max_price;
    uint8_t cloud;  // RPK_CLOUD_*
    std::string cloud_type;  // "SECURE" | "COMMUNITY"
    bool restricted = false;               // runpod.io/gpu-type-ids present (pod, else owner Job)
    std::vector<std::string> gpu_type_ids; // its parsed list
};
PodColumns PrepareColumns(const Pod& pod);  // the annotation half of PrepareRunPodParameters (:1255-1281)

// The pod side of the grid as the struct-of-arrays rpk_select takes (row i = pods[i]).
struct PodColumnsSoA {
    std::vector<int32_t> req_mem_gb, req_vcpu, req_ram_gb;
    std::vector<double> max_price;
    std::vector<uint8_t> cloud;
    std::vector<std::string> gpu_type_ids;  // raw runpod.io/gpu-type-ids value per row, "" = unrestricted
    void resize(size_t n) {
        req_mem_gb.resize(n); req_vcpu.resize(n); req_ram_gb.resize(n); max_price.resize(n); cloud.resize(n); gpu_type_ids.assign(n, "");
    }
    size_t size() const { return req_mem_gb.size(); }
};
// Column ingest for a whole batch: PrepareColumns for every pod, rows split contiguously over n_threads host
// threads (0 = one per hardware thread, capped so that a thread has at least a few thousand rows).  Same
// result as the per-pod producer, row for row.  At the batch sizes the grid kernel is built for this -- not
// the GPU -- is what a tick costs: see host_test --bench-columns and DESIGN.md section 8.
void PrepareColumnsBatch(const std::vector<PodPtr>& pods, PodColumnsSoA* out, int n_threads = 0);

// ---- Provider ----------------------------------------------------------------------------------------------
struct ProviderOptions {
    // The reference drives itself: NewProvider starts a 30 s status poll and a 30 s pending-pod processor
    // (kubelet.go:374-376, 292-303, 734-745) and NotifyPods starts a 10 s sweep goroutine (kubelet.go:718-729).
    // self_tick = true reproduces that with host threads; false leaves the ticks to the embedding process (tests).
    bool self_tick = false;
    double notify_interval_s = 10, periodic_interval_s = 30, pending_interval_s = 30;
};

class Provider {
public:
    // n_gpus GPUs behind one rpk ctx; throws std::runtime_error when the engine cannot start (no CPU fallback)
    Provider(std::shared_ptr<RunPodAPI> api, int n_gpus = 1, uint32_t max_pods = 1024, ProviderOptions opt = ProviderOptions());
    ~Provider();

    // node.PodLifecycleHandler (kubelet.go:384-711); empty string = nil error
    std::string CreatePod(const PodPtr& pod);
    std::string UpdatePod(const PodPtr& pod);
    std::string DeletePod(const PodPtr& pod);
    std::pair<PodPtr, std::string> GetPod(const std::string& ns, const std::string& name);
    std::pair<PodStatusView, std::string> GetPodStatus(const std::string& ns, const std::string& name);
    std::vector<PodPtr> GetPods();
    // node.PodNotifier (kubelet.go:713-731): stores the callback and -- with self_tick -- starts the 10 s sweep thread
    void NotifyPods(std::function<void(const PodPtr&)> cb);
    void StopTickers();  // ctx.Done() of the reference's goroutines

    // the two ticker bodies, batched
    void ProcessPendingPods();     // kubelet.go:747-814
    void UpdateAllPodStatuses();   // kubelet.go:816-974

    // observability for tests / the benchmark harness
    const InstanceInfo* Info(const std::string& ns, const std::string& name);
    uint64_t SelectCalls() const { return select_calls_; }
    uint64_t StatusCalls() const { return status_calls_; }
    uint64_t OfferUploads() const { return offer_uploads_; }
    uint64_t SetSelectCalls() const { return set_select_calls_; }  // rpk_select_sets calls (batches with gpu-type-ids)
    uint64_t SetUploads() const { return set_uploads_; }
    uint64_t HostCompares() const { return host_compares_; }  // sweeps' pods compared on the host (status longer than any slot)
    uint32_t Stride() const { return stride_; }
    void SetClock(double now_s) { now_ = now_s; }
    rpk_ctx* Ctx() { return ctx_; }

private:
    struct Tracked {
        PodPtr pod;
        InstanceInfo info;
        uint32_t slot;
    };
    static std::string Key(const std::string& ns, const std::string& name) { return ns + "-" + name; }  // kubelet.go:386
    bool RefreshOffersLocked(std::string* err);  // engine_mutex_ held
    bool DeployBatch(const std::vector<std::string>& keys);
    // restricted rows of a batch: distinct gpu-type-ids lists -> offer sets -> rpk_select_sets (engine_mutex_ held);
    // may_reuse = false uploads the sets even if they look resident
    bool SelectWithSetsLocked(const PodColumnsSoA& cols, int32_t* top5, bool may_reuse = true);
    void Notify(const PodPtr& pod);
    uint32_t AllocSlot();
    void SeedSlot(uint32_t slot);                // device previous state of ONE slot := records_[slot]
    void WidenRecords(uint32_t stride);          // re-encode every slot at a wider stride (sweeps are excluded by sweep_mutex_)
    void StartTicker(double interval_s, std::function<void()> body);

    std::shared_ptr<RunPodAPI> api_;
    rpk_ctx* ctx_ = nullptr;
    // kubelet.go:38-45 + the ctx lock + one sweep at a time.  Never nested, except sweep_mutex_ around the others.
    std::mutex pods_mutex_, notify_mutex_, deleted_mutex_, engine_mutex_, sweep_mutex_;
    std::map<std::string, Tracked> pods_;
    std::map<std::string, std::string> deleted_pods_;  // "ns/name" -> RunPod id (kubelet.go:628)
    std::function<void(const PodPtr&)> notify_;
    std::vector<GPUType> offers_;
    std::vector<uint8_t> records_;      // max_pods x stride_: what InstanceInfo says per slot (pods_mutex_)
    uint32_t stride_ = 16;              // every RunPod status fits 16 bytes; widened (32 .. 256) if an API string does not
    uint32_t want_stride_ = 16;
    std::vector<std::thread> tickers_;
    std::mutex tick_mutex_; std::condition_variable tick_cv_; bool tick_stop_ = false, notify_ticker_started_ = false;
    uint64_t host_compares_ = 0;
    std::vector<uint32_t> free_slots_;
    std::vector<std::string> slot_key_;
    uint32_t max_pods_;
    ProviderOptions opt_;
    double now_ = 0;
    uint64_t select_calls_ = 0, status_calls_ = 0, offer_uploads_ = 0, set_select_calls_ = 0, set_uploads_ = 0;
    // offer sets resident on the engine: set s = the ids of set_lists_[s], built on table upload number set_table_
    std::vector<std::vector<std::string>> set_lists_;
    uint64_t set_table_ = 0;
};

}  // namespace rpkhost
