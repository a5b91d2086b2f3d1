// provider.cc -- see rpk_host.hpp.  Host logic only: every P x G evaluation and every status diff goes
// through the C-ABI (include/rpk.h) to the GPU; there is no CPU implementation of either here.
#include <algorithm>
#include <cctype>
#include <cerrno>
#include <climits>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <stdexcept>
#include <thread>

#include "rpk_host.hpp"

namespace rpkhost {

// ---------------------------------------------------------------------------------------------------------
// column producers
// ---------------------------------------------------------------------------------------------------------

// getAnnotationWithFallback -- runpod_client.go:1102-1112
std::string GetAnnotationWithFallback(const Pod& pod, const std::string& key, const std::string& def) {
    auto it = pod.annotations.find(key);
    if (it != pod.annotations.end() && !it->second.empty()) return it->second;
    if (pod.owner_job) {
        auto jt = pod.owner_job->find(key);
        if (jt != pod.owner_job->end() && !jt->second.empty()) return jt->second;
    }
    return def;
}

// strings.ToUpper as far as it can matter for "SECURE"/"COMMUNITY": ASCII letters plus the two runes whose
// upper case is an ASCII letter (U+017F -> S, U+0131 -> I).
static std::string ToUpperForCloud(const std::string& s) {
    std::string out;
    for (size_t i = 0; i < s.size();) {
        unsigned char c = (unsigned char)s[i];
        if (c == 0xC5 && i + 1 < s.size() && (unsigned char)s[i + 1] == 0xBF) { out.push_back('S'); i += 2; continue; }
        if (c == 0xC4 && i + 1 < s.size() && (unsigned char)s[i + 1] == 0xB1) { out.push_back('I'); i += 2; continue; }
        out.push_back((char)(c >= 'a' && c <= 'z' ? c - 'a' + 'A' : c));
        ++i;
    }
    return out;
}

// validateCloudType -- runpod_client.go:1115-1134
std::string ValidateCloudType(const std::string& v) {
    if (v.empty()) return "SECURE";
    const std::string up = ToUpperForCloud(v);
    if (up == "SECURE" || up == "COMMUNITY") return up;
    return "SECURE";  // invalid (e.g. "STANDARD", runpod_test.go:89): warn and default
}

// strconv.Atoi on a 64-bit int: sign, digits only, range error on overflow
static bool GoAtoi(const std::string& s, long long* out) {
    if (s.empty()) return false;
    size_t i = 0;
    bool neg = false;
    if (s[0] == '+' || s[0] == '-') { neg = s[0] == '-'; i = 1; if (s.size() == 1) return false; }
    unsigned long long acc = 0;
    const unsigned long long lim = neg ? (1ull << 63) : (1ull << 63) - 1;
    for (; i < s.size(); ++i) {
        unsigned d = (unsigned)(s[i] - '0');
        if (d > 9) return false;
        if (acc > (lim - d) / 10) return false;
        acc = acc * 10 + d;
    }
    *out = neg ? (long long)(0 - acc) : (long long)acc;
    return true;
}

// extractGPUMemory -- runpod_client.go:1181-1191
long long ExtractGPUMemory(const std::string& v) {
    const long long def = 16;
    if (v.empty()) return def;
    long long m;
    if (GoAtoi(v, &m)) return m;
    return def;
}

static std::string TrimSpace(const std::string& s) {
    size_t a = 0, b = s.size();
    while (a < b && std::isspace((unsigned char)s[a])) ++a;
    while (b > a && std::isspace((unsigned char)s[b - 1])) --b;
    return s.substr(a, b - a);
}

std::vector<std::string> ParseGpuTypeIds(const std::string& v) {
    std::vector<std::string> out;
    if (v.empty()) return out;
    size_t start = 0;
    while (true) {  // strings.Split(v, ","): empty elements are kept ("a,,b" -> "a", "", "b"); they match no GPU type
        const size_t comma = v.find(',', start);
        out.push_back(TrimSpace(v.substr(start, comma == std::string::npos ? std::string::npos : comma - start)));
        if (comma == std::string::npos) break;
        start = comma + 1;
    }
    return out;
}

// GetRequestedPorts -- runpod_client.go:1381-1393 (the pod-spec half, extractPortsFromPod :1195-1246, is the
// caller's: Pod::container_ports already holds "port/protocol" strings)
std::vector<std::string> GetRequestedPorts(const Pod& pod) {
    auto it = pod.annotations.find(PortsAnnotation);
    if (it != pod.annotations.end() && !it->second.empty()) {
        std::vector<std::string> out;
        size_t start = 0;
        while (true) {
            size_t comma = it->second.find(',', start);
            out.push_back(TrimSpace(it->second.substr(start, comma == std::string::npos ? std::string::npos : comma - start)));
            if (comma == std::string::npos) break;
            start = comma + 1;
        }
        return out;
    }
    return pod.container_ports;
}

static bool HasSuffix(const std::string& s, const char* suf) {
    size_t n = std::strlen(suf);
    return s.size() >= n && s.compare(s.size() - n, n, suf) == 0;
}

// checkPortsExposed -- kubelet.go:566-605
bool CheckPortsExposed(const std::map<std::string, int>& port_mappings, const std::vector<std::string>& requested) {
    if (requested.empty()) return true;
    for (const auto& rp : requested) {
        bool found = false;
        for (const auto& kv : port_mappings)
            if (rp == kv.first + "/tcp" || rp == kv.first + "/http") { found = true; break; }
        if (found) continue;
        if (HasSuffix(rp, "/http")) continue;  // RunPod proxies HTTP ports; assumed available
        return false;                          // a TCP port must be in portMappings
    }
    return true;
}

static std::string ToLower(std::string s) {
    for (auto& c : s) c = (char)std::tolower((unsigned char)c);
    return s;
}

bool MessageHasError(const std::string& message) {  // kubelet.go:1907-1908
    const std::string low = ToLower(message);
    return low.find("error") != std::string::npos || low.find("fail") != std::string::npos;
}

// translateRunPodStatus -- kubelet.go:1848-2024: RunPod status (+ ports bit, + message) -> phase,
// readiness, container state.  Pure table; this string form serves GetPodStatus and the sweep's host-side
// fallback, the sweep itself uses StatusFromCode on the code the kernel emits for the CHANGED subset.
PodStatusView TranslateRunPodStatus(const std::string& status, const std::string& message, bool has_exposed_ports) {
    PodStatusView v;
    v.phase = "Unknown";
    v.message = message;
    if (status == PodRunning) {
        if (has_exposed_ports) {
            v.phase = "Running"; v.state = "Running"; v.started = true;
        } else {
            v.phase = "Pending"; v.state = "Waiting"; v.reason = "ContainerCreating";
            v.container_message = "Container reported as running but ports not yet exposed";  // :1885
        }
    } else if (status == PodStarting) {
        v.phase = "Pending"; v.state = "Waiting"; v.reason = "ContainerCreating"; v.container_message = message;
    } else if (status == PodExited) {
        v.state = "Terminated"; v.container_message = message;
        if (MessageHasError(message)) { v.exit_code = 1; v.reason = "Error"; v.phase = "Failed"; }
        else { v.exit_code = 0; v.reason = "Completed"; v.phase = "Succeeded"; }
    } else if (status == PodTerminating) {
        v.phase = "Running"; v.state = "Running"; v.started = true;
    } else if (status == PodTerminated) {
        v.phase = "Succeeded"; v.state = "Terminated"; v.reason = "Terminated"; v.exit_code = 0; v.container_message = message;
    } else if (status == PodNotFound) {
        v.phase = "Failed"; v.state = "Terminated"; v.reason = "PodDeleted"; v.exit_code = 1;
        v.container_message = "Pod was deleted from RunPod API";  // :1963
    } else {
        v.state = "Waiting"; v.reason = "ContainerStatusUnknown";
        v.container_message = "Unknown RunPod status: " + status;  // :1975
    }
    // readyCondition: True iff phase == Running (kubelet.go:1982-1985) -- the same set as containerStatus.Ready
    v.ready = v.phase == "Running";
    return v;
}

// the same decision read off the kernel's code (include/rpk.h RPK_CODE_*)
PodStatusView StatusFromCode(uint16_t code, const std::string& status, const std::string& message) {
    static const char* const kPhase[] = {"Unknown", "Pending", "Running", "Succeeded", "Failed", "Unknown", "Unknown", "Unknown"};
    static const char* const kState[] = {"Waiting", "Running", "Terminated", "Waiting"};
    static const char* const kReason[] = {"", "ContainerCreating", "Completed", "Error", "Terminated", "PodDeleted", "ContainerStatusUnknown", ""};
    PodStatusView v;
    v.phase = kPhase[RPK_CODE_PHASE(code)];
    v.ready = RPK_CODE_READY(code) != 0; v.started = RPK_CODE_STARTED(code) != 0;
    v.state = kState[RPK_CODE_STATE(code)];
    v.exit_code = (int)RPK_CODE_EXIT(code);
    v.reason = kReason[RPK_CODE_REASON(code)];
    v.message = message;
    switch (RPK_CODE_MESSAGE(code)) {
        case 1: v.container_message = "Container reported as running but ports not yet exposed"; break;
        case 2: v.container_message = "Pod was deleted from RunPod API"; break;
        case 3: v.container_message = "Unknown RunPod status: " + status; break;
        default: v.container_message = v.state == "Running" ? "" : message; break;  // ContainerStateRunning has no message
    }
    return v;
}

// canonical slot [len | flag << 7][status][0x00][ports][pad] (include/rpk.h)
bool EncodeStatusRecord(uint8_t* slot, uint32_t stride, const std::string& status, bool ports_exposed, bool message_has_error) {
    if (status.size() + 2 > stride - 1 || status.size() + 2 > 127) return false;
    std::memset(slot, 0, stride);
    slot[0] = (uint8_t)((status.size() + 2) | (message_has_error ? 0x80u : 0u));
    std::memcpy(slot + 1, status.data(), status.size());
    slot[1 + status.size() + 1] = ports_exposed ? 1 : 0;
    return true;
}

static int32_t ClampI32(long long v) { return v > INT32_MAX ? INT32_MAX : v < INT32_MIN ? INT32_MIN : (int32_t)v; }

// The annotation half of PrepareRunPodParameters (runpod_client.go:1255-1281): annotations (pod, then
// owner Job) -> the row of the grid.  Absent extension annotations reproduce the reference exactly
// (maxPrice = DefaultMaxPrice, vcpu = ram = 0).
//
// This is the caller side of the grid and, at the batch sizes the kernels are built for, the expensive side
// (host_test --bench-columns), so the row producer does getAnnotationWithFallback without its copies: keys
// are built once, lookups return pointers, and the two valid cloud spellings are recognised before the
// general upper-casing path.  host_test checks it row for row against the composition of the public,
// reference-shaped functions (GetAnnotationWithFallback / ValidateCloudType / ExtractGPUMemory).
namespace {
const std::string kKeyCloud = CloudTypeAnnotation, kKeyMem = GpuMemoryAnnotation, kKeyVcpu = VcpuAnnotation,
                  kKeyRam = RamAnnotation, kKeyMaxPrice = MaxPriceAnnotation, kKeyGpuTypes = GpuTypeIdsAnnotation;

// The six annotations the row reads.  One pass over the pod's annotation map (and one over the owner Job's, if a
// slot is still open) classifies each key by length + full compare, instead of five string-keyed tree searches
// per map: per key the result is getAnnotationWithFallback's (:1102-1112) -- the pod's non-empty value, else the
// Job's non-empty value, else nullptr (= the default).
enum Slot { kSlotCloud, kSlotMem, kSlotVcpu, kSlotRam, kSlotMaxPrice, kSlotGpuTypes, kSlots };
constexpr size_t CLen(const char* s) { size_t n = 0; while (s[n]) ++n; return n; }
static_assert(CLen(CloudTypeAnnotation) == 20 && CLen(GpuMemoryAnnotation) == 29 && CLen(VcpuAnnotation) == 23 &&
              CLen(RamAnnotation) == 25 && CLen(MaxPriceAnnotation) == 26 && CLen(GpuTypeIdsAnnotation) == 22,
              "ClassifyKey switches on these lengths");

inline int ClassifyKey(const std::string& k) {
    const std::string* want = nullptr;
    int slot = kSlots;
    switch (k.size()) {  // the six keys have six different lengths
        case 20: want = &kKeyCloud; slot = kSlotCloud; break;      // runpod.io/cloud-type  (runpod.io/templateId is 20 too)
        case 29: want = &kKeyMem; slot = kSlotMem; break;          // runpod.io/required-gpu-memory
        case 23: want = &kKeyVcpu; slot = kSlotVcpu; break;        // runpod.io/required-vcpu
        case 25: want = &kKeyRam; slot = kSlotRam; break;          // runpod.io/required-ram-gb
        case 26: want = &kKeyMaxPrice; slot = kSlotMaxPrice; break;  // runpod.io/max-price-per-hr
        case 22: want = &kKeyGpuTypes; slot = kSlotGpuTypes; break;  // runpod.io/gpu-type-ids
        default: return kSlots;
    }
    return k == *want ? slot : (int)kSlots;
}

inline void CollectAnnotations(const Pod& pod, const std::string* (&v)[kSlots]) {
    for (int i = 0; i < kSlots; ++i) v[i] = nullptr;
    for (const auto& kv : pod.annotations) {
        const int s = ClassifyKey(kv.first);
        if (s != kSlots && !kv.second.empty()) v[s] = &kv.second;
    }
    if (!pod.owner_job) return;
    for (const auto& kv : *pod.owner_job) {
        const int s = ClassifyKey(kv.first);
        if (s != kSlots && v[s] == nullptr && !kv.second.empty()) v[s] = &kv.second;
    }
}

struct Row { int32_t mem, vcpu, ram; double max_price; uint8_t cloud; const std::string* gpu_types; };

Row PrepareRow(const Pod& pod) {
    const std::string* a[kSlots];
    CollectAnnotations(pod, a);
    Row r;
    const std::string* v = a[kSlotCloud];
    if (!v || *v == "SECURE") r.cloud = RPK_CLOUD_SECURE;
    else if (*v == "COMMUNITY") r.cloud = RPK_CLOUD_COMMUNITY;
    else r.cloud = ValidateCloudType(*v) == "COMMUNITY" ? RPK_CLOUD_COMMUNITY : RPK_CLOUD_SECURE;
    v = a[kSlotMem];
    r.mem = ClampI32(v ? ExtractGPUMemory(*v) : 16);  // extractGPUMemory(""): 16 (:1182)
    long long x = 0;
    v = a[kSlotVcpu];
    r.vcpu = v && GoAtoi(*v, &x) ? ClampI32(x) : 0;
    v = a[kSlotRam];
    r.ram = v && GoAtoi(*v, &x) ? ClampI32(x) : 0;
    r.max_price = DefaultMaxPrice;
    v = a[kSlotMaxPrice];
    if (v) {
        char* end = nullptr;
        errno = 0;
        const double d = std::strtod(v->c_str(), &end);
        if (errno == 0 && end && *end == '\0' && end != v->c_str()) r.max_price = d;
    }
    r.gpu_types = a[kSlotGpuTypes];  // nullptr: unrestricted
    return r;
}
}  // namespace

PodColumns PrepareColumns(const Pod& pod) {
    const Row r = PrepareRow(pod);
    PodColumns c;
    c.req_mem_gb = r.mem; c.req_vcpu = r.vcpu; c.req_ram_gb = r.ram; c.max_price = r.max_price; c.cloud = r.cloud;
    c.cloud_type = r.cloud == RPK_CLOUD_COMMUNITY ? "COMMUNITY" : "SECURE";
    c.restricted = r.gpu_types != nullptr;
    if (r.gpu_types) c.gpu_type_ids = ParseGpuTypeIds(*r.gpu_types);
    return c;
}

void PrepareColumnsBatch(const std::vector<PodPtr>& pods, PodColumnsSoA* out, int n_threads) {
    const size_t P = pods.size();
    out->resize(P);
    auto run = [&](size_t lo, size_t hi) {
        for (size_t i = lo; i < hi; ++i) {
            const Row r = PrepareRow(*pods[i]);
            out->req_mem_gb[i] = r.mem; out->req_vcpu[i] = r.vcpu; out->req_ram_gb[i] = r.ram;
            out->max_price[i] = r.max_price; out->cloud[i] = r.cloud;
            if (r.gpu_types) out->gpu_type_ids[i] = *r.gpu_types;
        }
    };
    constexpr size_t kMinRowsPerThread = 4096;  // below this a thread costs more to start than it saves
    size_t t = n_threads > 0 ? (size_t)n_threads : (size_t)std::max(1u, std::thread::hardware_concurrency());
    t = std::min(t, std::max<size_t>(1, P / kMinRowsPerThread));
    if (t <= 1) { run(0, P); return; }
    std::vector<std::thread> th;
    th.reserve(t - 1);
    for (size_t k = 1; k < t; ++k) th.emplace_back(run, P * k / t, P * (k + 1) / t);
    run(0, P / t);
    for (auto& x : th) x.join();
}

// ---------------------------------------------------------------------------------------------------------
// Provider
// ---------------------------------------------------------------------------------------------------------
static uint32_t StrideFor(size_t status_len) {  // smallest slot that holds [len][status][0][ports]
    for (uint32_t st = 16; st <= 256; st <<= 1) if (status_len + 2 <= st - 1 && status_len + 2 <= 127) return st;
    return 0;  // longer than any slot: compared on the host
}

Provider::Provider(std::shared_ptr<RunPodAPI> api, int n_gpus, uint32_t max_pods, ProviderOptions opt)
    : api_(std::move(api)), max_pods_(max_pods), opt_(opt) {
    int rc = rpk_create(n_gpus, nullptr, &ctx_);
    if (rc != RPK_OK) throw std::runtime_error(std::string("rpk engine unavailable (no CPU fallback): ") + rpk_last_error(nullptr));
    records_.assign((size_t)max_pods_ * stride_, 0);
    slot_key_.assign(max_pods_, "");
    for (uint32_t s = max_pods_; s > 0; --s) free_slots_.push_back(s - 1);
    if (rpk_status_reset(ctx_, max_pods_) != RPK_OK) throw std::runtime_error(rpk_last_error(ctx_));
    // empty slots hold the all-zero record from now on: seed it so they never report
    if (rpk_status_seed(ctx_, max_pods_, records_.data(), stride_) != RPK_OK) throw std::runtime_error(rpk_last_error(ctx_));
    if (opt_.self_tick) {  // go provider.startPeriodicStatusUpdates(); go provider.startPendingPodProcessor() -- kubelet.go:374-376
        StartTicker(opt_.periodic_interval_s, [this] { UpdateAllPodStatuses(); });
        StartTicker(opt_.pending_interval_s, [this] { ProcessPendingPods(); });
    }
}

Provider::~Provider() {
    StopTickers();
    rpk_destroy(ctx_);
}

void Provider::StartTicker(double interval_s, std::function<void()> body) {
    tickers_.emplace_back([this, interval_s, body]() {
        std::unique_lock<std::mutex> lk(tick_mutex_);
        for (;;) {
            if (tick_cv_.wait_for(lk, std::chrono::duration<double>(interval_s), [this] { return tick_stop_; })) return;
            lk.unlock();
            try { body(); } catch (...) { /* a failed tick must not kill the ticker (the reference logs and goes on) */ }
            lk.lock();
        }
    });
}

void Provider::StopTickers() {
    { std::lock_guard<std::mutex> g(tick_mutex_); tick_stop_ = true; }
    tick_cv_.notify_all();
    for (auto& t : tickers_) if (t.joinable()) t.join();
    tickers_.clear();
}

uint32_t Provider::AllocSlot() {
    if (free_slots_.empty()) throw std::runtime_error("provider pod capacity exceeded");
    uint32_t s = free_slots_.back();
    free_slots_.pop_back();
    return s;
}

void Provider::Notify(const PodPtr& pod) {
    std::function<void(const PodPtr&)> cb;
    { std::lock_guard<std::mutex> g(notify_mutex_); cb = notify_; }
    if (!cb) return;
    try { cb(pod); } catch (...) { /* recover(): kubelet.go:938-946 */ }
}

// The device's previous state of ONE slot := what InstanceInfo says now.  The reference rewrites one map entry
// (kubelet.go:391-401, 976-1040); re-seeding the whole table here would silently adopt every other pod's pending
// change as "previous" and lose its notification.
void Provider::SeedSlot(uint32_t slot) {
    uint8_t rec[256];
    uint32_t stride;
    { std::lock_guard<std::mutex> g(pods_mutex_); stride = stride_; std::memcpy(rec, &records_[(size_t)slot * stride], stride); }
    std::lock_guard<std::mutex> g(engine_mutex_);
    rpk_status_seed_slots(ctx_, 1, &slot, rec, stride);
}

// CreatePod -- kubelet.go:384-418.  Tracks the pod (InstanceInfo{STARTING, ports not exposed}) and tries to
// deploy; a failed deploy is swallowed (returns nil) so that ProcessPendingPods retries it.
std::string Provider::CreatePod(const PodPtr& pod) {
    const std::string key = Key(pod->ns, pod->name);
    uint32_t slot;
    {
        std::lock_guard<std::mutex> g(pods_mutex_);
        auto it = pods_.find(key);
        Tracked t;
        t.slot = it != pods_.end() ? it->second.slot : AllocSlot();
        t.pod = std::make_shared<Pod>(*pod);  // DeepCopy
        t.info.PodName = pod->name; t.info.Namespace = pod->ns; t.info.Status = PodStarting;
        t.info.CreationTime = now_; t.info.RequestedPorts = GetRequestedPorts(*pod); t.info.PortsExposed = false;
        slot_key_[t.slot] = key;
        EncodeStatusRecord(&records_[(size_t)t.slot * stride_], stride_, t.info.Status, t.info.PortsExposed);
        slot = t.slot;
        pods_[key] = std::move(t);
    }
    SeedSlot(slot);  // previous state for the sweep = what InstanceInfo says now, for this slot only
    DeployBatch({key});  // errors are logged and swallowed: kubelet.go:406-415
    return "";
}

// UpdatePod -- kubelet.go:421-432
std::string Provider::UpdatePod(const PodPtr& pod) {
    std::lock_guard<std::mutex> g(pods_mutex_);
    auto it = pods_.find(Key(pod->ns, pod->name));
    if (it == pods_.end()) {  // the reference inserts into p.pods without an InstanceInfo; mirror the visible part
        Tracked t;
        t.slot = AllocSlot();
        t.pod = std::make_shared<Pod>(*pod);
        slot_key_[t.slot] = Key(pod->ns, pod->name);
        pods_[Key(pod->ns, pod->name)] = std::move(t);
    } else {
        it->second.pod = std::make_shared<Pod>(*pod);
    }
    return "";
}

// DeletePod -- kubelet.go:621-651
std::string Provider::DeletePod(const PodPtr& pod) {
    auto it = pod->annotations.find(PodIDAnnotation);
    if (it != pod->annotations.end() && !it->second.empty()) {
        { std::lock_guard<std::mutex> g(deleted_mutex_); deleted_pods_[pod->ns + "/" + pod->name] = it->second; }
        std::string err;
        api_->TerminatePod(it->second, &err);  // failure is only logged
    }
    std::lock_guard<std::mutex> g(pods_mutex_);
    auto pt = pods_.find(Key(pod->ns, pod->name));
    if (pt != pods_.end()) {
        const uint32_t s = pt->second.slot;
        std::memset(&records_[(size_t)s * stride_], 0, stride_);
        slot_key_[s].clear();
        free_slots_.push_back(s);
        pods_.erase(pt);
    }
    return "";
}

// GetPod -- kubelet.go:654-667
std::pair<PodPtr, std::string> Provider::GetPod(const std::string& ns, const std::string& name) {
    const std::string key = Key(ns, name);
    std::lock_guard<std::mutex> g(pods_mutex_);
    auto it = pods_.find(key);
    if (it == pods_.end()) return {nullptr, "pod " + key + " not found"};
    return {it->second.pod, ""};
}

// GetPodStatus -- kubelet.go:670-696 (live port check for RUNNING pods with requested ports)
std::pair<PodStatusView, std::string> Provider::GetPodStatus(const std::string& ns, const std::string& name) {
    const std::string key = Key(ns, name);
    InstanceInfo info;
    PodPtr pod;
    {
        std::lock_guard<std::mutex> g(pods_mutex_);
        auto it = pods_.find(key);
        if (it == pods_.end()) return {PodStatusView{}, "pod status not found for " + key};
        info = it->second.info; pod = it->second.pod;
    }
    bool has_ports = true;
    if (info.Status == PodRunning && !info.RequestedPorts.empty() && pod) {
        auto a = pod->annotations.find(PodIDAnnotation);
        if (a != pod->annotations.end() && !a->second.empty()) {
            DetailedStatus ds; std::string err;
            if (api_->GetDetailedPodStatus(a->second, &ds, &err)) has_ports = CheckPortsExposed(ds.PortMappings, info.RequestedPorts);
        }
    }
    return {TranslateRunPodStatus(info.Status, info.StatusMessage, has_ports), ""};
}

// GetPods -- kubelet.go:699-710
std::vector<PodPtr> Provider::GetPods() {
    std::lock_guard<std::mutex> g(pods_mutex_);
    std::vector<PodPtr> out;
    out.reserve(pods_.size());
    for (auto& kv : pods_) out.push_back(kv.second.pod);
    return out;
}

// NotifyPods -- kubelet.go:713-731: install the callback, return immediately, sweep every 10 s from a thread of our own
void Provider::NotifyPods(std::function<void(const PodPtr&)> cb) {
    { std::lock_guard<std::mutex> g(notify_mutex_); notify_ = std::move(cb); }
    if (!opt_.self_tick) return;
    std::lock_guard<std::mutex> g(tick_mutex_);
    if (notify_ticker_started_) return;  // a second NotifyPods replaces the callback, not the ticker
    notify_ticker_started_ = true;
    StartTicker(opt_.notify_interval_s, [this] { UpdateAllPodStatuses(); });
}

const InstanceInfo* Provider::Info(const std::string& ns, const std::string& name) {
    std::lock_guard<std::mutex> g(pods_mutex_);
    auto it = pods_.find(Key(ns, name));
    return it == pods_.end() ? nullptr : &it->second.info;
}

// Offer table refresh: ONE fetch per tick (the reference re-fetches per pod, runpod_client.go:447-455),
// uploaded only when it differs from the resident table.
bool Provider::RefreshOffersLocked(std::string* err) {
    std::vector<GPUType> fresh;
    if (!api_->FetchGPUTypes(&fresh, err)) return false;
    bool same = fresh.size() == offers_.size();
    for (size_t i = 0; same && i < fresh.size(); ++i) {
        const GPUType &a = fresh[i], &b = offers_[i];
        same = a.ID == b.ID && a.MemoryInGb == b.MemoryInGb && a.SecureCloud == b.SecureCloud && a.SecurePrice == b.SecurePrice &&
               a.CommunityCloud == b.CommunityCloud && a.CommunityPrice == b.CommunityPrice && a.VCPU == b.VCPU && a.RAMGb == b.RAMGb;
    }
    if (same && offer_uploads_ > 0) return true;
    const uint32_t G = (uint32_t)fresh.size();
    std::vector<int32_t> mem(G), vcpu(G), ram(G);
    std::vector<double> sp(G), cp(G);
    std::vector<uint8_t> flags(G);
    for (uint32_t i = 0; i < G; ++i) {
        mem[i] = fresh[i].MemoryInGb; vcpu[i] = fresh[i].VCPU; ram[i] = fresh[i].RAMGb;
        sp[i] = fresh[i].SecurePrice; cp[i] = fresh[i].CommunityPrice;
        flags[i] = (uint8_t)((fresh[i].SecureCloud ? RPK_FLAG_SECURE_CLOUD : 0) | (fresh[i].CommunityCloud ? RPK_FLAG_COMMUNITY_CLOUD : 0));
    }
    if (rpk_offers_upload(ctx_, G, mem.data(), vcpu.data(), ram.data(), sp.data(), cp.data(), flags.data()) != RPK_OK) {
        *err = rpk_last_error(ctx_);
        return false;
    }
    offers_ = std::move(fresh);
    ++offer_uploads_;
    return true;
}

// DeployPodToRunPod for a batch (kubelet.go:435-503 + runpod_client.go:1250-1343): columns from
// annotations -> ONE rpk_select over the whole batch -> gpuTypeIds per pod -> DeployPod -> annotations.
bool Provider::DeployBatch(const std::vector<std::string>& keys) {
    std::vector<PodPtr> pods;
    std::vector<std::string> live;
    {
        std::lock_guard<std::mutex> g(pods_mutex_);
        for (const auto& k : keys) {
            auto it = pods_.find(k);
            if (it != pods_.end() && it->second.pod) { pods.push_back(it->second.pod); live.push_back(k); }
        }
    }
    if (pods.empty()) return true;
    std::string err;
    const uint32_t P = (uint32_t)pods.size();
    PodColumnsSoA cols;
    PrepareColumnsBatch(pods, &cols);  // the whole batch's annotations -> columns, over the host threads
    std::vector<int32_t> best(P), top5((size_t)P * RPK_TOPK);
    std::vector<std::vector<std::string>> gpu_type_ids(P);  // params["gpuTypeIds"], runpod_client.go:1339
    {   // table refresh, selection and index -> id lookup under ONE lock: another thread's refresh cannot swap the table
        // between the select and the lookup (indices would resolve against a different, possibly shorter, table)
        std::lock_guard<std::mutex> g(engine_mutex_);
        if (!RefreshOffersLocked(&err)) return false;  // "failed to get GPU types": every pod of the batch retries later
        bool restricted = false;
        for (uint32_t i = 0; i < P && !restricted; ++i) restricted = !cols.gpu_type_ids[i].empty();
        if (!restricted) {  // no pod carries runpod.io/gpu-type-ids: the plain selection, exactly as without the annotation
            if (rpk_select(ctx_, P, cols.req_mem_gb.data(), cols.req_vcpu.data(), cols.req_ram_gb.data(), cols.max_price.data(),
                           cols.cloud.data(), best.data(), top5.data()) != RPK_OK) return false;
            ++select_calls_;
        } else if (!SelectWithSetsLocked(cols, top5.data()) && !(set_lists_.empty() && SelectWithSetsLocked(cols, top5.data(), false))) {
            return false;  // a failed reuse forgets the resident sets and uploads once more; a second failure retries next tick
        }
        for (uint32_t i = 0; i < P; ++i)
            for (int k = 0; k < RPK_TOPK; ++k) {
                const int32_t g = top5[(size_t)i * RPK_TOPK + k];
                if (g >= 0 && (size_t)g < offers_.size()) gpu_type_ids[i].push_back(offers_[(size_t)g].ID);
            }
    }
    bool all_ok = true;
    for (uint32_t i = 0; i < P; ++i) {
        const std::vector<std::string>& ids = gpu_type_ids[i];
        std::string id; double cost = 0;
        if (!api_->DeployPod(*pods[i], ids, cols.req_mem_gb[i], cols.cloud[i] == RPK_CLOUD_COMMUNITY ? "COMMUNITY" : "SECURE", &id, &cost, &err)) { all_ok = false; continue; }
        // updatePodWithRunPodInfo -- kubelet.go:505-562
        std::lock_guard<std::mutex> g(pods_mutex_);
        auto it = pods_.find(live[i]);
        if (it == pods_.end()) continue;
        auto np = std::make_shared<Pod>(*it->second.pod);
        np->annotations[PodIDAnnotation] = id;
        char buf[64]; snprintf(buf, sizeof(buf), "%f", cost);
        np->annotations[CostAnnotation] = buf;
        it->second.pod = np;
        it->second.info.ID = id; it->second.info.CostPerHr = cost;
    }
    return all_ok;
}

// A batch with runpod.io/gpu-type-ids: every distinct list, taken as a set of ids, becomes an offer set (ids absent from
// the table are ignored, so a list that matches nothing is an empty set and its pods get an empty gpuTypeIds -- "no
// eligible GPU types", retried like any other).  The resident sets are reused while the table is unchanged and hold
// every list of the batch; otherwise the batch's lists are uploaded, RPK_MAX_OFFER_SETS at a time, each group with one
// rpk_select_sets over its rows (the unrestricted rows go with the first group).  set_lists_ only names sets the engine
// holds: it is cleared before an upload (a failed upload leaves none behind) and after a failed select on reused sets.
bool Provider::SelectWithSetsLocked(const PodColumnsSoA& cols, int32_t* top5, bool may_reuse) {
    const uint32_t P = (uint32_t)cols.size();
    std::map<std::vector<std::string>, uint32_t> list_of;  // canonical list (sorted, unique ids) -> index in `lists`
    std::vector<std::vector<std::string>> lists;
    std::vector<uint32_t> row_list(P, UINT32_MAX);          // UINT32_MAX = unrestricted
    for (uint32_t i = 0; i < P; ++i) {
        if (cols.gpu_type_ids[i].empty()) continue;
        std::vector<std::string> ids = ParseGpuTypeIds(cols.gpu_type_ids[i]);
        std::sort(ids.begin(), ids.end());
        ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
        auto it = list_of.emplace(std::move(ids), (uint32_t)lists.size());
        if (it.second) lists.push_back(it.first->first);
        row_list[i] = it.first->second;
    }
    std::map<std::string, uint32_t> index_of;  // GPU type id -> table index
    for (uint32_t g = 0; g < (uint32_t)offers_.size(); ++g) index_of.emplace(offers_[g].ID, g);
    const uint32_t G = (uint32_t)offers_.size(), W = (G + 31) / 32;
    auto upload = [&](const std::vector<std::vector<std::string>>& group) {
        std::vector<uint32_t> words((size_t)group.size() * W, 0u);
        for (size_t s = 0; s < group.size(); ++s)
            for (const auto& id : group[s]) {
                auto f = index_of.find(id);
                if (f != index_of.end()) words[s * W + f->second / 32] |= 1u << (f->second & 31);
            }
        set_lists_.clear();
        if (rpk_offer_sets_upload(ctx_, (uint32_t)group.size(), G, words.empty() ? nullptr : words.data()) != RPK_OK) return false;
        ++set_uploads_;
        set_lists_ = group;
        set_table_ = offer_uploads_;
        return true;
    };
    // reuse the resident sets when they were built on this table and hold every list of the batch
    std::vector<uint32_t> resident_id(lists.size(), UINT32_MAX);
    bool reuse = may_reuse && set_table_ == offer_uploads_ && !set_lists_.empty();
    for (size_t l = 0; reuse && l < lists.size(); ++l) {
        auto f = std::find(set_lists_.begin(), set_lists_.end(), lists[l]);
        if (f == set_lists_.end()) reuse = false; else resident_id[l] = (uint32_t)(f - set_lists_.begin());
    }
    const size_t n_groups = reuse ? 1 : (lists.size() + RPK_MAX_OFFER_SETS - 1) / RPK_MAX_OFFER_SETS;
    PodColumnsSoA sub;
    std::vector<uint16_t> set_id;
    std::vector<int32_t> best, t5;
    std::vector<uint32_t> rows;
    for (size_t grp = 0; grp < n_groups; ++grp) {
        const size_t l0 = grp * RPK_MAX_OFFER_SETS, l1 = std::min(lists.size(), l0 + RPK_MAX_OFFER_SETS);
        if (!reuse && !upload(std::vector<std::vector<std::string>>(lists.begin() + (long)l0, lists.begin() + (long)l1))) return false;
        rows.clear();
        for (uint32_t i = 0; i < P; ++i)
            if (row_list[i] == UINT32_MAX ? grp == 0 : (row_list[i] >= l0 && row_list[i] < l1)) rows.push_back(i);
        const uint32_t n = (uint32_t)rows.size();
        if (n == 0) continue;
        sub.resize(n); set_id.resize(n); best.resize(n); t5.resize((size_t)n * RPK_TOPK);
        for (uint32_t j = 0; j < n; ++j) {
            const uint32_t i = rows[j];
            sub.req_mem_gb[j] = cols.req_mem_gb[i]; sub.req_vcpu[j] = cols.req_vcpu[i]; sub.req_ram_gb[j] = cols.req_ram_gb[i];
            sub.max_price[j] = cols.max_price[i]; sub.cloud[j] = cols.cloud[i];
            set_id[j] = row_list[i] == UINT32_MAX ? (uint16_t)RPK_SET_ALL
                                                  : (uint16_t)(reuse ? resident_id[row_list[i]] : row_list[i] - (uint32_t)l0);
        }
        if (rpk_select_sets(ctx_, n, sub.req_mem_gb.data(), sub.req_vcpu.data(), sub.req_ram_gb.data(), sub.max_price.data(),
                            sub.cloud.data(), set_id.data(), best.data(), t5.data()) != RPK_OK) {
            if (reuse) set_lists_.clear();  // the engine no longer holds them (e.g. its table was replaced)
            return false;
        }
        ++set_select_calls_;
        for (uint32_t j = 0; j < n; ++j) std::memcpy(top5 + (size_t)rows[j] * RPK_TOPK, t5.data() + (size_t)j * RPK_TOPK, RPK_TOPK * sizeof(int32_t));
    }
    return true;
}

// processPendingPods -- kubelet.go:747-814: every tracked pod that is Pending and has no RunPod id is
// (re)deployed; after 15 minutes of failures it is marked Failed and pushed through notifyFunc.
void Provider::ProcessPendingPods() {
    std::vector<std::string> keys;
    {
        std::lock_guard<std::mutex> g(pods_mutex_);
        for (auto& kv : pods_) {
            const Pod& p = *kv.second.pod;
            if (p.status.phase != "Pending") continue;                                  // :753
            auto a = p.annotations.find(PodIDAnnotation);
            if (a != p.annotations.end() && !a->second.empty()) continue;              // :769-775
            keys.push_back(kv.first);
        }
    }
    if (keys.empty()) return;
    DeployBatch(keys);
    for (const auto& k : keys) {  // give up after 15 minutes (:786-810)
        PodPtr failed;
        {
            std::lock_guard<std::mutex> g(pods_mutex_);
            auto it = pods_.find(k);
            if (it == pods_.end()) continue;
            auto a = it->second.pod->annotations.find(PodIDAnnotation);
            if (a != it->second.pod->annotations.end() && !a->second.empty()) continue;  // deployed now
            if (now_ - it->second.info.CreationTime <= 15 * 60) continue;
            auto np = std::make_shared<Pod>(*it->second.pod);
            np->status.phase = "Failed"; np->status.reason = "RunPodDeploymentFailed";
            np->status.message = "Failed to deploy pod to RunPod after multiple attempts";
            it->second.pod = np;
            failed = np;
        }
        Notify(failed);
    }
}

// Re-encode every tracked slot at a wider stride (a status string longer than the slot appeared).  Called with
// sweep_mutex_ held, before a sweep starts, so no staged sweep can be absorbed by the whole-table seed.
void Provider::WidenRecords(uint32_t stride) {
    std::vector<uint8_t> fresh;
    {
        std::lock_guard<std::mutex> g(pods_mutex_);
        fresh.assign((size_t)max_pods_ * stride, 0);
        for (auto& kv : pods_) {
            const Tracked& t = kv.second;
            if (!t.info.PodName.empty() || !t.info.Status.empty())
                EncodeStatusRecord(&fresh[(size_t)t.slot * stride], stride, t.info.Status, t.info.PortsExposed, MessageHasError(t.info.StatusMessage));
        }
        records_ = fresh; stride_ = stride;
    }
    std::lock_guard<std::mutex> g(engine_mutex_);
    rpk_status_seed(ctx_, max_pods_, fresh.data(), stride);
}

// updateAllPodStatuses -- kubelet.go:816-974.  The per-pod fetches stay sequential host I/O (out of scope);
// the compare of (status, portsExposed) against InstanceInfo for ALL tracked slots is one rpk_status_diff_codes,
// which also returns translateRunPodStatus's decision for every changed slot.
//
// Concurrency (the reference reaches this from two tickers while CreatePod / DeletePod run on other goroutines):
// fresh records are staged in a buffer private to the sweep -- a copy of records_ (what InstanceInfo says) with this
// sweep's fetches on top -- and records_ / InstanceInfo are updated per changed slot afterwards, under pods_mutex_,
// only if the slot still belongs to the pod the sweep fetched.  A changed slot whose update is not applied (the pod
// was created, deleted or re-created meanwhile) gets its device state re-seeded from records_, so device and host
// cannot drift apart.
void Provider::UpdateAllPodStatuses() {
    std::lock_guard<std::mutex> sweep_guard(sweep_mutex_);
    if (want_stride_ > stride_) WidenRecords(want_stride_);
    struct Fresh { std::string key, status, message; bool ports; uint32_t slot; bool host_compare; };
    std::vector<Fresh> fresh;
    std::vector<std::string> keys;
    std::vector<uint8_t> staged;
    uint32_t stride;
    {
        std::lock_guard<std::mutex> g(pods_mutex_);
        for (auto& kv : pods_) keys.push_back(kv.first);  // :818-823
        staged = records_;
        stride = stride_;
    }
    for (const auto& key : keys) {
        PodPtr pod; InstanceInfo info; uint32_t slot;
        {
            std::lock_guard<std::mutex> g(pods_mutex_);
            auto it = pods_.find(key);
            if (it == pods_.end() || !it->second.pod) continue;
            pod = it->second.pod; info = it->second.info; slot = it->second.slot;
        }
        if (pod->status.phase == "Succeeded" || pod->status.phase == "Failed") continue;  // :836
        auto a = pod->annotations.find(PodIDAnnotation);
        if (a == pod->annotations.end() || a->second.empty()) continue;                   // :841-844
        DetailedStatus ds; std::string err;
        if (!api_->GetDetailedPodStatus(a->second, &ds, &err)) continue;                  // :848-855 skip this cycle
        if (ds.DesiredStatus == PodNotFound) {                                            // :861-864 handleMissingRunPodInstance
            PodPtr np;
            {
                std::lock_guard<std::mutex> g(pods_mutex_);
                auto it = pods_.find(key);
                if (it == pods_.end() || it->second.slot != slot) continue;
                np = std::make_shared<Pod>(*it->second.pod);
                np->annotations.erase(PodIDAnnotation); np->annotations.erase(CostAnnotation);
                np->status = TranslateRunPodStatus(PodNotFound, "RunPod instance was deleted", true);
                it->second.pod = np;
                it->second.info.ID.clear(); it->second.info.Status = PodExited; it->second.info.StatusMessage = "RunPod instance not found";
                EncodeStatusRecord(&records_[(size_t)slot * stride_], stride_, it->second.info.Status, it->second.info.PortsExposed);
                if (stride_ == stride) std::memcpy(&staged[(size_t)slot * stride], &records_[(size_t)slot * stride], stride);
            }
            SeedSlot(slot);  // InstanceInfo was rewritten: so is the previous state -- of this slot, nothing else
            Notify(np);
            continue;
        }
        const bool ports = CheckPortsExposed(ds.PortMappings, info.RequestedPorts);         // :867
        Fresh f{key, ds.DesiredStatus, info.StatusMessage, ports, slot, false};
        if (!EncodeStatusRecord(&staged[(size_t)slot * stride], stride, ds.DesiredStatus, ports, MessageHasError(info.StatusMessage))) {
            // does not fit this table's slots: compare it the way the reference does (:870-873) this cycle, and widen
            // the table before the next sweep if any slot size can hold it
            f.host_compare = true;
            const uint32_t need = StrideFor(ds.DesiredStatus.size());
            if (need > want_stride_) want_stride_ = need;
        }
        fresh.push_back(std::move(f));
    }
    // ---- the diff: statusChanged || portsExposureChanged for every slot at once (:870-873) + the decision per changed slot ----
    std::vector<uint32_t> changed(max_pods_);
    std::vector<uint16_t> codes(max_pods_);
    uint32_t n_changed = 0;
    {
        std::lock_guard<std::mutex> g(engine_mutex_);
        if (rpk_status_diff_codes(ctx_, max_pods_, staged.data(), stride, changed.data(), codes.data(), &n_changed, nullptr) != RPK_OK) return;
        ++status_calls_;
    }
    std::map<uint32_t, const Fresh*> by_slot;
    for (const auto& f : fresh) by_slot[f.slot] = &f;
    auto apply = [&](const Fresh& f, const PodStatusView& view) -> PodPtr {  // :875-880, 883, 927-929 under podsMutex
        std::lock_guard<std::mutex> g(pods_mutex_);
        auto it = pods_.find(f.key);
        if (it == pods_.end() || it->second.slot != f.slot || slot_key_[f.slot] != f.key) return nullptr;
        it->second.info.Status = f.status;
        it->second.info.PortsExposed = f.ports;
        if (!f.host_compare && stride_ == stride) std::memcpy(&records_[(size_t)f.slot * stride], &staged[(size_t)f.slot * stride], stride);
        auto np = std::make_shared<Pod>(*it->second.pod);
        np->status = view;
        it->second.pod = np;
        return np;
    };
    std::vector<uint32_t> reseed;
    for (uint32_t i = 0; i < n_changed; ++i) {
        const uint32_t slot = changed[i];
        auto ft = by_slot.find(slot);
        PodPtr np;
        if (ft != by_slot.end() && !ft->second->host_compare)
            np = apply(*ft->second, StatusFromCode(codes[i], ft->second->status, ft->second->message));
        if (np) Notify(np);  // :936-954 (the k8s PATCH of :915 is out of scope; the callback path is the PodNotifier contract)
        else reseed.push_back(slot);  // reported but not applied: the device must not keep the staged record as "previous"
    }
    for (const auto& f : fresh) {  // statuses longer than any slot: string + bool compare on the host (:870-873)
        if (!f.host_compare) continue;
        ++host_compares_;
        bool differs;
        {
            std::lock_guard<std::mutex> g(pods_mutex_);
            auto it = pods_.find(f.key);
            if (it == pods_.end() || it->second.slot != f.slot) continue;
            differs = it->second.info.Status != f.status || it->second.info.PortsExposed != f.ports;
        }
        if (!differs) continue;
        PodPtr np = apply(f, TranslateRunPodStatus(f.status, f.message, f.ports));
        if (np) Notify(np);
    }
    if (!reseed.empty()) {
        std::vector<uint8_t> recs(reseed.size() * (size_t)stride);
        bool same_stride;
        {
            std::lock_guard<std::mutex> g(pods_mutex_);
            same_stride = stride_ == stride;
            if (same_stride) for (size_t i = 0; i < reseed.size(); ++i) std::memcpy(&recs[i * stride], &records_[(size_t)reseed[i] * stride], stride);
        }
        if (same_stride) {
            std::lock_guard<std::mutex> g(engine_mutex_);
            rpk_status_seed_slots(ctx_, (uint32_t)reseed.size(), reseed.data(), recs.data(), stride);
        }
    }
}

}  // namespace rpkhost
