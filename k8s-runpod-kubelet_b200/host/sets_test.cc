// sets_test.cc -- runpod.io/gpu-type-ids in the C++ Provider mirror: the annotation parser and column producer
// (`--cpu`), and DeployBatch restricting pods to their listed GPU types through rpk_select_sets (`--gpu`, scripted
// RunPod API over the ten-offer table of tests/golden/select_kat.json).
#include <cstdio>
#include <cstring>
#include <mutex>

#include "rpk_host.hpp"

using namespace rpkhost;

static int g_fail = 0, g_checks = 0;
#define CHECK(c) do { ++g_checks; if (!(c)) { ++g_fail; std::printf("FAIL %s:%d: %s\n", __FILE__, __LINE__, #c); } } while (0)
#define CHECK_EQ(a, b) do { ++g_checks; if (!((a) == (b))) { ++g_fail; std::printf("FAIL %s:%d: %s == %s\n", __FILE__, __LINE__, #a, #b); } } while (0)
using Ids = std::vector<std::string>;

static PodPtr MakePod(const std::string& name, Annotations ann = {}, std::shared_ptr<Annotations> job = nullptr) {
    auto p = std::make_shared<Pod>();
    p->ns = "default"; p->name = name; p->annotations = std::move(ann); p->owner_job = std::move(job);
    p->status.phase = "Pending";
    return p;
}

static void TestParser() {
    CHECK_EQ(ParseGpuTypeIds(""), Ids{});
    CHECK_EQ(ParseGpuTypeIds("A40"), Ids{"A40"});
    CHECK_EQ(ParseGpuTypeIds(" A40 , L4\t,A100 "), (Ids{"A40", "L4", "A100"}));  // TrimSpace per element
    CHECK_EQ(ParseGpuTypeIds("A40,,L4"), (Ids{"A40", "", "L4"}));                 // strings.Split keeps empty elements
    CHECK_EQ(ParseGpuTypeIds(","), (Ids{"", ""}));
    CHECK_EQ(ParseGpuTypeIds("A40,"), (Ids{"A40", ""}));
}

static void TestColumns() {
    auto job = std::make_shared<Annotations>(Annotations{{GpuTypeIdsAnnotation, "RTX4090, A5000"}});
    PodColumns c = PrepareColumns(*MakePod("job-only", {}, job));  // owner Job fallback
    CHECK(c.restricted); CHECK_EQ(c.gpu_type_ids, (Ids{"RTX4090", "A5000"}));
    c = PrepareColumns(*MakePod("override", {{GpuTypeIdsAnnotation, "L4"}}, job));  // the pod's value wins
    CHECK_EQ(c.gpu_type_ids, Ids{"L4"});
    c = PrepareColumns(*MakePod("empty-pod-value", {{GpuTypeIdsAnnotation, ""}}, job));  // empty = absent: Job's value
    CHECK_EQ(c.gpu_type_ids, (Ids{"RTX4090", "A5000"}));
    c = PrepareColumns(*MakePod("none"));
    CHECK(!c.restricted); CHECK(c.gpu_type_ids.empty());
    c = PrepareColumns(*MakePod("ws", {{GpuTypeIdsAnnotation, " A40 ,, L4 "}, {GpuMemoryAnnotation, "24"}}));
    CHECK(c.restricted); CHECK_EQ(c.gpu_type_ids, (Ids{"A40", "", "L4"})); CHECK_EQ(c.req_mem_gb, 24);
    // the batch producer carries the raw value row for row
    std::vector<PodPtr> pods = {MakePod("a", {}, job), MakePod("b"), MakePod("c", {{GpuTypeIdsAnnotation, "A40"}})};
    PodColumnsSoA soa;
    PrepareColumnsBatch(pods, &soa, 1);
    CHECK_EQ(soa.gpu_type_ids[0], "RTX4090, A5000"); CHECK_EQ(soa.gpu_type_ids[1], ""); CHECK_EQ(soa.gpu_type_ids[2], "A40");
}

struct FakeRunPod : RunPodAPI {
    std::vector<GPUType> types;
    std::mutex mu;
    bool fail_deploy = false;
    int deploys = 0;
    struct Call { std::string pod; Ids ids; };
    std::vector<Call> calls;
    bool FetchGPUTypes(std::vector<GPUType>* out, std::string*) override { std::lock_guard<std::mutex> g(mu); *out = types; return true; }
    bool DeployPod(const Pod& pod, const Ids& ids, int, const std::string&, std::string* id, double* cost, std::string* err) override {
        std::lock_guard<std::mutex> g(mu);
        calls.push_back({pod.name, ids});
        if (fail_deploy || ids.empty()) { *err = "no capacity"; return false; }
        *id = "rp-" + std::to_string(++deploys); *cost = 0.25;
        return true;
    }
    bool GetDetailedPodStatus(const std::string&, DetailedStatus*, std::string* err) override { *err = "n/a"; return false; }
    bool TerminatePod(const std::string&, std::string*) override { return true; }
    Ids IdsOf(const std::string& pod) const {
        for (auto it = calls.rbegin(); it != calls.rend(); ++it) if (it->pod == pod) return it->ids;
        return {"<not deployed>"};
    }
};

static std::vector<GPUType> KatTable() {  // tests/golden/select_kat.json (SURVEY.md 8c)
    return {{"A4000", "", 16, true, .32, true, .17}, {"A5000", "", 24, true, .36, true, .22}, {"RTX3090", "", 24, false, 0, true, .22},
            {"A40", "", 48, true, .40, false, 0},    {"RTX4090", "", 24, true, .69, true, .34}, {"L4", "", 24, true, .43, false, 0},
            {"A100", "", 80, true, 1.64, true, 1.19}, {"T4free", "", 16, true, 0, true, 0},     {"A4500", "", 20, true, .34, true, .19},
            {"edge", "", 32, true, .5, true, .5}};
}

static bool Deployed(Provider& prov, const std::string& name) {
    auto p = prov.GetPod("default", name).first;
    auto a = p ? p->annotations.find(PodIDAnnotation) : Annotations::iterator();
    return p && a != p->annotations.end() && !a->second.empty();
}

static void TestDeployBatch() {
    auto api = std::make_shared<FakeRunPod>();
    api->types = KatTable();
    Provider prov(api, 1, 1024);  // the last batch holds 300 pods
    // no annotation anywhere: the plain rpk_select, nothing else
    prov.CreatePod(MakePod("plain"));
    CHECK_EQ(prov.SelectCalls(), 1u); CHECK_EQ(prov.SetSelectCalls(), 0u); CHECK_EQ(prov.SetUploads(), 0u);
    CHECK_EQ(api->IdsOf("plain"), (Ids{"A4000", "A4500", "A5000", "A40", "L4"}));
    // a restricted pod gets only listed types, cheapest first (list order does not matter)
    prov.CreatePod(MakePod("r1", {{GpuTypeIdsAnnotation, "L4, A40 ,A5000"}}));
    CHECK_EQ(api->IdsOf("r1"), (Ids{"A5000", "A40", "L4"}));
    CHECK_EQ(prov.SelectCalls(), 1u); CHECK_EQ(prov.SetSelectCalls(), 1u); CHECK_EQ(prov.SetUploads(), 1u);
    // owner Job fallback; tie 0.22 -> lower table index
    auto job = std::make_shared<Annotations>(Annotations{{GpuTypeIdsAnnotation, "RTX4090,RTX3090,A5000"}, {GpuMemoryAnnotation, "24"},
                                                         {CloudTypeAnnotation, "COMMUNITY"}});
    prov.CreatePod(MakePod("r2", {}, job));
    CHECK_EQ(api->IdsOf("r2"), (Ids{"A5000", "RTX3090", "RTX4090"}));
    // ids absent from the table are ignored; a list of unknown ids deploys nothing and stays pending
    prov.CreatePod(MakePod("r3", {{GpuTypeIdsAnnotation, "H100, A40"}, {GpuMemoryAnnotation, "24"}}));
    CHECK_EQ(api->IdsOf("r3"), Ids{"A40"});
    prov.CreatePod(MakePod("unknown", {{GpuTypeIdsAnnotation, "H100,B200"}}));
    CHECK(api->IdsOf("unknown").empty()); CHECK(!Deployed(prov, "unknown"));
    // one batch mixing unrestricted and restricted pods: ONE rpk_select_sets, every row right
    api->fail_deploy = true;
    prov.CreatePod(MakePod("m-plain", {{GpuMemoryAnnotation, "48"}}));
    prov.CreatePod(MakePod("m-a", {{GpuTypeIdsAnnotation, "A100,edge"}, {MaxPriceAnnotation, "2.0"}}));
    prov.CreatePod(MakePod("m-b", {{GpuTypeIdsAnnotation, "edge, A100"}, {MaxPriceAnnotation, "2.0"}}));  // same set
    prov.CreatePod(MakePod("m-c", {{GpuTypeIdsAnnotation, "RTX3090"}}));  // SECURE: no secure flag -> nothing
    api->fail_deploy = false;
    api->calls.clear();
    const uint64_t sets0 = prov.SetSelectCalls(), sel0 = prov.SelectCalls();
    prov.ProcessPendingPods();
    CHECK_EQ(prov.SetSelectCalls(), sets0 + 1); CHECK_EQ(prov.SelectCalls(), sel0);
    CHECK_EQ(api->IdsOf("m-plain"), Ids{"A40"});
    CHECK_EQ(api->IdsOf("m-a"), (Ids{"edge", "A100"})); CHECK_EQ(api->IdsOf("m-b"), (Ids{"edge", "A100"}));
    CHECK(api->IdsOf("m-c").empty()); CHECK(api->IdsOf("unknown").empty());
    CHECK(Deployed(prov, "m-a") && Deployed(prov, "m-plain") && !Deployed(prov, "m-c"));
    // the sets resident on the engine are reused while the table and the lists do not change
    const uint64_t up0 = prov.SetUploads();
    prov.ProcessPendingPods();  // m-c and unknown again: both lists are resident
    CHECK_EQ(prov.SetUploads(), up0);
    // sets that went stale on the engine behind the provider's back (here: the same table uploaded again directly,
    // which makes every set stale): the reuse fails, the provider forgets them, uploads once more, same tick
    {
        std::vector<int32_t> mem; std::vector<double> sp, cp; std::vector<uint8_t> fl;
        for (const auto& g : api->types) {
            mem.push_back(g.MemoryInGb); sp.push_back(g.SecurePrice); cp.push_back(g.CommunityPrice);
            fl.push_back((uint8_t)((g.SecureCloud ? 1 : 0) | (g.CommunityCloud ? 2 : 0)));
        }
        std::vector<int32_t> zero(mem.size(), 0);
        CHECK_EQ(rpk_offers_upload(prov.Ctx(), (uint32_t)mem.size(), mem.data(), zero.data(), zero.data(), sp.data(), cp.data(), fl.data()), RPK_OK);
    }
    prov.CreatePod(MakePod("stale", {{GpuTypeIdsAnnotation, "edge, A100"}, {MaxPriceAnnotation, "2.0"}}));  // a resident list
    CHECK_EQ(api->IdsOf("stale"), (Ids{"edge", "A100"}));
    CHECK_EQ(prov.SetUploads(), up0 + 1);
    const uint64_t up1 = prov.SetUploads();
    // a changed table re-uploads the sets
    api->types[5].SecurePrice = 0.30;  // L4 becomes the cheapest of r1's list
    prov.CreatePod(MakePod("r4", {{GpuTypeIdsAnnotation, "A5000,A40,L4"}}));
    CHECK_EQ(api->IdsOf("r4"), (Ids{"L4", "A5000", "A40"}));
    CHECK_EQ(prov.SetUploads(), up1 + 1); CHECK_EQ(prov.OfferUploads(), 2u);
    // more distinct lists than RPK_MAX_OFFER_SETS in one batch: several calls, same answers
    api->fail_deploy = true;
    const char* names[3] = {"A40", "L4", "A5000"};
    for (int i = 0; i < 300; ++i)
        prov.CreatePod(MakePod("many" + std::to_string(i), {{GpuTypeIdsAnnotation, std::string(names[i % 3]) + ",x" + std::to_string(i)}}));
    api->fail_deploy = false;
    api->calls.clear();
    const uint64_t sets1 = prov.SetSelectCalls();
    prov.ProcessPendingPods();
    CHECK_EQ(prov.SetSelectCalls(), sets1 + 2);
    for (int i = 0; i < 300; ++i) CHECK_EQ(api->IdsOf("many" + std::to_string(i)), Ids{names[i % 3]});
}

int main(int argc, char** argv) {
    const bool gpu = argc > 1 && std::strcmp(argv[1], "--gpu") == 0;
    TestParser();
    TestColumns();
    if (gpu) TestDeployBatch();
    std::printf("%s: %d checks, %d failed (%s)\n", g_fail ? "FAILED" : "ok", g_checks, g_fail, gpu ? "gpu" : "cpu");
    return g_fail ? 1 : 0;
}
