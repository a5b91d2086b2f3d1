// rpk_api.cu -- the C-ABI of include/rpk.h: argument checks, device buffers, H2D/D2H, shard fan-out.
// No CPU implementation of any kernel lives here (or anywhere in the product): if CUDA is unusable every
// entry point returns an error.
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <exception>
#include <functional>
#include <memory>
#include <mutex>
#include <new>
#include <thread>

#include "rpk_internal.cuh"

using namespace rpk;

struct PeerBinding { int n = 0, my_rank = 0, inline_wait = 0; uint32_t* flags[RPK_MAX_GPUS] = {}; };

// One host thread per extra GPU of a multi-GPU ctx: the per-shard halves of rpk_select / rpk_status_diff / rpk_tick
// (a dozen cudaMemcpyAsync + launches each) are issued in parallel instead of one shard after the other -- with 8
// GPUs behind one caller thread the serial issue, not PCIe, was the end-to-end bound.
struct ShardWorkers {
    struct W {
        std::thread th; std::mutex m; std::condition_variable cv;
        std::function<void()> job; bool has = false, quit = false;
    };
    std::vector<std::unique_ptr<W>> w;
    std::mutex dm; std::condition_variable dcv; int pending = 0;
    std::vector<std::exception_ptr> err;

    void start(int n) {
        err.resize((size_t)n);
        for (int i = 1; i < n; ++i) {
            w.emplace_back(new W());
            W* x = w.back().get();
            x->th = std::thread([this, x]() {
                for (;;) {
                    std::function<void()> job;
                    {
                        std::unique_lock<std::mutex> lk(x->m);
                        x->cv.wait(lk, [x] { return x->has || x->quit; });
                        if (x->quit) return;
                        job = std::move(x->job); x->has = false;
                    }
                    job();
                    { std::lock_guard<std::mutex> g(dm); --pending; }
                    dcv.notify_one();
                }
            });
        }
    }
    void stop() {
        for (auto& x : w) { { std::lock_guard<std::mutex> g(x->m); x->quit = true; } x->cv.notify_one(); x->th.join(); }
        w.clear();
    }
    // fn(s) for every shard s in [0, n): shard 0 on the calling thread, the others on their workers; rethrows the first failure
    template <typename F>
    void run(int n, F&& fn) {
        for (auto& e : err) e = nullptr;
        if (n > 1) {
            { std::lock_guard<std::mutex> g(dm); pending = n - 1; }
            for (int s = 1; s < n; ++s) {
                W* x = w[(size_t)s - 1].get();
                { std::lock_guard<std::mutex> g(x->m); x->job = [this, s, &fn]() { try { fn(s); } catch (...) { err[(size_t)s] = std::current_exception(); } }; x->has = true; }
                x->cv.notify_one();
            }
        }
        try { fn(0); } catch (...) { err[0] = std::current_exception(); }
        if (n > 1) { std::unique_lock<std::mutex> lk(dm); dcv.wait(lk, [this] { return pending == 0; }); }
        for (auto& e : err) if (e) std::rethrow_exception(e);
    }
};

struct rpk_ctx {
    std::vector<DeviceState> devs;
    std::vector<PeerBinding> bind;  // per shard: flag arrays bound with rpk_peer_bind
    ShardWorkers workers;
    std::vector<std::pair<int, void*>> ipc_owned, ipc_mapped;  // (shard, ptr)
    std::string err;
    rpk_stats stats;
    uint64_t launches = 0;
};

static thread_local std::string g_create_err;

namespace {

int fail(rpk_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg; else g_create_err = msg;
    return code;
}

template <typename F>
int guarded(rpk_ctx* ctx, F&& f) {
    try {
        return f();
    } catch (const CudaError& e) {
        char buf[512];
        snprintf(buf, sizeof(buf), "CUDA error %d (%s) at %s:%d: %s", (int)e.err, cudaGetErrorString(e.err), e.file, e.line, e.what);
        cudaGetLastError();  // clear the sticky-free error state
        return fail(ctx, e.err == cudaErrorMemoryAllocation ? RPK_ENOMEM : RPK_ECUDA, buf);
    } catch (const std::bad_alloc&) {
        return fail(ctx, RPK_ENOMEM, "host allocation failed");
    } catch (...) {
        return fail(ctx, RPK_ECUDA, "unexpected exception");
    }
}

inline void shard_range(uint32_t total, int n, int s, uint32_t* lo, uint32_t* hi) {
    *lo = (uint32_t)((uint64_t)total * (uint64_t)s / (uint64_t)n);
    *hi = (uint32_t)((uint64_t)total * (uint64_t)(s + 1) / (uint64_t)n);
}

void fill_offer_args(const OfferTable& t, SelectArgs& a) {
    for (int c = 0; c < 2; ++c) {
        a.view[c].packed = t.v_packed[c].p; a.view[c].bitmap = t.v_bitmap[c].p; a.view[c].bitmapT = t.v_bitmapT[c].p; a.view[c].wide = t.v_wide[c].p;
        a.view[c].price = t.v_price[c].p; a.view[c].perm = t.v_perm[c].p;
    }
    a.G = t.G; a.Gpad = t.Gpad; a.pk = t.pk; a.nsub = t.nsub;
    for (int d = 0; d < 3; ++d) { a.distinct[d] = t.distinct[d].p; a.D[d] = t.D[d]; }
}

// scratch for one select over P rows against table t of ds (in lane ln); returns rows-per-warp.  *use_persist: the batch
// takes the persistent bit-sliced kernel (plan in *pl).
int prepare_select_scratch(DeviceState& ds, const OfferTable& t, DeviceState::Lane& ln, uint32_t P, SelectArgs& a, PersistPlan* pl, bool* use_persist) {
    const int R = t.pk.bm_words ? 32 * pick_rows_per_lane(P, t.G, ds.sm_count) : pick_rows_per_warp(P, ds.sm_count);
    const uint32_t tiles = select_tiles_max(P, R);
    ln.rw.reserve(P); ln.order.reserve((size_t)kGroups * P); ln.pos.reserve(P);
    const size_t need = std::max<size_t>((size_t)2 * kGroups + tiles, (size_t)P / 8 + 3 * kGroups);  // worst case (1 row per warp): never regrown mid-pipeline
    if (need > ln.ctrs.cap || ln.ctrs_dirty) {
        // the counters are zero between calls by construction (finish_tile); a fresh or suspect buffer is zeroed here
        ln.ctrs.reserve(need);
        RPK_CUDA(cudaMemset(ln.ctrs.p, 0, ln.ctrs.cap * sizeof(uint32_t)));
        RPK_CUDA(cudaDeviceSynchronize());
        ln.ctrs_dirty = false;
    }
    a.rw = ln.rw.p; a.order = ln.order.p; a.pos = ln.pos.p;
    a.counts = ln.ctrs.p; a.done = ln.ctrs.p + kGroups; a.tile_ctr = ln.ctrs.p + 2 * kGroups;
    a.P = P;
    *use_persist = t.pk.bm_words && (P > kFusedRowsMax || t.pk.no_fused) && !t.pk.no_persist && persist_plan(a, ds.sm_count, pl);
    if (*use_persist) {
        ln.key.reserve(P); ln.ord_rw.reserve(P);
        const size_t hdr_words = persist_hdr_words(t.G, t.pk.bm_words);
        const bool fresh = !ln.hist.p || hdr_words > ln.hdr.cap;
        ln.hist.reserve(2 * kMaxClasses); ln.cursor.reserve(2 * kMaxClasses); ln.hdr.reserve(hdr_words);
        if (fresh || ln.persist_dirty) {  // zero between calls by construction (k_pod_classify's last block, the pushers)
            RPK_CUDA(cudaMemset(ln.hist.p, 0, ln.hist.cap * sizeof(uint32_t)));
            RPK_CUDA(cudaMemset(ln.cursor.p, 0, ln.cursor.cap * sizeof(uint32_t)));
            RPK_CUDA(cudaMemset(ln.hdr.p, 0, ln.hdr.cap * sizeof(uint32_t)));
            RPK_CUDA(cudaDeviceSynchronize());
            ln.persist_dirty = false;
        }
        a.key = ln.key.p; a.ord_rw = ln.ord_rw.p; a.hist = ln.hist.p; a.cursor = ln.cursor.p; a.hdr = ln.hdr.p;
    }
    return R;
}

// The device entry points of a shard share ctx-owned scratch (tickets, queue cursors, look-back state).  Calls on ONE
// stream are ordered by the stream; a call on a different stream than the previous one first waits for that one's
// completion event, so two streams can never run on the same scratch at once.  Inside a stream capture the guard is
// skipped (events recorded outside a capture cannot be waited on inside it): a captured step must keep each entry
// point on one stream, as bench.py does.
struct ScratchGuard {
    cudaStream_t* last; cudaEvent_t ev; cudaStream_t st; bool capturing = false;
    ScratchGuard(cudaStream_t* last_stream, cudaEvent_t event, cudaStream_t stream) : last(last_stream), ev(event), st(stream) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); cs = cudaStreamCaptureStatusNone; }
        capturing = cs != cudaStreamCaptureStatusNone;
        if (!capturing && *last != nullptr && *last != st) RPK_CUDA(cudaStreamWaitEvent(st, ev, 0));
    }
    void done() {
        if (capturing) return;
        RPK_CUDA(cudaEventRecord(ev, st));
        *last = st;
    }
};

void bind_flags(const rpk_ctx* ctx, int shard, SelectArgs& a) {
    a.n_flags = 0; a.my_rank = 0;
    if ((size_t)shard >= ctx->bind.size()) return;
    const PeerBinding& b = ctx->bind[(size_t)shard];
    for (int r = 0; r < b.n; ++r) a.flags[r] = b.flags[r];
    a.n_flags = b.n; a.my_rank = b.my_rank; a.inline_wait = b.inline_wait;
}

// Which of the output vectors lives on GPU `shard` (the others are peers' memory); -1 if none does.  Vectors this ctx
// allocated (rpk_ipc_alloc) or mapped from a peer (rpk_ipc_open) are known exactly; anything else is asked of the driver.
int find_local_vector(const rpk_ctx* ctx, int shard, int dev, int n_out, int32_t* const* ptrs) {
    if (n_out == 1) return 0;
    for (int o = 1; o < n_out; ++o)  // the push kernel moves 16-byte units: every vector must share the slice's alignment
        if (((uintptr_t)ptrs[o] & 15u) != ((uintptr_t)ptrs[0] & 15u)) return -1;
    for (int o = 0; o < n_out; ++o)
        for (const auto& m : ctx->ipc_owned) if (m.first == shard && m.second == (void*)ptrs[o]) return o;
    for (int o = 0; o < n_out; ++o) {
        bool mapped = false;
        for (const auto& m : ctx->ipc_mapped) if (m.second == (void*)ptrs[o]) { mapped = true; break; }
        if (mapped) continue;  // a peer's vector, whatever the driver reports for IPC mappings
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, ptrs[o]) != cudaSuccess) { cudaGetLastError(); continue; }
        if (at.type == cudaMemoryTypeDevice && at.device == dev) return o;
    }
    return -1;
}

// launch_select with the lane's counters marked suspect until every launch of the call was accepted
int run_select(DeviceState::Lane& ln, const SelectArgs& a, int R, const PersistPlan* pl, cudaStream_t st) {
    ln.ctrs_dirty = true; ln.persist_dirty = true;
    const int n = launch_select(a, R, pl, st);
    ln.ctrs_dirty = false; ln.persist_dirty = false;
    return n;
}

// Row sub-batches of the host entry point.  The first one is small, so that the first kernel starts after ~3 MB of
// H2D; the following ones grow (128k, 256k, 384k, 512k, 512k ... rows), because every select call pays a fixed ~40 us
// (class sort, stage load, queue tail) that eight equal sub-batches paid eight times: with growing sizes each kernel
// is about as long as the upload of the next, larger sub-batch.
constexpr uint32_t kSubBatchRows = 131072;
constexpr uint32_t kSubBatchMaxMul = 4;
inline uint32_t sub_batch_rows(int j, uint32_t remaining) {
    const uint32_t want = kSubBatchRows * (uint32_t)((j + 1) < (int)kSubBatchMaxMul ? (j + 1) : (int)kSubBatchMaxMul);
    return remaining < want + kSubBatchRows / 2 ? remaining : want;  // do not leave a sliver behind
}
inline uint32_t sub_batch_cap(uint32_t Ps) {  // largest sub-batch a shard of Ps rows produces
    uint32_t cap = 0, left = Ps;
    for (int j = 0; left; ++j) { const uint32_t nb = sub_batch_rows(j, left); cap = nb > cap ? nb : cap; left -= nb; }
    return cap ? cap : 1;
}

// Latency path of the host entry point (micro-batches, one GPU): the five pod columns are packed into one
// pinned block -> ONE H2D; best and top5 come back in ONE D2H; one stream synchronise.  Same kernels.
int select_small(rpk_ctx* ctx, DeviceState& ds, uint32_t P, const int32_t* req_mem_gb, const int32_t* req_vcpu,
                 const int32_t* req_ram_gb, const double* max_price, const uint8_t* cloud, int32_t* best, int32_t* top5,
                 uint64_t* launches) {
    (void)ctx;
    RPK_CUDA(cudaSetDevice(ds.dev));
    const size_t in_cap = (size_t)kSmallBatch * 24, out_cap = (size_t)kSmallBatch * 6 * 4;
    if (!ds.h_small) RPK_CUDA(cudaHostAlloc((void**)&ds.h_small, in_cap + out_cap, cudaHostAllocPortable));
    ds.d_small_in.reserve(in_cap); ds.d_small_out.reserve((size_t)kSmallBatch * 6);
    const size_t o_mem = 0, o_vcpu = (size_t)P * 4, o_ram = (size_t)P * 8, o_price = ((size_t)P * 12 + 7) & ~(size_t)7,
                 o_cloud = o_price + (size_t)P * 8, total = o_cloud + P;
    unsigned char* h = ds.h_small;
    memcpy(h + o_mem, req_mem_gb, (size_t)P * 4);
    if (req_vcpu) memcpy(h + o_vcpu, req_vcpu, (size_t)P * 4);
    if (req_ram_gb) memcpy(h + o_ram, req_ram_gb, (size_t)P * 4);
    if (max_price) memcpy(h + o_price, max_price, (size_t)P * 8);
    if (cloud) memcpy(h + o_cloud, cloud, P);
    DeviceState::Lane& ln = ds.lane[0];
    cudaStream_t st = ln.stream;
    unsigned char* d = ds.d_small_in.p;
    RPK_CUDA(cudaMemcpyAsync(d, h, total, cudaMemcpyHostToDevice, st));
    SelectArgs a{};
    a.req_mem = (const int32_t*)(d + o_mem); a.req_vcpu = req_vcpu ? (const int32_t*)(d + o_vcpu) : nullptr;
    a.req_ram = req_ram_gb ? (const int32_t*)(d + o_ram) : nullptr; a.max_price = max_price ? (const double*)(d + o_price) : nullptr;
    a.cloud = cloud ? (const uint8_t*)(d + o_cloud) : nullptr;
    a.P = P;
    fill_offer_args(ds.main, a);
    PersistPlan pl; bool persist = false;
    const int R = prepare_select_scratch(ds, ds.main, ln, P, a, &pl, &persist);
    a.best_out[0] = ds.d_small_out.p; a.n_out = 1; a.self_out = 0; a.row0 = 0; a.top5 = top5 ? ds.d_small_out.p + P : nullptr;
    *launches += (uint64_t)run_select(ln, a, R, persist ? &pl : nullptr, st);
    int32_t* hout = (int32_t*)(ds.h_small + in_cap);
    RPK_CUDA(cudaMemcpyAsync(hout, ds.d_small_out.p, (size_t)P * 4 * (top5 ? 6 : 1), cudaMemcpyDeviceToHost, st));
    RPK_CUDA(cudaStreamSynchronize(st));
    memcpy(best, hout, (size_t)P * 4);
    if (top5) memcpy(top5, hout + P, (size_t)P * 4 * RPK_TOPK);
    return RPK_OK;
}

bool has_int32_max(const int32_t* col, uint32_t n) {
    if (!col) return false;
    for (uint32_t i = 0; i < n; ++i) if (col[i] == INT32_MAX) return true;
    return false;
}


// Buffers of the pipelined host select, sized from the calling thread (peers write into each other's best_full, so
// every GPU's vector must exist before any shard is enqueued).  After the first call of a size this only compares
// capacities.
void reserve_select(rpk_ctx* ctx, uint32_t P, bool vcpu, bool ram, bool price, bool cloud, bool top5) {
    const int n = (int)ctx->devs.size();
    for (int s = 0; s < n; ++s) {
        DeviceState& ds = ctx->devs[(size_t)s];
        uint32_t lo, hi; shard_range(P, n, s, &lo, &hi);
        const uint32_t Ps = hi - lo;
        const uint32_t cap = sub_batch_cap(Ps);
        bool grow = P > ds.best_full.cap;
        for (auto& ln : ds.lane) {
            grow = grow || cap > ln.p_req_mem.cap || (vcpu && cap > ln.p_req_vcpu.cap) || (ram && cap > ln.p_req_ram.cap) ||
                   (price && cap > ln.p_max_price.cap) || (cloud && cap > ln.p_cloud.cap) || (top5 && (size_t)cap * RPK_TOPK > ln.top5.cap);
            if (cap == Ps) break;  // a single sub-batch uses lane 0 only
        }
        if (!grow) continue;
        RPK_CUDA(cudaSetDevice(ds.dev));
        ds.best_full.reserve(P);
        for (auto& ln : ds.lane) {
            ln.p_req_mem.reserve(cap);
            if (vcpu) ln.p_req_vcpu.reserve(cap);
            if (ram) ln.p_req_ram.reserve(cap);
            if (price) ln.p_max_price.reserve(cap);
            if (cloud) ln.p_cloud.reserve(cap);
            if (top5) ln.top5.reserve((size_t)cap * RPK_TOPK);
            if (cap == Ps) break;
        }
    }
}

// One shard's half of the host select: row sub-batches alternate between two lanes; within a lane everything is stream
// ordered (H2D -> kernels -> D2H), across lanes copies and kernels overlap.  ds.ev[0] / ds.ev[3] bracket it on ds.stream;
// the caller synchronises ds.stream.
void enqueue_select_shard(rpk_ctx* ctx, int s, uint32_t P, const int32_t* req_mem_gb, const int32_t* req_vcpu, const int32_t* req_ram_gb,
                          const double* max_price, const uint8_t* cloud, int32_t* best, int32_t* top5, uint64_t* launches) {
    const int n = (int)ctx->devs.size();
    DeviceState& ds = ctx->devs[(size_t)s];
    uint32_t lo, hi; shard_range(P, n, s, &lo, &hi);
    RPK_CUDA(cudaSetDevice(ds.dev));
    RPK_CUDA(cudaEventRecord(ds.ev[0], ds.stream));
    for (auto& ln : ds.lane) RPK_CUDA(cudaStreamWaitEvent(ln.stream, ds.ev[0], 0));
    int j = 0;
    for (uint32_t b0 = lo, nb = 0; b0 < hi; b0 += nb, ++j) {
        nb = sub_batch_rows(j, hi - b0);
        DeviceState::Lane& ln = ds.lane[j % DeviceState::kLanes];
        cudaStream_t st = ln.stream;
        RPK_CUDA(cudaMemcpyAsync(ln.p_req_mem.p, req_mem_gb + b0, (size_t)nb * 4, cudaMemcpyHostToDevice, st));
        if (req_vcpu) RPK_CUDA(cudaMemcpyAsync(ln.p_req_vcpu.p, req_vcpu + b0, (size_t)nb * 4, cudaMemcpyHostToDevice, st));
        if (req_ram_gb) RPK_CUDA(cudaMemcpyAsync(ln.p_req_ram.p, req_ram_gb + b0, (size_t)nb * 4, cudaMemcpyHostToDevice, st));
        if (max_price) RPK_CUDA(cudaMemcpyAsync(ln.p_max_price.p, max_price + b0, (size_t)nb * 8, cudaMemcpyHostToDevice, st));
        if (cloud) RPK_CUDA(cudaMemcpyAsync(ln.p_cloud.p, cloud + b0, (size_t)nb, cudaMemcpyHostToDevice, st));
        SelectArgs a{};
        a.req_mem = ln.p_req_mem.p; a.req_vcpu = req_vcpu ? ln.p_req_vcpu.p : nullptr; a.req_ram = req_ram_gb ? ln.p_req_ram.p : nullptr;
        a.max_price = max_price ? ln.p_max_price.p : nullptr; a.cloud = cloud ? ln.p_cloud.p : nullptr;
        a.P = nb;
        fill_offer_args(ds.main, a);
        PersistPlan pl; bool persist = false;
        const int R = prepare_select_scratch(ds, ds.main, ln, nb, a, &pl, &persist);
        for (int o = 0; o < n; ++o) a.best_out[o] = ctx->devs[(size_t)o].best_full.p;
        a.n_out = n; a.row0 = b0; a.top5 = top5 ? ln.top5.p : nullptr;
        a.self_out = s;  // own vector; finished push blocks / sub-batches are forwarded to the peers
        *launches += (uint64_t)run_select(ln, a, R, persist ? &pl : nullptr, st);
        RPK_CUDA(cudaMemcpyAsync(best + b0, ds.best_full.p + b0, (size_t)nb * 4, cudaMemcpyDeviceToHost, st));
        if (top5) RPK_CUDA(cudaMemcpyAsync(top5 + (size_t)b0 * RPK_TOPK, ln.top5.p, (size_t)nb * RPK_TOPK * 4, cudaMemcpyDeviceToHost, st));
    }
    for (auto& ln : ds.lane) {
        RPK_CUDA(cudaEventRecord(ln.done, ln.stream));
        RPK_CUDA(cudaStreamWaitEvent(ds.stream, ln.done, 0));
    }
    RPK_CUDA(cudaEventRecord(ds.ev[3], ds.stream));
}

}  // namespace

extern "C" {

int rpk_abi_version(void) { return RPK_ABI_VERSION; }

const char* rpk_last_error(const rpk_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

void* rpk_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void rpk_host_free(void* p) { if (p) cudaFreeHost(p); }

int rpk_create(int n_gpus, const int* device_ids, rpk_ctx** out) {
    if (!out) return fail(nullptr, RPK_EINVAL, "rpk_create: out is NULL");
    *out = nullptr;
    if (n_gpus < 1 || n_gpus > RPK_MAX_GPUS) return fail(nullptr, RPK_EINVAL, "rpk_create: n_gpus must be in [1, 8]");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(nullptr, RPK_ENODEV, std::string("rpk_create: no CUDA device (") + cudaGetErrorString(e) + "); there is no CPU fallback");
    }
    rpk_ctx* ctx = new (std::nothrow) rpk_ctx();
    if (!ctx) return fail(nullptr, RPK_ENOMEM, "rpk_create: host allocation failed");
    memset(&ctx->stats, 0, sizeof(ctx->stats));
    int rc = guarded(nullptr, [&]() -> int {
        ctx->devs.resize((size_t)n_gpus);
        for (int i = 0; i < n_gpus; ++i) {
            const int dev = device_ids ? device_ids[i] : i;
            if (dev < 0 || dev >= count) return fail(nullptr, RPK_EINVAL, "rpk_create: device id out of range");
            for (int j = 0; j < i; ++j) if (ctx->devs[(size_t)j].dev == dev) return fail(nullptr, RPK_EINVAL, "rpk_create: duplicate device id");
            cudaDeviceProp prop;
            RPK_CUDA(cudaGetDeviceProperties(&prop, dev));
            if (prop.major != 10) {
                char buf[160];
                snprintf(buf, sizeof(buf), "rpk_create: device %d is sm_%d%d; this library holds sm_100a code only and has no fallback", dev, prop.major, prop.minor);
                return fail(nullptr, RPK_ENODEV, buf);
            }
            DeviceState& ds = ctx->devs[(size_t)i];
            ds.dev = dev; ds.sm_count = prop.multiProcessorCount;
            RPK_CUDA(cudaSetDevice(dev));
            // the selection is the latency-critical half of a tick, the sweep is background work: when both have CTAs
            // pending, the block scheduler places the selection's first (measured: the sweep beside a 1M-row select
            // costs 5 us instead of 15)
            int prio_lo = 0, prio_hi = 0;
            RPK_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
            RPK_CUDA(cudaStreamCreateWithPriority(&ds.stream, cudaStreamNonBlocking, prio_hi));
            RPK_CUDA(cudaStreamCreateWithPriority(&ds.status_stream, cudaStreamNonBlocking, prio_lo));
            for (auto& ev : ds.ev) RPK_CUDA(cudaEventCreate(&ev));
            RPK_CUDA(cudaEventCreateWithFlags(&ds.ev_sel, cudaEventDisableTiming));
            RPK_CUDA(cudaEventCreateWithFlags(&ds.ev_st, cudaEventDisableTiming));
            for (auto& ln : ds.lane) {
                RPK_CUDA(cudaStreamCreateWithPriority(&ln.stream, cudaStreamNonBlocking, prio_hi));
                RPK_CUDA(cudaEventCreateWithFlags(&ln.done, cudaEventDisableTiming));
            }
        }
        for (int i = 0; i < n_gpus && n_gpus > 1; ++i) {
            RPK_CUDA(cudaSetDevice(ctx->devs[(size_t)i].dev));
            for (int j = 0; j < n_gpus; ++j) {
                if (i == j) continue;
                int can = 0;
                RPK_CUDA(cudaDeviceCanAccessPeer(&can, ctx->devs[(size_t)i].dev, ctx->devs[(size_t)j].dev));
                if (!can) return fail(nullptr, RPK_ENODEV, "rpk_create: GPUs of the ctx cannot access each other (NVLink/P2P required for n_gpus > 1)");
                cudaError_t pe = cudaDeviceEnablePeerAccess(ctx->devs[(size_t)j].dev, 0);
                if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) RPK_CUDA(pe);
                cudaGetLastError();
            }
        }
        ctx->stats.n_gpus = (uint32_t)n_gpus;
        ctx->workers.start(n_gpus);
        return RPK_OK;
    });
    if (rc != RPK_OK) { rpk_destroy(ctx); return rc; }
    *out = ctx;
    return RPK_OK;
}

void rpk_destroy(rpk_ctx* ctx) {
    if (!ctx) return;
    ctx->workers.stop();
    for (auto& m : ctx->ipc_mapped) if (cudaSetDevice(ctx->devs[(size_t)m.first].dev) == cudaSuccess) cudaIpcCloseMemHandle(m.second);
    for (auto& m : ctx->ipc_owned) if (cudaSetDevice(ctx->devs[(size_t)m.first].dev) == cudaSuccess) { cudaDeviceSynchronize(); cudaFree(m.second); }
    cudaGetLastError();
    for (auto& ds : ctx->devs) {
        if (ds.dev < 0) continue;
        if (cudaSetDevice(ds.dev) != cudaSuccess) { cudaGetLastError(); continue; }
        if (ds.stream) cudaStreamSynchronize(ds.stream);
        ds.raw_mem.release(); ds.raw_vcpu.release(); ds.raw_ram.release(); ds.raw_sp.release(); ds.raw_cp.release(); ds.raw_flags.release();
        ds.sort_keys.release(); ds.sort_vals.release();
        ds.main.release();
        for (auto& t : ds.sets) t.release();
        ds.sets.clear();
        ds.set_words.release(); ds.set_members.release(); ds.set_mem.release(); ds.set_vcpu.release(); ds.set_ram.release();
        ds.set_sp.release(); ds.set_cp.release(); ds.set_flags.release(); ds.ss.release();
        ds.dcount.release();
        for (auto& ln : ds.lane) {
            if (ln.stream) cudaStreamSynchronize(ln.stream);
            ln.release();
            if (ln.done) cudaEventDestroy(ln.done);
            if (ln.stream) cudaStreamDestroy(ln.stream);
        }
        ds.best_full.release(); ds.d_small_in.release(); ds.d_small_out.release();
        if (ds.h_small) { cudaFreeHost(ds.h_small); ds.h_small = nullptr; }
        ds.s_records.release(); ds.s_hash_prev.release(); ds.s_hash_out.release(); ds.s_changed.release(); ds.s_misc.release(); ds.s_tile_state.release(); ds.s_stage_idx.release();
        ds.s_stage_code.release(); ds.s_unit_cnt.release(); ds.s_seed_slots.release(); ds.s_seed_recs.release();
        if (ds.h_changed) { cudaFreeHost(ds.h_changed); ds.h_changed = nullptr; }
        if (ds.status_stream) { cudaStreamSynchronize(ds.status_stream); cudaStreamDestroy(ds.status_stream); }
        for (auto& ev : ds.ev) if (ev) cudaEventDestroy(ev);
        if (ds.ev_sel) cudaEventDestroy(ds.ev_sel);
        if (ds.ev_st) cudaEventDestroy(ds.ev_st);
        if (ds.stream) cudaStreamDestroy(ds.stream);
        cudaGetLastError();
    }
    delete ctx;
}

int rpk_offers_upload(rpk_ctx* ctx, uint32_t G, const int32_t* mem_gb, const int32_t* vcpu, const int32_t* ram_gb,
                      const double* secure_price, const double* community_price, const uint8_t* flags) {
    if (!ctx) return RPK_EINVAL;
    if (G > 0 && (!mem_gb || !secure_price || !community_price || !flags))
        return fail(ctx, RPK_EINVAL, "rpk_offers_upload: mem_gb, secure_price, community_price and flags are required");
    if (G > (1u << 26)) return fail(ctx, RPK_EINVAL, "rpk_offers_upload: G above 2^26 offers is not supported");
    if (has_int32_max(mem_gb, G) || has_int32_max(vcpu, G) || has_int32_max(ram_gb, G))
        return fail(ctx, RPK_EINVAL, "rpk_offers_upload: offer columns must be < INT32_MAX (requests saturate there)");
    return guarded(ctx, [&]() -> int {
        for (auto& ds : ctx->devs) {
            RPK_CUDA(cudaSetDevice(ds.dev));
            ds.offers_ready = false;
            ++ds.table_version;  // offer sets built on the previous table are stale from here on
            ds.force_kind = 0;
            // test hook (exercise every kernel on any table): consulted once per table upload, never on the select path
            if (const char* fk = getenv("RPK_FORCE_KERNEL")) {
                if (!strcmp(fk, "generic")) ds.force_kind = 1; else if (!strcmp(fk, "packed")) ds.force_kind = 2;
                else if (!strcmp(fk, "packed_pos")) ds.force_kind = 3; else if (!strcmp(fk, "bitmap")) ds.force_kind = 4;
                else if (!strcmp(fk, "bitmap_grouped")) ds.force_kind = 5;  // every batch size through the persistent kernel
                else if (!strcmp(fk, "bitmap_grid")) ds.force_kind = 6;     // ... through the first-generation grid kernel
            }
            const size_t n = G ? G : 1;
            ds.raw_mem.reserve(n); ds.raw_vcpu.reserve(n); ds.raw_ram.reserve(n); ds.raw_sp.reserve(n); ds.raw_cp.reserve(n); ds.raw_flags.reserve(n);
            if (G) {
                RPK_CUDA(cudaMemcpyAsync(ds.raw_mem.p, mem_gb, (size_t)G * 4, cudaMemcpyHostToDevice, ds.stream));
                if (vcpu) RPK_CUDA(cudaMemcpyAsync(ds.raw_vcpu.p, vcpu, (size_t)G * 4, cudaMemcpyHostToDevice, ds.stream));
                else RPK_CUDA(cudaMemsetAsync(ds.raw_vcpu.p, 0, (size_t)G * 4, ds.stream));
                if (ram_gb) RPK_CUDA(cudaMemcpyAsync(ds.raw_ram.p, ram_gb, (size_t)G * 4, cudaMemcpyHostToDevice, ds.stream));
                else RPK_CUDA(cudaMemsetAsync(ds.raw_ram.p, 0, (size_t)G * 4, ds.stream));
                RPK_CUDA(cudaMemcpyAsync(ds.raw_sp.p, secure_price, (size_t)G * 8, cudaMemcpyHostToDevice, ds.stream));
                RPK_CUDA(cudaMemcpyAsync(ds.raw_cp.p, community_price, (size_t)G * 8, cudaMemcpyHostToDevice, ds.stream));
                RPK_CUDA(cudaMemcpyAsync(ds.raw_flags.p, flags, (size_t)G, cudaMemcpyHostToDevice, ds.stream));
            }
            OfferIngest in{G, ds.raw_mem.p, ds.raw_vcpu.p, ds.raw_ram.p, ds.raw_sp.p, ds.raw_cp.p, ds.raw_flags.p};
            ctx->launches += (uint64_t)launch_offer_ingest(ds, ds.main, in, ds.stream);
            RPK_CUDA(cudaStreamSynchronize(ds.stream));
            ds.offers_ready = true;
        }
        const DeviceState& d0 = ctx->devs[0];
        ctx->stats.select_kernel_kind = d0.main.pk.bm_words ? 4u : d0.main.pk.bits ? (d0.main.pk.pos_bits ? 3u : 2u) : 1u;
        ctx->stats.distinct_mem = d0.main.D[0]; ctx->stats.distinct_vcpu = d0.main.D[1]; ctx->stats.distinct_ram = d0.main.D[2];
        ctx->stats.packed_bits = d0.main.pk.bits;
        return RPK_OK;
    });
}

int rpk_select_device_gather(rpk_ctx* ctx, int shard, uint32_t P, const int32_t* d_req_mem_gb, const int32_t* d_req_vcpu,
                             const int32_t* d_req_ram_gb, const double* d_max_price, const uint8_t* d_cloud,
                             int n_out, int32_t* const* d_best_full, uint32_t row0, int32_t* d_top5, void* stream) {
    if (!ctx) return RPK_EINVAL;
    if (shard < 0 || (size_t)shard >= ctx->devs.size()) return fail(ctx, RPK_EINVAL, "rpk_select_device: shard out of range");
    if (P == 0) return RPK_OK;
    if (!d_req_mem_gb || !d_best_full || n_out < 1 || n_out > RPK_MAX_GPUS) return fail(ctx, RPK_EINVAL, "rpk_select_device: req_mem_gb and 1..8 output vectors are required");
    for (int o = 0; o < n_out; ++o) if (!d_best_full[o]) return fail(ctx, RPK_EINVAL, "rpk_select_device: NULL output vector");
    DeviceState& ds = ctx->devs[(size_t)shard];
    if (!ds.offers_ready) return fail(ctx, RPK_ESTATE, "rpk_select: no offer table uploaded (call rpk_offers_upload first)");
    return guarded(ctx, [&]() -> int {
        RPK_CUDA(cudaSetDevice(ds.dev));
        SelectArgs a{};
        a.req_mem = d_req_mem_gb; a.req_vcpu = d_req_vcpu; a.req_ram = d_req_ram_gb; a.max_price = d_max_price; a.cloud = d_cloud;
        a.P = P;
        fill_offer_args(ds.main, a);
        PersistPlan pl; bool persist = false;
        const int R = prepare_select_scratch(ds, ds.main, ds.lane[0], P, a, &pl, &persist);
        for (int o = 0; o < n_out; ++o) a.best_out[o] = d_best_full[o];
        a.n_out = n_out; a.row0 = row0; a.top5 = d_top5;
        a.self_out = find_local_vector(ctx, shard, ds.dev, n_out, d_best_full);
        if (n_out > 1) bind_flags(ctx, shard, a);
        cudaStream_t st = stream ? (cudaStream_t)stream : ds.stream;
        ScratchGuard guard(&ds.sel_last_stream, ds.ev_sel, st);
        ctx->launches += (uint64_t)run_select(ds.lane[0], a, R, persist ? &pl : nullptr, st);
        guard.done();
        ctx->stats.select_calls += 1;
        ctx->stats.offer_scores += (uint64_t)P * ds.main.G;
        return RPK_OK;
    });
}

int rpk_select_device(rpk_ctx* ctx, int shard, uint32_t P, const int32_t* d_req_mem_gb, const int32_t* d_req_vcpu,
                      const int32_t* d_req_ram_gb, const double* d_max_price, const uint8_t* d_cloud, int32_t* d_best,
                      int32_t* d_top5, void* stream) {
    int32_t* outs[1] = {d_best};
    return rpk_select_device_gather(ctx, shard, P, d_req_mem_gb, d_req_vcpu, d_req_ram_gb, d_max_price, d_cloud, 1, outs, 0, d_top5, stream);
}

int rpk_select(rpk_ctx* ctx, uint32_t P, const int32_t* req_mem_gb, const int32_t* req_vcpu, const int32_t* req_ram_gb,
               const double* max_price, const uint8_t* cloud, int32_t* best, int32_t* top5) {
    if (!ctx) return RPK_EINVAL;
    if (P == 0) return RPK_OK;
    if (!req_mem_gb || !best) return fail(ctx, RPK_EINVAL, "rpk_select: req_mem_gb and best are required");
    for (auto& ds : ctx->devs) if (!ds.offers_ready) return fail(ctx, RPK_ESTATE, "rpk_select: no offer table uploaded (call rpk_offers_upload first)");
    return guarded(ctx, [&]() -> int {
        const int n = (int)ctx->devs.size();
        if (n == 1 && P <= kSmallBatch) {
            int rc = select_small(ctx, ctx->devs[0], P, req_mem_gb, req_vcpu, req_ram_gb, max_price, cloud, best, top5, &ctx->launches);
            ctx->stats.last_select_kernel_ms = 0.f; ctx->stats.last_select_total_ms = 0.f;
            ctx->stats.select_calls += 1;
            ctx->stats.offer_scores += (uint64_t)P * ctx->devs[0].main.G;
            return rc;
        }
        std::vector<uint64_t> launches((size_t)n, 0);
        std::vector<float> ms((size_t)n, 0.f);
        reserve_select(ctx, P, req_vcpu != nullptr, req_ram_gb != nullptr, max_price != nullptr, cloud != nullptr, top5 != nullptr);
        ctx->workers.run(n, [&](int s) {
            enqueue_select_shard(ctx, s, P, req_mem_gb, req_vcpu, req_ram_gb, max_price, cloud, best, top5, &launches[(size_t)s]);
            DeviceState& ds = ctx->devs[(size_t)s];
            RPK_CUDA(cudaStreamSynchronize(ds.stream));
            RPK_CUDA(cudaEventElapsedTime(&ms[(size_t)s], ds.ev[0], ds.ev[3]));
        });
        float tmax = 0.f;
        for (int s = 0; s < n; ++s) { ctx->launches += launches[(size_t)s]; tmax = ms[(size_t)s] > tmax ? ms[(size_t)s] : tmax; }
        ctx->stats.last_select_kernel_ms = 0.f;  // copies and kernels overlap in the pipelined host path: only the total is meaningful
        ctx->stats.last_select_total_ms = tmax;
        ctx->stats.select_calls += 1;
        ctx->stats.offer_scores += (uint64_t)P * ctx->devs[0].main.G;
        return RPK_OK;
    });
}

// ---- offer sets --------------------------------------------------------------------------------------------

int rpk_offer_sets_upload(rpk_ctx* ctx, uint32_t n_sets, uint32_t G, const uint32_t* members) {
    if (!ctx) return RPK_EINVAL;
    if (n_sets > RPK_MAX_OFFER_SETS) return fail(ctx, RPK_EINVAL, "rpk_offer_sets_upload: at most RPK_MAX_OFFER_SETS (256) sets");
    for (auto& ds : ctx->devs) if (!ds.offers_ready) return fail(ctx, RPK_ESTATE, "rpk_offer_sets_upload: no offer table uploaded (call rpk_offers_upload first)");
    if (G != ctx->devs[0].main.G) return fail(ctx, RPK_EINVAL, "rpk_offer_sets_upload: G differs from the resident offer table's");
    const uint32_t W = (G + 31) / 32;
    if (n_sets > 0 && W > 0 && !members) return fail(ctx, RPK_EINVAL, "rpk_offer_sets_upload: members is NULL");
    // member counts from the words themselves (bits >= G ignored): the host sizes every sub-table without a readback
    std::vector<uint32_t> counts(n_sets, 0);
    for (uint32_t s = 0; s < n_sets; ++s) {
        uint32_t c = 0;
        for (uint32_t w = 0; w < W; ++w) {
            uint32_t m = members[(size_t)s * W + w];
            if ((w + 1) * 32 > G) m &= (1u << (G - w * 32)) - 1u;
            c += (uint32_t)__builtin_popcount(m);
        }
        counts[s] = c;
    }
    return guarded(ctx, [&]() -> int {
        for (auto& ds : ctx->devs) {
            RPK_CUDA(cudaSetDevice(ds.dev));
            ds.sets_ready = false;
            for (size_t s = n_sets; s < ds.sets.size(); ++s) ds.sets[s].release();
            ds.sets.resize(n_sets);
            if (n_sets && W) {
                ds.set_words.reserve((size_t)n_sets * W);
                RPK_CUDA(cudaMemcpyAsync(ds.set_words.p, members, (size_t)n_sets * W * 4, cudaMemcpyHostToDevice, ds.stream));
            }
            ctx->launches += (uint64_t)launch_offer_sets_build(ds, n_sets, ds.set_words.p, counts.data(), ds.stream);
            RPK_CUDA(cudaStreamSynchronize(ds.stream));
            ds.sets_ready = true;
            ds.sets_version = ds.table_version;
        }
        return RPK_OK;
    });
}

namespace {

struct SetCols {  // one shard's pod columns on its device (nullable ones as in rpk_select)
    const int32_t* mem; const int32_t* vcpu; const int32_t* ram; const double* price; const uint8_t* cloud; const uint16_t* set_id;
};

int check_sets_state(rpk_ctx* ctx, const DeviceState& ds) {
    if (!ds.offers_ready) return fail(ctx, RPK_ESTATE, "rpk_select_sets: no offer table uploaded (call rpk_offers_upload first)");
    if (!ds.sets_ready || ds.sets_version != ds.table_version)
        return fail(ctx, RPK_ESTATE, "rpk_select_sets: no offer sets for the current offer table (call rpk_offer_sets_upload after rpk_offers_upload)");
    return RPK_OK;
}

// One shard's restricted select on stream st: partition the rows by set id, one select per non-empty bin against its
// set's sub-table (lane 0's scratch, one bin after the other), write-back in row order.  Synchronises st once (the bin
// counts); with no set column it is one plain select against the resident table.  *scores += sum of P_s * G_s.
void select_sets_shard(DeviceState& ds, uint32_t P, const SetCols& c, int32_t* d_best, int32_t* d_top5, cudaStream_t st,
                       uint64_t* launches, uint64_t* scores) {
    DeviceState::Lane& ln = ds.lane[0];
    auto select_on = [&](const OfferTable& t, uint32_t n, const int32_t* m, const int32_t* v, const int32_t* r, const double* pr,
                         const uint8_t* cl, int32_t* best_vec, uint32_t row0, int32_t* top5) {
        SelectArgs a{};
        a.req_mem = m; a.req_vcpu = v; a.req_ram = r; a.max_price = pr; a.cloud = cl;
        a.P = n;
        fill_offer_args(t, a);
        PersistPlan pl; bool persist = false;
        const int R = prepare_select_scratch(ds, t, ln, n, a, &pl, &persist);
        a.best_out[0] = best_vec; a.n_out = 1; a.self_out = 0; a.row0 = row0; a.top5 = top5;
        *launches += (uint64_t)run_select(ln, a, R, persist ? &pl : nullptr, st);
        *scores += (uint64_t)n * t.G;
    };
    if (!c.set_id) { select_on(ds.main, P, c.mem, c.vcpu, c.ram, c.price, c.cloud, d_best, 0, d_top5); return; }
    const uint32_t n_sets = (uint32_t)ds.sets.size(), nb = n_sets + 2;
    DeviceState::SetSelect& ss = ds.ss;
    ss.p_mem.reserve(P); ss.rows.reserve(P); ss.tmp_best.reserve(P); ss.hist.reserve(2 * (RPK_MAX_OFFER_SETS + 2));
    if (c.vcpu) ss.p_vcpu.reserve(P);
    if (c.ram) ss.p_ram.reserve(P);
    if (c.price) ss.p_price.reserve(P);
    if (c.cloud) ss.p_cloud.reserve(P);
    if (d_top5) ss.tmp_top5.reserve((size_t)P * RPK_TOPK);
    if (!ss.h_counts) RPK_CUDA(cudaHostAlloc((void**)&ss.h_counts, (RPK_MAX_OFFER_SETS + 2) * sizeof(uint32_t), cudaHostAllocPortable));
    RPK_CUDA(cudaMemsetAsync(ss.hist.p, 0, (size_t)2 * nb * sizeof(uint32_t), st));
    SetPartitionArgs pa{};
    pa.P = P; pa.n_sets = n_sets; pa.set_id = c.set_id;
    pa.req_mem = c.mem; pa.req_vcpu = c.vcpu; pa.req_ram = c.ram; pa.max_price = c.price; pa.cloud = c.cloud;
    pa.o_mem = ss.p_mem.p; pa.o_vcpu = ss.p_vcpu.p; pa.o_ram = ss.p_ram.p; pa.o_price = ss.p_price.p; pa.o_cloud = ss.p_cloud.p;
    pa.rows = ss.rows.p; pa.hist = ss.hist.p;
    *launches += (uint64_t)launch_set_partition(pa, st);
    RPK_CUDA(cudaMemcpyAsync(ss.h_counts, ss.hist.p, (size_t)nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    RPK_CUDA(cudaStreamSynchronize(st));  // the one synchronisation: bin sizes decide the launches below
    uint32_t start = 0;
    for (uint32_t b = 0; b < nb; ++b) {
        const uint32_t cnt = ss.h_counts[b];
        if (cnt == 0) continue;
        const OfferTable* t = b < n_sets ? &ds.sets[b] : b == n_sets ? &ds.main : nullptr;
        int32_t* t5 = d_top5 ? ss.tmp_top5.p + (size_t)start * RPK_TOPK : nullptr;
        if (t && t->G) {
            select_on(*t, cnt, ss.p_mem.p + start, c.vcpu ? ss.p_vcpu.p + start : nullptr, c.ram ? ss.p_ram.p + start : nullptr,
                      c.price ? ss.p_price.p + start : nullptr, c.cloud ? ss.p_cloud.p + start : nullptr, ss.tmp_best.p, start, t5);
        } else {  // empty set or unknown id: nothing is feasible
            RPK_CUDA(cudaMemsetAsync(ss.tmp_best.p + start, 0xFF, (size_t)cnt * 4, st));
            if (t5) RPK_CUDA(cudaMemsetAsync(t5, 0xFF, (size_t)cnt * RPK_TOPK * 4, st));
        }
        start += cnt;
    }
    *launches += (uint64_t)launch_set_unpermute(P, ss.rows.p, ss.tmp_best.p, d_top5 ? ss.tmp_top5.p : nullptr, d_best, d_top5, st);
}

}  // namespace

int rpk_select_sets_device(rpk_ctx* ctx, int shard, uint32_t P, const int32_t* d_req_mem_gb, const int32_t* d_req_vcpu,
                           const int32_t* d_req_ram_gb, const double* d_max_price, const uint8_t* d_cloud,
                           const uint16_t* d_set_id, int32_t* d_best, int32_t* d_top5, void* stream) {
    if (!ctx) return RPK_EINVAL;
    if (shard < 0 || (size_t)shard >= ctx->devs.size()) return fail(ctx, RPK_EINVAL, "rpk_select_sets_device: shard out of range");
    if (P == 0) return RPK_OK;
    if (!d_req_mem_gb || !d_best) return fail(ctx, RPK_EINVAL, "rpk_select_sets_device: req_mem_gb and best are required");
    DeviceState& ds = ctx->devs[(size_t)shard];
    if (!ds.offers_ready) return fail(ctx, RPK_ESTATE, "rpk_select_sets: no offer table uploaded (call rpk_offers_upload first)");
    if (d_set_id) { if (int rc = check_sets_state(ctx, ds)) return rc; }
    return guarded(ctx, [&]() -> int {
        RPK_CUDA(cudaSetDevice(ds.dev));
        cudaStream_t st = stream ? (cudaStream_t)stream : ds.stream;
        if (d_set_id) {  // the bin counts are read back mid-call: refuse a capturing stream before enqueuing anything
            cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
            RPK_CUDA(cudaStreamIsCapturing(st, &cs));
            if (cs != cudaStreamCaptureStatusNone)
                return fail(ctx, RPK_ESTATE, "rpk_select_sets_device: the stream is being captured; with set ids the call synchronises it once and cannot be captured");
        }
        ScratchGuard guard(&ds.sel_last_stream, ds.ev_sel, st);
        uint64_t scores = 0;
        const SetCols c{d_req_mem_gb, d_req_vcpu, d_req_ram_gb, d_max_price, d_cloud, d_set_id};
        select_sets_shard(ds, P, c, d_best, d_top5, st, &ctx->launches, &scores);
        guard.done();
        ctx->stats.select_calls += 1;
        ctx->stats.offer_scores += scores;
        return RPK_OK;
    });
}

int rpk_select_sets(rpk_ctx* ctx, uint32_t P, const int32_t* req_mem_gb, const int32_t* req_vcpu, const int32_t* req_ram_gb,
                    const double* max_price, const uint8_t* cloud, const uint16_t* set_id, int32_t* best, int32_t* top5) {
    if (!ctx) return RPK_EINVAL;
    if (P == 0) return RPK_OK;
    if (!req_mem_gb || !best) return fail(ctx, RPK_EINVAL, "rpk_select_sets: req_mem_gb and best are required");
    for (auto& ds : ctx->devs) {
        if (!ds.offers_ready) return fail(ctx, RPK_ESTATE, "rpk_select_sets: no offer table uploaded (call rpk_offers_upload first)");
        if (set_id) { if (int rc = check_sets_state(ctx, ds)) return rc; }
    }
    return guarded(ctx, [&]() -> int {
        const int n = (int)ctx->devs.size();
        std::vector<uint64_t> launches((size_t)n, 0), scores((size_t)n, 0);
        // rows are sharded like rpk_select's; each shard is one sub-batch: H2D, partition + selects, D2H
        ctx->workers.run(n, [&](int s) {
            DeviceState& ds = ctx->devs[(size_t)s];
            uint32_t lo, hi; shard_range(P, n, s, &lo, &hi);
            const uint32_t Ps = hi - lo;
            if (Ps == 0) return;
            RPK_CUDA(cudaSetDevice(ds.dev));
            DeviceState::SetSelect& ss = ds.ss;
            cudaStream_t st = ds.stream;
            ScratchGuard guard(&ds.sel_last_stream, ds.ev_sel, st);
            ss.in_mem.reserve(Ps); ss.out_best.reserve(Ps);
            RPK_CUDA(cudaMemcpyAsync(ss.in_mem.p, req_mem_gb + lo, (size_t)Ps * 4, cudaMemcpyHostToDevice, st));
            SetCols c{ss.in_mem.p, nullptr, nullptr, nullptr, nullptr, nullptr};
            if (req_vcpu) { ss.in_vcpu.reserve(Ps); RPK_CUDA(cudaMemcpyAsync(ss.in_vcpu.p, req_vcpu + lo, (size_t)Ps * 4, cudaMemcpyHostToDevice, st)); c.vcpu = ss.in_vcpu.p; }
            if (req_ram_gb) { ss.in_ram.reserve(Ps); RPK_CUDA(cudaMemcpyAsync(ss.in_ram.p, req_ram_gb + lo, (size_t)Ps * 4, cudaMemcpyHostToDevice, st)); c.ram = ss.in_ram.p; }
            if (max_price) { ss.in_price.reserve(Ps); RPK_CUDA(cudaMemcpyAsync(ss.in_price.p, max_price + lo, (size_t)Ps * 8, cudaMemcpyHostToDevice, st)); c.price = ss.in_price.p; }
            if (cloud) { ss.in_cloud.reserve(Ps); RPK_CUDA(cudaMemcpyAsync(ss.in_cloud.p, cloud + lo, (size_t)Ps, cudaMemcpyHostToDevice, st)); c.cloud = ss.in_cloud.p; }
            if (set_id) { ss.in_set.reserve(Ps); RPK_CUDA(cudaMemcpyAsync(ss.in_set.p, set_id + lo, (size_t)Ps * 2, cudaMemcpyHostToDevice, st)); c.set_id = ss.in_set.p; }
            if (top5) ss.out_top5.reserve((size_t)Ps * RPK_TOPK);
            select_sets_shard(ds, Ps, c, ss.out_best.p, top5 ? ss.out_top5.p : nullptr, st, &launches[(size_t)s], &scores[(size_t)s]);
            RPK_CUDA(cudaMemcpyAsync(best + lo, ss.out_best.p, (size_t)Ps * 4, cudaMemcpyDeviceToHost, st));
            if (top5) RPK_CUDA(cudaMemcpyAsync(top5 + (size_t)lo * RPK_TOPK, ss.out_top5.p, (size_t)Ps * RPK_TOPK * 4, cudaMemcpyDeviceToHost, st));
            guard.done();
            RPK_CUDA(cudaStreamSynchronize(st));
        });
        for (int s = 0; s < n; ++s) { ctx->launches += launches[(size_t)s]; ctx->stats.offer_scores += scores[(size_t)s]; }
        ctx->stats.select_calls += 1;
        return RPK_OK;
    });
}

// ---- cross-process peer vectors (CUDA IPC) ---------------------------------------------------------------

int rpk_ipc_alloc(rpk_ctx* ctx, int shard, size_t bytes, void** d_ptr, unsigned char handle_out[64]) {
    if (!ctx) return RPK_EINVAL;
    if (shard < 0 || (size_t)shard >= ctx->devs.size() || !d_ptr || !handle_out || bytes == 0) return fail(ctx, RPK_EINVAL, "rpk_ipc_alloc: bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle is 64 bytes");
    return guarded(ctx, [&]() -> int {
        RPK_CUDA(cudaSetDevice(ctx->devs[(size_t)shard].dev));
        void* p = nullptr;
        RPK_CUDA(cudaMalloc(&p, bytes));
        RPK_CUDA(cudaMemset(p, 0, bytes));
        cudaIpcMemHandle_t h;
        cudaError_t e = cudaIpcGetMemHandle(&h, p);
        if (e != cudaSuccess) { cudaFree(p); RPK_CUDA(e); }
        memcpy(handle_out, &h, 64);
        ctx->ipc_owned.emplace_back(shard, p);
        *d_ptr = p;
        return RPK_OK;
    });
}

int rpk_ipc_open(rpk_ctx* ctx, int shard, const unsigned char handle[64], void** d_peer_ptr) {
    if (!ctx) return RPK_EINVAL;
    if (shard < 0 || (size_t)shard >= ctx->devs.size() || !handle || !d_peer_ptr) return fail(ctx, RPK_EINVAL, "rpk_ipc_open: bad argument");
    return guarded(ctx, [&]() -> int {
        RPK_CUDA(cudaSetDevice(ctx->devs[(size_t)shard].dev));
        cudaIpcMemHandle_t h;
        memcpy(&h, handle, 64);
        void* p = nullptr;
        RPK_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        ctx->ipc_mapped.emplace_back(shard, p);
        *d_peer_ptr = p;
        return RPK_OK;
    });
}

static int drop_entry(std::vector<std::pair<int, void*>>& v, int shard, void* p) {
    for (size_t i = 0; i < v.size(); ++i)
        if (v[i].first == shard && v[i].second == p) { v.erase(v.begin() + (long)i); return 1; }
    return 0;
}

int rpk_ipc_close(rpk_ctx* ctx, int shard, void* d_peer_ptr) {
    if (!ctx) return RPK_EINVAL;
    if (!drop_entry(ctx->ipc_mapped, shard, d_peer_ptr)) return fail(ctx, RPK_EINVAL, "rpk_ipc_close: pointer was not opened by this ctx");
    return guarded(ctx, [&]() -> int {
        RPK_CUDA(cudaSetDevice(ctx->devs[(size_t)shard].dev));
        RPK_CUDA(cudaIpcCloseMemHandle(d_peer_ptr));
        return RPK_OK;
    });
}

int rpk_ipc_free(rpk_ctx* ctx, int shard, void* d_ptr) {
    if (!ctx) return RPK_EINVAL;
    if (!drop_entry(ctx->ipc_owned, shard, d_ptr)) return fail(ctx, RPK_EINVAL, "rpk_ipc_free: pointer was not allocated by this ctx");
    return guarded(ctx, [&]() -> int {
        RPK_CUDA(cudaSetDevice(ctx->devs[(size_t)shard].dev));
        RPK_CUDA(cudaFree(d_ptr));
        return RPK_OK;
    });
}

int rpk_peer_fence(rpk_ctx* ctx, int shard, int n, uint32_t* const* d_flags, int my_rank, uint32_t epoch, void* stream) {
    if (!ctx) return RPK_EINVAL;
    if (shard < 0 || (size_t)shard >= ctx->devs.size() || n < 1 || n > RPK_MAX_GPUS || !d_flags || my_rank < 0 || my_rank >= n)
        return fail(ctx, RPK_EINVAL, "rpk_peer_fence: bad argument");
    for (int r = 0; r < n; ++r) if (!d_flags[r]) return fail(ctx, RPK_EINVAL, "rpk_peer_fence: NULL flag array");
    DeviceState& ds = ctx->devs[(size_t)shard];
    return guarded(ctx, [&]() -> int {
        RPK_CUDA(cudaSetDevice(ds.dev));
        PeerFenceArgs a{};
        for (int r = 0; r < n; ++r) a.flags[r] = d_flags[r];
        a.n = n; a.my_rank = my_rank; a.epoch = epoch;
        ctx->launches += (uint64_t)launch_peer_fence(a, stream ? (cudaStream_t)stream : ds.stream);
        return RPK_OK;
    });
}

int rpk_peer_bind(rpk_ctx* ctx, int shard, int n, uint32_t* const* d_flags, int my_rank) {
    if (!ctx) return RPK_EINVAL;
    if (shard < 0 || (size_t)shard >= ctx->devs.size() || n < 0 || n > RPK_MAX_GPUS || (n > 0 && (!d_flags || my_rank < 0 || my_rank >= n)))
        return fail(ctx, RPK_EINVAL, "rpk_peer_bind: bad argument");
    for (int r = 0; r < n; ++r) if (!d_flags[r]) return fail(ctx, RPK_EINVAL, "rpk_peer_bind: NULL flag array");
    if (ctx->bind.size() < ctx->devs.size()) ctx->bind.resize(ctx->devs.size());
    PeerBinding& b = ctx->bind[(size_t)shard];
    const int keep = b.inline_wait;
    b = PeerBinding{};
    for (int r = 0; r < n; ++r) b.flags[r] = d_flags[r];
    b.n = n; b.my_rank = my_rank; b.inline_wait = keep;
    return RPK_OK;
}

int rpk_peer_inline_wait(rpk_ctx* ctx, int shard, int on) {
    if (!ctx) return RPK_EINVAL;
    if (shard < 0 || (size_t)shard >= ctx->devs.size()) return fail(ctx, RPK_EINVAL, "rpk_peer_inline_wait: shard out of range");
    if (ctx->bind.size() < ctx->devs.size()) ctx->bind.resize(ctx->devs.size());
    ctx->bind[(size_t)shard].inline_wait = on ? 1 : 0;
    return RPK_OK;
}

int rpk_peer_wait(rpk_ctx* ctx, int shard, unsigned what, void* stream) {
    if (!ctx) return RPK_EINVAL;
    if (shard < 0 || (size_t)shard >= ctx->devs.size() || (what & ~3u) || !what) return fail(ctx, RPK_EINVAL, "rpk_peer_wait: bad argument");
    if ((size_t)shard >= ctx->bind.size() || ctx->bind[(size_t)shard].n == 0) return fail(ctx, RPK_ESTATE, "rpk_peer_wait: no flags bound (rpk_peer_bind)");
    DeviceState& ds = ctx->devs[(size_t)shard];
    return guarded(ctx, [&]() -> int {
        RPK_CUDA(cudaSetDevice(ds.dev));
        const PeerBinding& b = ctx->bind[(size_t)shard];
        PeerFenceArgs a{};
        for (int r = 0; r < b.n; ++r) a.flags[r] = b.flags[r];
        a.n = b.n; a.my_rank = b.my_rank; a.epoch = 0;
        ctx->launches += (uint64_t)launch_peer_wait(a, what, stream ? (cudaStream_t)stream : ds.stream);
        return RPK_OK;
    });
}

/* test / integration hook: device pointer of GPU `shard`'s copy of the last full assignment vector */
const int32_t* rpk_best_device_ptr(const rpk_ctx* ctx, int shard) {
    if (!ctx || shard < 0 || (size_t)shard >= ctx->devs.size()) return nullptr;
    return ctx->devs[(size_t)shard].best_full.p;
}

// ---- status --------------------------------------------------------------------------------------------

static int check_stride(rpk_ctx* ctx, uint32_t stride) {
    if (stride < 16 || stride > 256 || (stride & 15)) return fail(ctx, RPK_EINVAL, "status stride must be a multiple of 16 in [16, 256]");
    return RPK_OK;
}

int rpk_status_reset(rpk_ctx* ctx, uint32_t N) {
    if (!ctx) return RPK_EINVAL;
    return guarded(ctx, [&]() -> int {
        const int n = (int)ctx->devs.size();
        for (int s = 0; s < n; ++s) {
            DeviceState& ds = ctx->devs[(size_t)s];
            uint32_t lo, hi; shard_range(N, n, s, &lo, &hi);
            RPK_CUDA(cudaSetDevice(ds.dev));
            ds.s_hash_prev.reserve((hi - lo) ? (hi - lo) : 1);
            RPK_CUDA(cudaMemsetAsync(ds.s_hash_prev.p, 0, (size_t)((hi - lo) ? (hi - lo) : 1) * 8, ds.stream));
            RPK_CUDA(cudaStreamSynchronize(ds.stream));
            ds.statusN = N; ds.status_sized = true;
        }
        return RPK_OK;
    });
}

namespace {

// look-back state / tickets of the status kernels: zero between calls by construction; zeroed here when (re)allocated
void reserve_status_state(DeviceState& ds, uint32_t N, uint32_t stride) {
    const size_t need = status_state_words(N, stride, ds.sm_count);
    if (need > ds.s_tile_state.cap || !ds.s_misc.p || ds.status_dirty) {
        ds.s_tile_state.reserve(need);
        ds.s_misc.reserve(64);
        RPK_CUDA(cudaMemset(ds.s_tile_state.p, 0, ds.s_tile_state.cap * sizeof(unsigned long long)));
        RPK_CUDA(cudaMemset(ds.s_misc.p, 0, ds.s_misc.cap * sizeof(uint32_t)));
        RPK_CUDA(cudaDeviceSynchronize());
        ds.status_dirty = false;
    }
}

struct StatusHostArgs {
    uint32_t N; const uint8_t* records; uint32_t stride;
    uint32_t* changed_idx; uint16_t* changed_code; uint32_t* n_changed; uint64_t* hashes_out; bool report;
};

// Sizes one shard's buffers (calling thread).  The changed list comes back through mapped pinned memory -- the kernel's
// final copy writes indices, codes and the count straight into it, so the host needs ONE stream synchronise and no
// device-to-host copy whose size it would first have to learn.
void reserve_status_shard(rpk_ctx* ctx, int s, const StatusHostArgs& h) {
    const int n = (int)ctx->devs.size();
    DeviceState& ds = ctx->devs[(size_t)s];
    uint32_t lo, hi; shard_range(h.N, n, s, &lo, &hi);
    const uint32_t Ns = hi - lo, cap = Ns ? Ns : 1;
    RPK_CUDA(cudaSetDevice(ds.dev));
    ds.s_records.reserve((size_t)cap * h.stride);
    ds.s_stage_idx.reserve(cap + 64); ds.s_unit_cnt.reserve(cap / 32 + 2);
    if (h.changed_code) ds.s_stage_code.reserve(cap + 64);
    if (h.hashes_out) ds.s_hash_out.reserve(cap);
    reserve_status_state(ds, cap, h.stride);
    const size_t need = h.report ? (size_t)cap * (h.changed_code ? 6 : 4) + 64 : 64;
    if (need > ds.h_changed_cap) {
        if (ds.h_changed) RPK_CUDA(cudaFreeHost(ds.h_changed));
        ds.h_changed = nullptr; ds.h_changed_cap = 0;
        const size_t want = need + need / 4;
        RPK_CUDA(cudaHostAlloc((void**)&ds.h_changed, want, cudaHostAllocMapped | cudaHostAllocPortable));
        RPK_CUDA(cudaHostGetDevicePointer((void**)&ds.d_changed_map, ds.h_changed, 0));
        ds.h_changed_cap = want;
    }
}

// One shard's half of a host sweep, enqueued on ds.stream (ds.ev[0..2] bracket copy and kernel); the caller synchronises.
void enqueue_status_shard(rpk_ctx* ctx, int s, const StatusHostArgs& h, uint64_t* launches) {
    const int n = (int)ctx->devs.size();
    DeviceState& ds = ctx->devs[(size_t)s];
    uint32_t lo, hi; shard_range(h.N, n, s, &lo, &hi);
    const uint32_t Ns = hi - lo, cap = Ns ? Ns : 1;
    RPK_CUDA(cudaSetDevice(ds.dev));
    RPK_CUDA(cudaEventRecord(ds.ev[0], ds.stream));
    if (Ns) RPK_CUDA(cudaMemcpyAsync(ds.s_records.p, h.records + (size_t)lo * h.stride, (size_t)Ns * h.stride, cudaMemcpyHostToDevice, ds.stream));
    RPK_CUDA(cudaEventRecord(ds.ev[1], ds.stream));
    // mapped block: [count : 64 bytes][indices : cap u32][codes : cap u16]
    uint32_t* m_count = reinterpret_cast<uint32_t*>(ds.d_changed_map);
    uint32_t* m_idx = reinterpret_cast<uint32_t*>(ds.d_changed_map + 64);
    uint16_t* m_code = reinterpret_cast<uint16_t*>(ds.d_changed_map + 64 + (size_t)cap * 4);
    *reinterpret_cast<volatile uint32_t*>(ds.h_changed) = 0u;
    StatusArgs a{};
    a.records = ds.s_records.p; a.stride = h.stride; a.N = Ns; a.hash_prev = ds.s_hash_prev.p;
    a.hash_out = h.hashes_out ? ds.s_hash_out.p : nullptr;
    a.changed_idx = h.report ? m_idx : nullptr; a.n_changed = h.report ? m_count : nullptr;
    a.changed_code = h.report && h.changed_code ? m_code : nullptr;
    a.idx_base = lo; a.tile_state = ds.s_tile_state.p; a.tile_counter = ds.s_misc.p;
    a.stage_idx = ds.s_stage_idx.p; a.stage_code = h.changed_code ? ds.s_stage_code.p : nullptr; a.unit_cnt = ds.s_unit_cnt.p;
    ds.status_dirty = true;
    if (Ns) *launches += (uint64_t)launch_status_diff(a, ds.stream);
    ds.status_dirty = false;
    RPK_CUDA(cudaEventRecord(ds.ev[2], ds.stream));
    if (h.hashes_out && Ns) RPK_CUDA(cudaMemcpyAsync(h.hashes_out + lo, ds.s_hash_out.p, (size_t)Ns * 8, cudaMemcpyDeviceToHost, ds.stream));
}

// after the shard's stream has been synchronised: this shard's part of the caller's arrays (ascending over shards)
uint32_t collect_status_shard(rpk_ctx* ctx, int s, const StatusHostArgs& h, uint32_t out_at) {
    const int n = (int)ctx->devs.size();
    DeviceState& ds = ctx->devs[(size_t)s];
    uint32_t lo, hi; shard_range(h.N, n, s, &lo, &hi);
    const uint32_t Ns = hi - lo, cap = Ns ? Ns : 1;
    if (!h.report || !Ns) return 0;
    const uint32_t cnt = *reinterpret_cast<volatile uint32_t*>(ds.h_changed);
    memcpy(h.changed_idx + out_at, ds.h_changed + 64, (size_t)cnt * 4);
    if (h.changed_code) memcpy(h.changed_code + out_at, ds.h_changed + 64 + (size_t)cap * 4, (size_t)cnt * 2);
    return cnt;
}

int status_host(rpk_ctx* ctx, const StatusHostArgs& h) {
    if (!ctx) return RPK_EINVAL;
    if (int rc = check_stride(ctx, h.stride)) return rc;
    if (h.N > 0 && !h.records) return fail(ctx, RPK_EINVAL, "rpk_status_diff: records is NULL");
    if (h.report && (!h.n_changed || (h.N > 0 && !h.changed_idx))) return fail(ctx, RPK_EINVAL, "rpk_status_diff: changed_idx and n_changed are required");
    if (!ctx->devs[0].status_sized) { if (int rc = rpk_status_reset(ctx, h.N)) return rc; }
    if (ctx->devs[0].statusN != h.N) return fail(ctx, RPK_ESTATE, "rpk_status_diff: N differs from the tracked table (call rpk_status_reset to resize)");
    return guarded(ctx, [&]() -> int {
        const int n = (int)ctx->devs.size();
        for (int s = 0; s < n; ++s) reserve_status_shard(ctx, s, h);
        std::vector<uint64_t> launches((size_t)n, 0);
        std::vector<float> km((size_t)n, 0.f), tm((size_t)n, 0.f);
        ctx->workers.run(n, [&](int s) {
            enqueue_status_shard(ctx, s, h, &launches[(size_t)s]);
            DeviceState& ds = ctx->devs[(size_t)s];
            RPK_CUDA(cudaEventRecord(ds.ev[3], ds.stream));
            RPK_CUDA(cudaStreamSynchronize(ds.stream));
            RPK_CUDA(cudaEventElapsedTime(&km[(size_t)s], ds.ev[1], ds.ev[2]));
            RPK_CUDA(cudaEventElapsedTime(&tm[(size_t)s], ds.ev[0], ds.ev[3]));
        });
        uint32_t total = 0;
        float kmax = 0.f, tmax = 0.f;
        for (int s = 0; s < n; ++s) {
            total += collect_status_shard(ctx, s, h, total);
            ctx->launches += launches[(size_t)s];
            kmax = km[(size_t)s] > kmax ? km[(size_t)s] : kmax; tmax = tm[(size_t)s] > tmax ? tm[(size_t)s] : tmax;
        }
        if (h.report) *h.n_changed = total;
        ctx->stats.last_status_kernel_ms = kmax; ctx->stats.last_status_total_ms = tmax;
        ctx->stats.status_calls += 1; ctx->stats.status_records += h.N;
        return RPK_OK;
    });
}

}  // namespace

int rpk_status_diff(rpk_ctx* ctx, uint32_t N, const uint8_t* records, uint32_t stride, uint32_t* changed_idx,
                    uint32_t* n_changed, uint64_t* hashes_out) {
    return status_host(ctx, StatusHostArgs{N, records, stride, changed_idx, nullptr, n_changed, hashes_out, true});
}

int rpk_status_diff_codes(rpk_ctx* ctx, uint32_t N, const uint8_t* records, uint32_t stride, uint32_t* changed_idx,
                          uint16_t* changed_code, uint32_t* n_changed, uint64_t* hashes_out) {
    return status_host(ctx, StatusHostArgs{N, records, stride, changed_idx, changed_code, n_changed, hashes_out, true});
}

int rpk_status_seed(rpk_ctx* ctx, uint32_t N, const uint8_t* records, uint32_t stride) {
    return status_host(ctx, StatusHostArgs{N, records, stride, nullptr, nullptr, nullptr, nullptr, false});
}

int rpk_status_seed_slots(rpk_ctx* ctx, uint32_t n_slots, const uint32_t* slots, const uint8_t* records, uint32_t stride) {
    if (!ctx) return RPK_EINVAL;
    if (int rc = check_stride(ctx, stride)) return rc;
    if (n_slots == 0) return RPK_OK;
    if (!slots || !records) return fail(ctx, RPK_EINVAL, "rpk_status_seed_slots: slots and records are required");
    if (!ctx->devs[0].status_sized) return fail(ctx, RPK_ESTATE, "rpk_status_seed_slots: no tracked table (call rpk_status_reset first)");
    const uint32_t N = ctx->devs[0].statusN;
    for (uint32_t i = 0; i < n_slots; ++i) if (slots[i] >= N) return fail(ctx, RPK_EINVAL, "rpk_status_seed_slots: slot index outside the tracked table");
    return guarded(ctx, [&]() -> int {
        const int n = (int)ctx->devs.size();
        for (int s = 0; s < n; ++s) {  // a handful of slots: every GPU gets the list and keeps the ones of its shard
            DeviceState& ds = ctx->devs[(size_t)s];
            uint32_t lo, hi; shard_range(N, n, s, &lo, &hi);
            bool any = false;
            for (uint32_t i = 0; i < n_slots && !any; ++i) any = slots[i] >= lo && slots[i] < hi;
            if (!any) continue;
            RPK_CUDA(cudaSetDevice(ds.dev));
            ds.s_seed_slots.reserve(n_slots); ds.s_seed_recs.reserve((size_t)n_slots * stride);
            RPK_CUDA(cudaMemcpyAsync(ds.s_seed_slots.p, slots, (size_t)n_slots * 4, cudaMemcpyHostToDevice, ds.stream));
            RPK_CUDA(cudaMemcpyAsync(ds.s_seed_recs.p, records, (size_t)n_slots * stride, cudaMemcpyHostToDevice, ds.stream));
            ctx->launches += (uint64_t)launch_status_seed_slots(n_slots, ds.s_seed_slots.p, ds.s_seed_recs.p, stride, ds.s_hash_prev.p, lo, hi, ds.stream);
            RPK_CUDA(cudaStreamSynchronize(ds.stream));
        }
        return RPK_OK;
    });
}

// One tick of the kubelet: the pending-pod selection (processPendingPods, kubelet.go:747-814) and the status sweep
// (updateAllPodStatuses, kubelet.go:816-974) are independent, so their copies and kernels are enqueued together --
// the sweep's upload runs behind the selection's, the kernels of one under the copies of the other -- and the
// call synchronises once.
int rpk_tick(rpk_ctx* ctx, uint32_t P, const int32_t* req_mem_gb, const int32_t* req_vcpu, const int32_t* req_ram_gb,
             const double* max_price, const uint8_t* cloud, int32_t* best, int32_t* top5, uint32_t N, const uint8_t* records,
             uint32_t stride, uint32_t* changed_idx, uint16_t* changed_code, uint32_t* n_changed) {
    if (!ctx) return RPK_EINVAL;
    const StatusHostArgs h{N, records, stride, changed_idx, changed_code, n_changed, nullptr, true};
    if (int rc = check_stride(ctx, stride)) return rc;
    if (P > 0 && (!req_mem_gb || !best)) return fail(ctx, RPK_EINVAL, "rpk_tick: req_mem_gb and best are required");
    if (N > 0 && !records) return fail(ctx, RPK_EINVAL, "rpk_tick: records is NULL");
    if (!n_changed || (N > 0 && !changed_idx)) return fail(ctx, RPK_EINVAL, "rpk_tick: changed_idx and n_changed are required");
    if (P > 0) for (auto& ds : ctx->devs) if (!ds.offers_ready) return fail(ctx, RPK_ESTATE, "rpk_tick: no offer table uploaded (call rpk_offers_upload first)");
    if (!ctx->devs[0].status_sized) { if (int rc = rpk_status_reset(ctx, N)) return rc; }
    if (ctx->devs[0].statusN != N) return fail(ctx, RPK_ESTATE, "rpk_tick: N differs from the tracked table (call rpk_status_reset to resize)");
    return guarded(ctx, [&]() -> int {
        const int n = (int)ctx->devs.size();
        if (P > 0) reserve_select(ctx, P, req_vcpu != nullptr, req_ram_gb != nullptr, max_price != nullptr, cloud != nullptr, top5 != nullptr);
        for (int s = 0; s < n; ++s) reserve_status_shard(ctx, s, h);
        std::vector<uint64_t> launches((size_t)n, 0);
        ctx->workers.run(n, [&](int s) {
            DeviceState& ds = ctx->devs[(size_t)s];
            // the selection goes first: its kernels are the long pole and start after the first 128k-row sub-batch has
            // landed; the sweep's records follow on the status stream and its kernel runs under the selection's tail
            if (P > 0) enqueue_select_shard(ctx, s, P, req_mem_gb, req_vcpu, req_ram_gb, max_price, cloud, best, top5, &launches[(size_t)s]);
            RPK_CUDA(cudaSetDevice(ds.dev));
            cudaStream_t keep = ds.stream;
            ds.stream = ds.status_stream;  // the sweep's copies and kernel: its own stream, concurrent with the lanes
            try { enqueue_status_shard(ctx, s, h, &launches[(size_t)s]); } catch (...) { ds.stream = keep; throw; }
            ds.stream = keep;
            RPK_CUDA(cudaStreamSynchronize(ds.status_stream));
            if (P > 0) RPK_CUDA(cudaStreamSynchronize(ds.stream));
        });
        uint32_t total = 0;
        for (int s = 0; s < n; ++s) { total += collect_status_shard(ctx, s, h, total); ctx->launches += launches[(size_t)s]; }
        *n_changed = total;
        ctx->stats.status_calls += 1; ctx->stats.status_records += N;
        if (P > 0) { ctx->stats.select_calls += 1; ctx->stats.offer_scores += (uint64_t)P * ctx->devs[0].main.G; }
        return RPK_OK;
    });
}

namespace {
int status_device(rpk_ctx* ctx, int shard, uint32_t N, const uint8_t* d_records, uint32_t stride, uint64_t* d_hash_prev,
                  uint32_t idx_base, uint32_t* d_changed_idx, uint16_t* d_changed_code, uint32_t* d_n_changed, int n_out,
                  uint32_t* const* d_xchg, uint32_t cap, int my_rank, void* stream) {
    if (!ctx) return RPK_EINVAL;
    if (shard < 0 || (size_t)shard >= ctx->devs.size()) return fail(ctx, RPK_EINVAL, "rpk_status_diff_device: shard out of range");
    if (int rc = check_stride(ctx, stride)) return rc;
    if (N > 0 && (!d_records || !d_hash_prev)) return fail(ctx, RPK_EINVAL, "rpk_status_diff_device: NULL column");
    if (n_out == 0 && N > 0 && !d_changed_idx) return fail(ctx, RPK_EINVAL, "rpk_status_diff_device: d_changed_idx is NULL");
    if (!d_n_changed) return fail(ctx, RPK_EINVAL, "rpk_status_diff_device: d_n_changed is NULL");
    if (((uintptr_t)d_records | (uintptr_t)d_hash_prev) & 15) return fail(ctx, RPK_EINVAL, "rpk_status_diff_device: d_records and d_hash_prev must be 16-byte aligned");
    if (n_out < 0 || n_out > RPK_MAX_GPUS || (n_out > 0 && (!d_xchg || my_rank < 0 || my_rank >= n_out || N > cap)))
        return fail(ctx, RPK_EINVAL, "rpk_status_diff_device_gather: bad exchange arguments (N must fit the per-rank capacity)");
    if (n_out > 0 && stride != 16 && stride != 32) return fail(ctx, RPK_EINVAL, "rpk_status_diff_device_gather: strides 16 and 32 only");
    DeviceState& ds = ctx->devs[(size_t)shard];
    return guarded(ctx, [&]() -> int {
        RPK_CUDA(cudaSetDevice(ds.dev));
        reserve_status_state(ds, N ? N : 1, stride);
        ds.s_stage_idx.reserve((N ? N : 1) + 64); ds.s_unit_cnt.reserve(N / 32 + 2);
        if (d_changed_code || n_out > 0) ds.s_stage_code.reserve((N ? N : 1) + 64);
        StatusArgs a{};
        a.records = d_records; a.stride = stride; a.N = N; a.hash_prev = d_hash_prev; a.hash_out = nullptr;
        a.changed_idx = d_changed_idx; a.changed_code = d_changed_code; a.n_changed = d_n_changed; a.idx_base = idx_base;
        a.tile_state = ds.s_tile_state.p; a.tile_counter = ds.s_misc.p;
        a.stage_idx = ds.s_stage_idx.p; a.stage_code = (d_changed_code || n_out > 0) ? ds.s_stage_code.p : nullptr; a.unit_cnt = ds.s_unit_cnt.p;
        a.n_out = n_out; a.my_rank = my_rank;
        for (int o = 0; o < n_out; ++o) {  // rank o's buffer: [counts : 8 words][n_out index regions of cap][n_out code regions of cap u16]
            uint32_t* base = d_xchg[o];
            a.out_count[o] = base;
            a.out_idx[o] = base + 8 + (size_t)my_rank * cap;
            a.out_code[o] = reinterpret_cast<uint16_t*>(base + 8 + (size_t)n_out * cap) + (size_t)my_rank * cap;
        }
        if (n_out > 0 && (size_t)shard < ctx->bind.size()) {
            const PeerBinding& b = ctx->bind[(size_t)shard];
            for (int r = 0; r < b.n; ++r) a.flags[r] = b.flags[r];
            a.n_flags = b.n; a.inline_wait = b.inline_wait;
        }
        cudaStream_t st = stream ? (cudaStream_t)stream : ds.stream;
        ScratchGuard guard(&ds.st_last_stream, ds.ev_st, st);
        ds.status_dirty = true;
        ctx->launches += (uint64_t)launch_status_diff(a, st);
        ds.status_dirty = false;
        guard.done();
        ctx->stats.status_calls += 1; ctx->stats.status_records += N;
        return RPK_OK;
    });
}
}  // namespace

int rpk_status_diff_device(rpk_ctx* ctx, int shard, uint32_t N, const uint8_t* d_records, uint32_t stride,
                           uint64_t* d_hash_prev, uint32_t* d_changed_idx, uint32_t* d_n_changed, void* stream) {
    return status_device(ctx, shard, N, d_records, stride, d_hash_prev, 0, d_changed_idx, nullptr, d_n_changed, 0, nullptr, 0, 0, stream);
}

int rpk_status_diff_device_codes(rpk_ctx* ctx, int shard, uint32_t N, const uint8_t* d_records, uint32_t stride,
                                 uint64_t* d_hash_prev, uint32_t* d_changed_idx, uint16_t* d_changed_code, uint32_t* d_n_changed, void* stream) {
    return status_device(ctx, shard, N, d_records, stride, d_hash_prev, 0, d_changed_idx, d_changed_code, d_n_changed, 0, nullptr, 0, 0, stream);
}

size_t rpk_xchg_bytes(int n_ranks, uint32_t cap) { return (size_t)(8 + (size_t)n_ranks * cap) * 4 + (size_t)n_ranks * cap * 2 + 16; }

int rpk_status_diff_device_gather(rpk_ctx* ctx, int shard, uint32_t N, const uint8_t* d_records, uint32_t stride,
                                  uint64_t* d_hash_prev, uint32_t idx_base, int n_ranks, uint32_t* const* d_xchg, uint32_t cap,
                                  int my_rank, uint32_t* d_n_changed, void* stream) {
    return status_device(ctx, shard, N, d_records, stride, d_hash_prev, idx_base, nullptr, nullptr, d_n_changed, n_ranks, d_xchg, cap, my_rank, stream);
}

int rpk_stats_get(const rpk_ctx* ctx, rpk_stats* out) {
    if (!ctx || !out) return RPK_EINVAL;
    *out = ctx->stats;
    return RPK_OK;
}

uint64_t rpk_launch_count(const rpk_ctx* ctx) { return ctx ? ctx->launches : 0; }

}  // extern "C"
