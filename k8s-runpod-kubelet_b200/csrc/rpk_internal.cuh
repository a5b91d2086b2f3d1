// rpk_internal.cuh -- shared declarations of the rpk engine (not part of the C-ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "rpk.h"

namespace rpk {

constexpr uint32_t kNone = 0xFFFFFFFFu;      // "no feasible position"
constexpr uint32_t kGroups = 8;              // row groups: cloud view x (vcpu constrains) x (ram constrains)
constexpr int kWarpsPerCta = 8;              // select kernels: 256 threads
constexpr int kCtaThreads = kWarpsPerCta * 32;
constexpr uint32_t kChunk = 128;             // offers per warp-iteration (LDS.128 per lane)
constexpr uint32_t kSegPacked = 16384;       // packed words staged per CTA (64 KB); a power of two (see kPosBits)
constexpr uint32_t kPosBits = 14;            // log2(kSegPacked): position-in-segment bits of a "pos" packed word
constexpr uint32_t kSegWide = 4096;          // wide int4 views staged per CTA (64 KB)

// Layout of the packed offer word (sorted-by-price order, one u32 per offer), from bit `sh_ram` up:
//   [guard1][mem rank' : b1][guard2][vcpu rank : b2][guard3][ram rank : b3][position in segment : pos_bits]
// rank' = rank+1 (0 = offer not available in this cloud).  A pod's word holds its thresholds in the same
// fields with guards 0, so (offer - pod) keeps a field's guard iff offer_field >= pod_field.
// pos_bits = kPosBits when bits <= 32 - kPosBits: the low bits then carry the offer's position inside its
// 16384-offer segment and the kernel reduces key = (~d & guard) | (d & pos_mask) with a plain unsigned min
// (feasible keys are positions, infeasible ones are >= 2^pos_bits).  Otherwise pos_bits = 0 and the kernel
// tracks the position itself with predicated selects.
struct PackLayout {
    uint32_t guard;    // the three guard bits
    uint32_t sh_mem;   // shift of the mem field
    uint32_t sh_vcpu;  // shift of the vcpu field
    uint32_t sh_ram;   // shift of the ram field (= pos_bits)
    uint32_t pos_bits; // kPosBits or 0
    uint32_t bits;     // field + guard bits used (0 = table not packable -> generic kernel)
    // bit-sliced view (kernel kind 4): per 32-offer chunk, kBmStride words; word i < bm_words is the 32-bit
    // mask "offer j of the chunk passes threshold i" -- mem thresholds first (rank' >= t', t' = 1..D_mem+1, so
    // unavailable offers fail all of them), then vcpu thresholds 0..D_vcpu, then ram thresholds 0..D_ram.
    uint32_t bm_words; // D_mem+1 + D_vcpu+1 + D_ram+1 if that fits 64 words, else 0
    uint32_t bm_off_vcpu, bm_off_ram;
    uint32_t bm_stride; // words per chunk row: 32 (conflict-free) or 64 (up to 64 thresholds; words 32 apart share a bank)
    uint32_t no_fused;  // test hook (RPK_FORCE_KERNEL=bitmap_grouped): small batches also take the three-launch path
    uint32_t no_persist; // test hook (RPK_FORCE_KERNEL=bitmap_grid): the first-generation (tile x segment) grid kernel
};
constexpr uint32_t kBmMaxStride = 64;
constexpr uint32_t kBmSegBytes = 65536;      // bit-sliced rows staged per CTA: 512 chunks (stride 32) or 256 (stride 64)
constexpr uint32_t kFusedRowsMax = 16384;    // up to this many rows one fused launch beats the multi-kernel paths
constexpr uint32_t kSmallBatch = 4096;       // rows: the host entry point's single-copy latency path
// transposed bit-sliced view (persistent kernel): the chunk axis is cut into 64-chunk sub-ranges; sub-range s holds
// bm_words rows of kSubStride words -- word (threshold i, chunk 64 s + k) at bmT[(s * bm_words + i) * kSubStride + k].
// 68 = 64 + 4: consecutive threshold rows start 4 words (one 16-byte bank group) apart, so an LDS.128 whose lanes
// read up to 8 different threshold rows at the same chunk offset is conflict-free.
constexpr uint32_t kSubChunks = 64;
constexpr uint32_t kSubStride = 68;
constexpr uint32_t kMaxClasses = 4096;       // row classes (cloud x thresholds) the pod-side counting sort distinguishes
// control words of the persistent select (Lane::hdr)
// (words 0..3 are written before the grid kernel starts; RowsDone is polled while it runs and sits on a cache line of
// its own; Pushed counts CTAs in the push tail; the queue cursors start on the next line)
enum : uint32_t { kHdrRows0 = 0, kHdrRows1 = 1, kHdrWork0 = 2, kHdrWork1 = 3, kHdrRowsDone = 32, kHdrPushed = 64,
                  kHdrCursors = 96 };

struct OfferView {       // one per cloud, all arrays in price-sorted order, length Gpad
    uint32_t* packed = nullptr;
    uint32_t* bitmap = nullptr;  // [Gpad/32][bm_stride]
    uint32_t* bitmapT = nullptr; // [nsub][bm_words][kSubStride] (transposed, see kSubChunks)
    int4* wide = nullptr;     // (mem_gb, vcpu, ram_gb, offer index)
    double* price = nullptr;  // NaN when the offer is not available in this cloud / padding
    int32_t* perm = nullptr;  // offer index, -1 when unavailable / padding
};

struct SelectArgs {
    // pod columns of this shard (device); nullable ones follow the C-ABI defaults
    const int32_t* req_mem;
    const int32_t* req_vcpu;
    const int32_t* req_ram;
    const double* max_price;
    const uint8_t* cloud;
    uint32_t P;
    // offer views
    OfferView view[2];
    uint32_t G, Gpad;
    const int32_t* distinct[3];
    uint32_t D[3];
    PackLayout pk;
    // per-call scratch
    uint32_t* rw;        // [P] packed thresholds
    uint32_t* order;     // [kGroups][P] row indices per group
    uint32_t* pos;       // [P] best sorted position so far (atomicMin target)
    uint32_t* counts;    // [kGroups] rows per group          } zero between calls: the grid kernel's last CTAs
    uint32_t* done;      // [1] row tiles finished             } clear them again (finish_tile), so no memset is
    uint32_t* tile_ctr;  // [ntiles] CTAs arrived per row tile } launched per call
    // outputs: the shard's slice is written into every peer's full-length vector at row0
    int32_t* best_out[RPK_MAX_GPUS];
    int n_out;
    int self_out;        // which of best_out lives on this GPU: the select kernels store there only and k_gather_push copies
                         // the slice to the peers in 16-byte NVLink stores; -1 = unknown, the kernels store to every vector
    uint32_t row0;
    int32_t* top5;       // [P*5] local, nullable
    // persistent bit-sliced path (kind 4, batches above the fused kernel's size)
    uint32_t nsub;       // 64-chunk sub-ranges of the transposed view
    uint16_t* key;       // [P] row class (0xFFFF: neither cloud)
    uint2* ord_rw;       // [P] {row id, threshold word} in class order (pos[] is indexed the same way): ONE scattered store per row
    uint32_t* hist;      // [kMaxClasses] rows per class       } zero between calls (k_pod_classify's last block)
    uint32_t* cursor;    // [kMaxClasses] class write cursors
    uint32_t* hdr;       // control words, kHdr*
    // peer flags bound with rpk_peer_bind: the warp that finishes the last push signals every peer (n_flags = 0: none)
    uint32_t* flags[RPK_MAX_GPUS];
    int n_flags, my_rank;
    int inline_wait;     // the signalling warp also waits for every peer's signal (rpk_peer_inline_wait)
    uint32_t tune_natural_order;  // tuning hook (RPK_TUNE=order=natural): row tiles in group order instead of heaviest first
};

struct StatusArgs {
    const uint8_t* records;
    uint32_t stride;
    uint32_t N;
    uint64_t* hash_prev;    // updated in place
    uint64_t* hash_out;     // nullable
    uint32_t* changed_idx;  // nullable (seed, or a sharded sweep that only fills the exchange buffers)
    uint16_t* changed_code; // nullable: translateRunPodStatus code per changed slot (rpk.h RPK_CODE_*)
    uint32_t* n_changed;    // nullable (seed)
    uint32_t idx_base;      // added to emitted indices (shard offset)
    unsigned long long* tile_state;  // look-back state: one entry per CTA (strides 16/32) or per tile (other strides); zero between calls
    uint32_t* tile_counter;          // [2] scheduling ticket, finished CTAs; zero between calls
    uint32_t* stage_idx;             // [N] per-warp ordered index segments (strides 16/32)
    uint16_t* stage_code;            // [N] codes staged alongside
    uint32_t* unit_cnt;              // [N / 64 + 1] changed slots per 64-slot unit (strides 16/32)
    // sharded sweep: the changed list also goes into region `my_rank` of every rank's exchange buffer
    int n_out, my_rank;
    uint32_t* out_idx[RPK_MAX_GPUS];    // start of this rank's index region in rank o's buffer
    uint16_t* out_code[RPK_MAX_GPUS];   // ... code region (nullable)
    uint32_t* out_count[RPK_MAX_GPUS];  // rank o's count words (one per source rank)
    uint32_t* flags[RPK_MAX_GPUS];      // bound peer flags: the CTA that finishes last signals (n_flags = 0: none)
    int n_flags, inline_wait;
};

// launchers (each returns the number of kernels it launched, or throws CudaError)
struct CudaError { cudaError_t err; const char* what; const char* file; int line; };
#define RPK_CUDA(x) do { cudaError_t e__ = (x); if (e__ != cudaSuccess) throw ::rpk::CudaError{e__, #x, __FILE__, __LINE__}; } while (0)

struct OfferIngest {   // raw device columns in, views out
    uint32_t G;
    const int32_t* mem; const int32_t* vcpu; const int32_t* ram;  // vcpu/ram never null here (zero-filled)
    const double* secure_price; const double* community_price; const uint8_t* flags;
};

struct DeviceState;
struct OfferTable;
int launch_offer_ingest(DeviceState& ds, OfferTable& t, const OfferIngest& in, cudaStream_t st);
// offer sets (offers.cu): member lists of n_sets sets from their membership words (W = ceil(G/32) per set) and one
// sub-table per non-empty set; counts[s] = members of set s (computed by the caller from the same words)
int launch_offer_sets_build(DeviceState& ds, uint32_t n_sets, const uint32_t* d_words, const uint32_t* counts, cudaStream_t st);
// offer sets (sets.cu): partition of pod rows by set id and the write-back in row order
struct SetPartitionArgs {
    uint32_t P, n_sets;             // bins: 0..n_sets-1 the sets, n_sets = RPK_SET_ALL, n_sets+1 = out of range
    const uint16_t* set_id;
    const int32_t* req_mem; const int32_t* req_vcpu; const int32_t* req_ram; const double* max_price; const uint8_t* cloud;
    int32_t* o_mem; int32_t* o_vcpu; int32_t* o_ram; double* o_price; uint8_t* o_cloud;  // partitioned copies (present columns)
    uint32_t* rows;                 // [P] row id of partitioned position i
    uint32_t* hist;                 // [n_sets + 2] rows per bin, then [n_sets + 2] write cursors (zeroed by the caller)
};
int launch_set_partition(const SetPartitionArgs& a, cudaStream_t st);
int launch_set_unpermute(uint32_t P, const uint32_t* rows, const int32_t* tmp_best, const int32_t* tmp_top5, int32_t* best,
                         int32_t* top5, cudaStream_t st);
struct PersistPlan;
int launch_select(const SelectArgs& a, int rows_per_warp, const PersistPlan* pl, cudaStream_t st);
uint32_t select_tiles_max(uint32_t P, int rows_per_warp);
int pick_rows_per_warp(uint32_t P, int sm_count);
int pick_rows_per_lane(uint32_t P, uint32_t G, int sm_count);
int launch_status_diff(const StatusArgs& a, cudaStream_t st);
struct PeerFenceArgs { uint32_t* flags[RPK_MAX_GPUS]; int n; int my_rank; uint32_t epoch; };
int launch_peer_fence(const PeerFenceArgs& a, cudaStream_t st);
int launch_peer_signal(const PeerFenceArgs& a, uint32_t word0, cudaStream_t st);
int launch_peer_wait(const PeerFenceArgs& a, uint32_t what, cudaStream_t st);
// persistent bit-sliced select (select_persist.cu)
struct PersistPlan { uint32_t cap_subs, S, per, qspan, Qi, grid, smem_bytes; int rpl, minb; };
bool persist_plan(const SelectArgs& a, int sm_count, PersistPlan* pl);
uint32_t persist_hdr_words(uint32_t G, uint32_t bm_words);
int launch_select_persist(const SelectArgs& a, const PersistPlan& pl, cudaStream_t st);
uint32_t status_tiles(uint32_t N, uint32_t stride);
uint32_t status_state_words(uint32_t N, uint32_t stride, int sm_count);
int launch_status_seed_slots(uint32_t n, const uint32_t* d_slots, const uint8_t* d_records, uint32_t stride, uint64_t* hash_prev,
                             uint32_t lo, uint32_t hi, cudaStream_t st);

template <typename T>
struct DevBuf {  // grow-only device buffer
    T* p = nullptr;
    size_t cap = 0;
    void reserve(size_t n) {
        if (n <= cap) return;
        if (p) RPK_CUDA(cudaFree(p));
        p = nullptr; cap = 0;
        size_t want = n + n / 4 + 256;
        RPK_CUDA(cudaMalloc(&p, want * sizeof(T)));
        cap = want;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// The views of one offer table as the select kernels consume them: the resident table, or the sub-table of an offer
// set (whose perm / wide.w hold global offer ids, so the kernels emit global indices directly).
struct OfferTable {
    uint32_t G = 0, Gpad = 0;
    DevBuf<uint32_t> v_packed[2]; DevBuf<uint32_t> v_bitmap[2]; DevBuf<uint32_t> v_bitmapT[2]; uint32_t nsub = 0; DevBuf<int4> v_wide[2]; DevBuf<double> v_price[2]; DevBuf<int32_t> v_perm[2];
    DevBuf<int32_t> distinct[3];
    uint32_t D[3] = {0, 0, 0};
    PackLayout pk = {};
    void release() {
        for (int c = 0; c < 2; ++c) { v_packed[c].release(); v_bitmap[c].release(); v_bitmapT[c].release(); v_wide[c].release(); v_price[c].release(); v_perm[c].release(); }
        for (int d = 0; d < 3; ++d) distinct[d].release();
        G = Gpad = nsub = 0;
    }
};

struct DeviceState {
    int dev = -1;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    // offer table
    OfferTable main;
    bool offers_ready = false;
    uint64_t table_version = 0;  // bumped by every rpk_offers_upload
    DevBuf<int32_t> raw_mem, raw_vcpu, raw_ram; DevBuf<double> raw_sp, raw_cp; DevBuf<uint8_t> raw_flags;
    DevBuf<unsigned long long> sort_keys; DevBuf<uint32_t> sort_vals;  // shared by every ingest (resident table and sets)
    DevBuf<uint32_t> dcount;
    int force_kind = 0;  // RPK_FORCE_KERNEL (tests): 0 auto, 1 generic, 2 packed+select, 3 packed+pos, 4 bit-sliced
    // offer sets: one sub-table per set (G = 0 for an empty set: never selected against), valid while
    // sets_version == table_version
    std::vector<OfferTable> sets;
    bool sets_ready = false;
    uint64_t sets_version = 0;
    DevBuf<uint32_t> set_words, set_members;  // membership words as uploaded; ascending member lists, set after set
    DevBuf<int32_t> set_mem, set_vcpu, set_ram; DevBuf<double> set_sp, set_cp; DevBuf<uint8_t> set_flags;  // gathered raw columns
    // rpk_select_sets scratch: partitioned pod columns, row ids, bin counts, results in partitioned order; host path staging
    struct SetSelect {
        DevBuf<int32_t> p_mem, p_vcpu, p_ram; DevBuf<double> p_price; DevBuf<uint8_t> p_cloud;
        DevBuf<uint32_t> rows, hist; DevBuf<int32_t> tmp_best, tmp_top5;
        DevBuf<int32_t> in_mem, in_vcpu, in_ram; DevBuf<double> in_price; DevBuf<uint8_t> in_cloud; DevBuf<uint16_t> in_set;
        DevBuf<int32_t> out_best, out_top5;
        uint32_t* h_counts = nullptr;  // pinned: bin counts read back once per call
        void release() {
            p_mem.release(); p_vcpu.release(); p_ram.release(); p_price.release(); p_cloud.release(); rows.release(); hist.release();
            tmp_best.release(); tmp_top5.release(); in_mem.release(); in_vcpu.release(); in_ram.release(); in_price.release();
            in_cloud.release(); in_set.release(); out_best.release(); out_top5.release();
            if (h_counts) cudaFreeHost(h_counts);
            h_counts = nullptr;
        }
    } ss;
    // select scratch.  The host entry point pipelines row sub-batches over four lanes (stream + staging +
    // scratch each) so that the H2D of one sub-batch, the kernels of another and the D2H of a third overlap;
    // the device entry points use lane 0's scratch on the caller's stream.
    struct Lane {
        cudaStream_t stream = nullptr;
        cudaEvent_t done = nullptr;
        DevBuf<int32_t> p_req_mem, p_req_vcpu, p_req_ram; DevBuf<double> p_max_price; DevBuf<uint8_t> p_cloud;
        DevBuf<int32_t> top5;
        DevBuf<uint32_t> rw, order, pos, ctrs;
        DevBuf<uint16_t> key; DevBuf<uint2> ord_rw; DevBuf<uint32_t> hist, cursor, hdr;  // persistent path
        bool ctrs_dirty = false;  // a select on this lane failed between its launches: re-zero the counters before the next one
        bool persist_dirty = false;
        void release() {
            p_req_mem.release(); p_req_vcpu.release(); p_req_ram.release(); p_max_price.release(); p_cloud.release();
            top5.release(); rw.release(); order.release(); pos.release(); ctrs.release();
            key.release(); ord_rw.release(); hist.release(); cursor.release(); hdr.release();
        }
    };
    static constexpr int kLanes = 4;  // one per sub-batch of a 1M-row call: no upload ever waits for a kernel to free its buffers
    Lane lane[kLanes];
    DevBuf<int32_t> best_full;
    // small-batch (latency) path: one pinned staging block in, one out
    unsigned char* h_small = nullptr; DevBuf<unsigned char> d_small_in; DevBuf<int32_t> d_small_out;
    // status
    DevBuf<uint8_t> s_records; DevBuf<uint64_t> s_hash_prev, s_hash_out; DevBuf<uint32_t> s_changed, s_misc;
    DevBuf<unsigned long long> s_tile_state; DevBuf<uint32_t> s_stage_idx; DevBuf<uint16_t> s_stage_code, s_changed_code; DevBuf<uint32_t> s_unit_cnt;
    DevBuf<uint32_t> s_seed_slots; DevBuf<uint8_t> s_seed_recs;
    unsigned char* h_changed = nullptr; unsigned char* d_changed_map = nullptr; size_t h_changed_cap = 0;  // mapped pinned: count, indices, codes
    cudaStream_t status_stream = nullptr;  // rpk_tick: the sweep next to the selection
    // device entry points: the stream that last used the select / status scratch, and its completion event
    cudaStream_t sel_last_stream = nullptr, st_last_stream = nullptr;
    cudaEvent_t ev_sel = nullptr, ev_st = nullptr;
    bool status_dirty = false;             // a status launch failed midway: re-zero the look-back state before the next one
    uint32_t statusN = 0; bool status_sized = false;
};

}  // namespace rpk
