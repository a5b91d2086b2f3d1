/*
 * rpk.h -- C-ABI of the B200 batch scheduling engine ("rpk") for the RunPod virtual kubelet.
 *
 * This is the whole drop-in boundary: what a cgo binding under pkg/virtual_kubelet calls in place of
 * the two Go loop bodies on the hot path (INTEGRATION.md shows the binding):
 *
 *   reference (paths relative to /root/reference/pkg/virtual_kubelet/)        replaced by
 *   ------------------------------------------------------------------------  ---------------------
 *   Client.GetGPUTypes filter loop          runpod_client.go:465-495          rpk_offers_upload +
 *   sort.Slice by price + take <=5          runpod_client.go:497-509          rpk_select
 *   per-pod call site                        runpod_client.go:1281             (one call per batch of pods)
 *   updateAllPodStatuses diff predicate      kubelet.go:857-880                rpk_status_diff
 *   previous-state table (InstanceInfo)      runpod_client.go:98-109,          device-resident hash column,
 *                                            kubelet.go:41-45                  rpk_status_seed / _reset
 *
 * Conventions
 *   - plain C, no torch / C++ types; every pointer is CALLER-OWNED memory borrowed for the duration of
 *     the call only (cgo pointer rule: C must not retain Go pointers).  Device memory is ctx-owned.
 *   - return value 0 = ok, <0 = error code below; never aborts, never throws across the boundary; the
 *     message is available from rpk_last_error().
 *   - a ctx is NOT re-entrant: serialise calls on one ctx (the Go wrapper holds a mutex -- at least four
 *     goroutines can reach it: kubelet.go:384, 718, 292, 734).  Every call binds its CUDA device itself
 *     (goroutines migrate between OS threads).
 *   - there is NO CPU fallback: without a usable sm_100 device rpk_create fails and the provider must
 *     refuse to start.
 *   - "host" entry points take host pointers (pageable or pinned; pinned from rpk_host_alloc is faster);
 *     "_device" entry points take device pointers on the shard's GPU and enqueue on the given stream
 *     without synchronising it.
 */
#ifndef RPK_H_
#define RPK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RPK_ABI_VERSION 2

#define RPK_OK 0
#define RPK_EINVAL (-1)  /* bad argument (NULL, size, INT32_MAX in an offer column, ...) */
#define RPK_ECUDA (-2)   /* a CUDA call failed; message has the CUDA error string */
#define RPK_ENOMEM (-3)  /* host or device allocation failed */
#define RPK_ESTATE (-4)  /* call order: select before offers_upload, diff with other N than reset, ... */
#define RPK_ENODEV (-5)  /* no usable sm_100 device */

/* cloud column values: validateCloudType's result (runpod_client.go:1115-1134).  Any other byte behaves
 * like a cloudType string that is neither (runpod_client.go:469-475): nothing is feasible. */
#define RPK_CLOUD_SECURE 0
#define RPK_CLOUD_COMMUNITY 1

/* flags column bits: GPUType.SecureCloud / GPUType.CommunityCloud (runpod_client.go:87,89) */
#define RPK_FLAG_SECURE_CLOUD 1u
#define RPK_FLAG_COMMUNITY_CLOUD 2u

#define RPK_TOPK 5              /* "Take up to 5 GPUs", runpod_client.go:502-509 */
#define RPK_DEFAULT_MAX_PRICE 0.5 /* DefaultMaxPrice, runpod_client.go:48 */
#define RPK_MAX_GPUS 8

typedef struct rpk_ctx rpk_ctx;

typedef struct rpk_stats {
    uint64_t select_calls;        /* rpk_select + rpk_select_device (+ the _sets variants) */
    uint64_t offer_scores;        /* sum of P*G over those calls (sets: sum of P_s*G_s, the grid evaluated) */
    uint64_t status_calls;
    uint64_t status_records;      /* sum of N */
    float last_select_kernel_ms;  /* 0: rpk_select overlaps copies and kernels (sub-batch pipeline), only the total is meaningful */
    float last_select_total_ms;   /* rpk_select: H2D + kernels + D2H of the last call (0 on the micro-batch latency path) */
    float last_status_kernel_ms;
    float last_status_total_ms;
    uint32_t select_kernel_kind;  /* 0 none, 1 generic int32 compare, 2 packed rank fields + select,
                                     3 packed + embedded position (min), 4 bit-sliced threshold masks */
    uint32_t n_gpus;
    uint32_t distinct_mem, distinct_vcpu, distinct_ram; /* distinct offer values found at upload */
    uint32_t packed_bits;         /* bits used by the packed offer word incl. guards (<=32), 0 if generic */
} rpk_stats;

/* ---- lifecycle ------------------------------------------------------------------------------------ */

/* n_gpus in [1, RPK_MAX_GPUS]; device_ids == NULL means 0..n_gpus-1.  With n_gpus > 1 (one host process
 * driving a whole box, the shape a Go kubelet has) pod rows / status slots are split into contiguous
 * shards, one per GPU, and every GPU writes its shard of the assignment vector straight into all peers'
 * copies over NVLink (peer access is enabled here). */
int rpk_create(int n_gpus, const int* device_ids, rpk_ctx** out);
void rpk_destroy(rpk_ctx* ctx);
/* ctx-owned string, valid until the next call on that ctx; ctx == NULL returns the last rpk_create error
 * of the calling thread. */
const char* rpk_last_error(const rpk_ctx* ctx);
int rpk_abi_version(void);

/* pinned host memory for callers that want full-speed H2D/D2H (Go: C.rpk_host_alloc-backed slices) */
void* rpk_host_alloc(size_t bytes);
void rpk_host_free(void* p);

/* ---- offer table: []GPUType as struct-of-arrays (runpod_client.go:83-95) ------------------------- */

/* Copies the G-row table to every GPU of the ctx and prepares the two per-cloud views (sorted by price,
 * ties by offer index) the select kernels consume.  vcpu / ram_gb may be NULL (= all 0: the reference has
 * no such fields).  Prices are the Go float64 values, compared with IEEE semantics on the device
 * (price > 0 && price < maxPrice, runpod_client.go:478).  mem_gb/vcpu/ram_gb must be < INT32_MAX.
 * Replaces the per-pod GraphQL decode of the same table (runpod_client.go:447-455). */
int rpk_offers_upload(rpk_ctx* ctx, uint32_t G, const int32_t* mem_gb, const int32_t* vcpu, const int32_t* ram_gb,
                      const double* secure_price, const double* community_price, const uint8_t* flags);

/* ---- selection: P pods x G offers ----------------------------------------------------------------- */

/* For pod row p: feasible(g) = cloud ok && price > 0 && price < max_price[p] && mem_gb[g] >= req_mem_gb[p]
 * && vcpu[g] >= req_vcpu[p] && ram_gb[g] >= req_ram_gb[p]; best[p] = the feasible offer with the lowest
 * price, ties to the lowest offer index, or -1 (an empty gpuTypeIds is not an error,
 * runpod_client.go:511-517).  top5 (nullable, P*5, -1 padded) is the whole gpuTypeIds list in order.
 * NULL req_vcpu / req_ram_gb = 0; NULL max_price = 0.5 for every pod (the reference's only behaviour,
 * runpod_client.go:1281); NULL cloud = SECURE.  P == 0 is a no-op. */
int rpk_select(rpk_ctx* ctx, uint32_t P, const int32_t* req_mem_gb, const int32_t* req_vcpu,
               const int32_t* req_ram_gb, const double* max_price, const uint8_t* cloud, int32_t* best,
               int32_t* top5);

/* Same on device-resident columns of GPU `shard` (index into the ctx's device list), enqueued on `stream`
 * (a cudaStream_t; NULL = the ctx's own stream for that shard; pass cudaStreamLegacy (0x1) for the legacy
 * default stream).  Does not synchronise.  d_best must hold
 * P int32; d_top5 is nullable.  Used by one-process-per-GPU callers that shard pod rows themselves. */
int rpk_select_device(rpk_ctx* ctx, int shard, uint32_t P, const int32_t* d_req_mem_gb, const int32_t* d_req_vcpu,
                      const int32_t* d_req_ram_gb, const double* d_max_price, const uint8_t* d_cloud,
                      int32_t* d_best, int32_t* d_top5, void* stream);

/* Shard + all-gather: the shard's P results end up at [row0, row0+P) of EVERY vector in d_best_full[0..n_out)
 * -- the caller's own full-length vector and its peers' (peer-mapped device pointers: cudaDeviceEnablePeerAccess
 * in one process, cudaIpcOpenMemHandle across processes).  The select kernels write the vector that lives on
 * GPU `shard`; a copy kernel launched behind them pushes the finished slice into the other vectors with 16-byte
 * stores over NVLink, so no collective follows; the caller only needs a barrier (rpk_peer_fence) before reading
 * a peer-written vector.  All vectors must share the slice's 16-byte alignment (same offset from cudaMalloc'ed
 * bases); if none of them lives on GPU `shard`, or the alignments differ, every result is stored into all
 * vectors directly from the select epilogue instead (slower, same result).  After one call of a given size the
 * function only enqueues launches, so it can be captured in a CUDA graph. */
int rpk_select_device_gather(rpk_ctx* ctx, int shard, uint32_t P, const int32_t* d_req_mem_gb,
                             const int32_t* d_req_vcpu, const int32_t* d_req_ram_gb, const double* d_max_price,
                             const uint8_t* d_cloud, int n_out, int32_t* const* d_best_full, uint32_t row0,
                             int32_t* d_top5, void* stream);

/* Cross-process peer vectors for one-process-per-GPU callers (torchrun-style): allocate a plain cudaMalloc
 * buffer on GPU `shard` and export its 64-byte CUDA IPC handle; another process opens the handle and gets a
 * device pointer it can pass in d_best_full[] of rpk_select_device_gather (peer access over NVLink is
 * enabled by the open).  Buffers/mappings are released by rpk_ipc_free / rpk_ipc_close or rpk_destroy. */
int rpk_ipc_alloc(rpk_ctx* ctx, int shard, size_t bytes, void** d_ptr, unsigned char handle_out[64]);
int rpk_ipc_open(rpk_ctx* ctx, int shard, const unsigned char handle[64], void** d_peer_ptr);
int rpk_ipc_close(rpk_ctx* ctx, int shard, void* d_peer_ptr);
int rpk_ipc_free(rpk_ctx* ctx, int shard, void* d_ptr);

/* Cross-GPU fence for the fused gather (one tiny kernel, no NCCL): lane r stores `epoch` into rank r's flag
 * array at index my_rank (system-scope fence first, so every peer store issued by earlier work of this stream
 * -- the gather's NVLink stores -- is visible before the flag), then spins until its own flag array
 * shows `epoch` from every rank.  d_flags[r] is rank r's array of >= n uint32 (zero-initialised,
 * rpk_ipc_alloc'ed and rpk_ipc_open'ed like the vectors); epochs must increase by one per fence.
 * epoch = 0 selects the self-counting mode: the kernel keeps the count in word 32 of the rank's own array
 * (arrays of >= 33 words), so the launch has no per-call argument and can be captured in a CUDA graph and
 * replayed; all ranks of a group must use the same mode for the life of the arrays. */
int rpk_peer_fence(rpk_ctx* ctx, int shard, int n, uint32_t* const* d_flags, int my_rank, uint32_t epoch, void* stream);

/* Split fence for the fused gather.  rpk_peer_bind registers the N flag arrays of a peer group with GPU `shard` of
 * this ctx (d_flags[r] = rank r's array of >= 64 uint32, zero-initialised, rpk_ipc_alloc'ed / rpk_ipc_open'ed like the
 * vectors; n = 0 unbinds).  While bound, every rpk_select_device_gather on that shard with n_out > 1 SIGNALS by itself:
 * the warp that pushes the last block of the slice (or a one-warp kernel behind the copy kernel on the small-batch
 * paths, or behind nothing for an empty shard) bumps the rank's select epoch (word 32 of its own array) and stores it
 * into word `my_rank` of every peer's array, after a system-scope fence.  rpk_status_diff_device_gather does the same
 * with the status epoch (word 33, flag words 8 + my_rank).  rpk_peer_wait enqueues the other half: one warp that
 * spins until every rank's flag shows this rank's own current epoch (what: bit 0 = select, bit 1 = status sweep;
 * all ranks of a group must issue the same sequence of gathers).  Launches carry no per-call value, so a step can be
 * captured in a CUDA graph and replayed.  Do not mix rpk_peer_fence and the bound mode on the same arrays (both use
 * words 0..7 and 32).
 * Ordering given: a peer's results are visible after the wait.  NOT given: once rank A has passed the wait of step e it
 * may run step e+1 and overwrite its slice of rank B's vector while B still reads step e -- consumers that read the
 * vector every step alternate between two sets of vectors (even / odd steps), as bench.py does. */
int rpk_peer_bind(rpk_ctx* ctx, int shard, int n, uint32_t* const* d_flags, int my_rank);
int rpk_peer_wait(rpk_ctx* ctx, int shard, unsigned what, void* stream);
/* on != 0: the warp that signals also WAITS (spins on its own flag words) until every rank of the group has signalled
 * the same epoch, so a bound gather only completes once all peers' results have landed and no rpk_peer_wait launch is
 * needed (one kernel boundary less per step).  All ranks of a group must use the same setting.  A host thread that
 * drives SEVERAL shards of a group must enable it only after one call of each size has sized the scratch: a call that
 * allocates synchronises its device, which would wait for a kernel that waits for a peer not launched yet. */
int rpk_peer_inline_wait(rpk_ctx* ctx, int shard, int on);

/* ---- offer sets: restrict a pod to a list of offers (runpod.io/gpu-type-ids) ------------------------ */

/* An offer set is a sub-table: a pod restricted to set s gets exactly what rpk_select would give it against a table
 * holding only the members of s, in their relative order -- same filter, same price order with ties to the lowest
 * GLOBAL offer index, same <= 5 list -- and the indices returned are global offer indices. */
#define RPK_MAX_OFFER_SETS 256
#define RPK_SET_ALL 0xFFFFu   /* set_id value: unrestricted (the whole table, = rpk_select) */

/* Set s = offers g of the resident table with bit (g & 31) of members[s*W + g/32] set, W = ceil(G/32); bits >= G are
 * ignored.  G must equal the resident table's G (RPK_EINVAL otherwise).  Replaces all previous sets; n_sets = 0 clears
 * them.  Built on every GPU of the ctx.  A later rpk_offers_upload makes the sets stale: rpk_select_sets then fails with
 * RPK_ESTATE until the sets are uploaded again (indices would otherwise refer to another table). */
int rpk_offer_sets_upload(rpk_ctx* ctx, uint32_t n_sets, uint32_t G, const uint32_t* members);

/* rpk_select with one more column: set_id[p] restricts pod p to set set_id[p].  RPK_SET_ALL = the whole table;
 * any other id >= n_sets behaves like an empty set (best -1, top5 all -1), the same convention as an unknown cloud byte.
 * NULL set_id = every row RPK_SET_ALL = rpk_select's result (no sets need to be uploaded for that).  Does not write the
 * device-resident full vector (rpk_best_device_ptr keeps the last rpk_select's). */
int rpk_select_sets(rpk_ctx* ctx, uint32_t P, const int32_t* req_mem_gb, const int32_t* req_vcpu, const int32_t* req_ram_gb,
                    const double* max_price, const uint8_t* cloud, const uint16_t* set_id, int32_t* best, int32_t* top5);
/* Device-resident variant on GPU `shard`.  It reads back the per-set row counts once, so it synchronises `stream` once
 * and cannot be captured in a CUDA graph: on a capturing stream it returns RPK_ESTATE before enqueuing anything (with
 * d_set_id NULL it only enqueues, like rpk_select_device, and may be captured).  Shares the
 * shard's select scratch with rpk_select_device (see rpk_status_diff_device). */
int rpk_select_sets_device(rpk_ctx* ctx, int shard, uint32_t P, const int32_t* d_req_mem_gb, const int32_t* d_req_vcpu,
                           const int32_t* d_req_ram_gb, const double* d_max_price, const uint8_t* d_cloud,
                           const uint16_t* d_set_id, int32_t* d_best, int32_t* d_top5, void* stream);

/* Device pointer of GPU `shard`'s copy of the full assignment vector written by the last rpk_select
 * (ctx-owned; every GPU of the ctx holds the whole vector after the call). */
const int32_t* rpk_best_device_ptr(const rpk_ctx* ctx, int shard);

/* ---- status sweep diff ------------------------------------------------------------------------------ */

/* records: N slots of `stride` bytes (stride a multiple of 16, 16..256):
 *   [b0][status ASCII][0x00][ports_exposed:u8][zero pad],  b0 = len | flag << 7,  len = strlen(status)+2 <= min(stride-1, 127)
 * i.e. exactly the two fields compared at kubelet.go:870-871.  A slot's 64-bit XXH64 (seed 0) over its zero-padded
 * prefix in whole 8-byte lanes -- bytes [0, 8*ceil((1+len)/8)), flag bit cleared: the length byte is inside, so the
 * value is self-delimiting and does not depend on the stride -- is compared with the hash kept on the device from the
 * previous call; slots that differ (or have never been seen) are returned ascending in changed_idx[0..*n_changed)
 * (capacity N) and their stored hash is replaced (kubelet.go:875-880).  hashes_out (nullable, N) receives the new hash
 * column.  The flag bit is the host's "statusMessage contains error/fail" (kubelet.go:1907-1908): not a compared field,
 * not hashed, only used by the codes below.  Strides 16 (status <= 13 chars: every RunPod status) and 32 take the
 * streaming kernel; wider strides exist for longer strings. */
int rpk_status_diff(rpk_ctx* ctx, uint32_t N, const uint8_t* records, uint32_t stride, uint32_t* changed_idx,
                    uint32_t* n_changed, uint64_t* hashes_out);

/* What translateRunPodStatus (kubelet.go:1848-2024) decides for a slot, as a 16-bit code -- emitted per CHANGED slot
 * next to its index, so the caller builds v1.PodStatus for the changed subset without touching the strings again:
 *   bits 2:0  phase      0 Unknown 1 Pending 2 Running 3 Succeeded 4 Failed
 *   bit  3    ready      containerStatus.Ready and the Ready / ContainersReady conditions (kubelet.go:1972-1975)
 *   bit  4    started    containerStatus.Started
 *   bits 6:5  state      0 Waiting 1 Running 2 Terminated
 *   bit  7    exit code  (0 / 1)
 *   bits 10:8 reason     0 none 1 ContainerCreating 2 Completed 3 Error 4 Terminated 5 PodDeleted 6 ContainerStatusUnknown
 *   bits 12:11 message   0 statusMessage  1 "Container reported as running but ports not yet exposed" (:1885)
 *                        2 "Pod was deleted from RunPod API" (:1963)  3 "Unknown RunPod status: <status>" (:1975) */
#define RPK_CODE_PHASE(c) ((c) & 7u)
#define RPK_CODE_READY(c) (((c) >> 3) & 1u)
#define RPK_CODE_STARTED(c) (((c) >> 4) & 1u)
#define RPK_CODE_STATE(c) (((c) >> 5) & 3u)
#define RPK_CODE_EXIT(c) (((c) >> 7) & 1u)
#define RPK_CODE_REASON(c) (((c) >> 8) & 7u)
#define RPK_CODE_MESSAGE(c) (((c) >> 11) & 3u)
/* rpk_status_diff + changed_code[0..*n_changed) (nullable = rpk_status_diff) */
int rpk_status_diff_codes(rpk_ctx* ctx, uint32_t N, const uint8_t* records, uint32_t stride, uint32_t* changed_idx,
                          uint16_t* changed_code, uint32_t* n_changed, uint64_t* hashes_out);

/* Load previous state without reporting (CreatePod / LoadRunning fill InstanceInfo the same way,
 * kubelet.go:393-400, 1380-1535). */
int rpk_status_seed(rpk_ctx* ctx, uint32_t N, const uint8_t* records, uint32_t stride);
/* ... of individual slots: records holds n_slots packed slots of `stride` bytes, records[i] becomes the previous state
 * of slot slots[i] (CreatePod writes ONE InstanceInfo, kubelet.go:391-401; handleMissingRunPodInstance rewrites one,
 * :976-1040).  Nothing else is touched, so a sweep whose records are already staged loses nothing. */
int rpk_status_seed_slots(rpk_ctx* ctx, uint32_t n_slots, const uint32_t* slots, const uint8_t* records, uint32_t stride);
/* Forget all previous hashes and (re)size the table to N slots: every slot reports changed next time. */
int rpk_status_reset(rpk_ctx* ctx, uint32_t N);

/* One tick: rpk_select (P rows; P = 0 skips it) and rpk_status_diff_codes (N slots) enqueued together -- the two are
 * independent (processPendingPods kubelet.go:747-814, updateAllPodStatuses :816-974), so the sweep's upload follows the
 * selection's on the PCIe link while the selection's kernels run, every shard of a multi-GPU ctx is driven by its own
 * host thread, and the call synchronises once.  Argument meaning as in the two calls. */
int rpk_tick(rpk_ctx* ctx, uint32_t P, const int32_t* req_mem_gb, const int32_t* req_vcpu, const int32_t* req_ram_gb,
             const double* max_price, const uint8_t* cloud, int32_t* best, int32_t* top5, uint32_t N, const uint8_t* records,
             uint32_t stride, uint32_t* changed_idx, uint16_t* changed_code, uint32_t* n_changed);

/* Device-resident variant on GPU `shard`: d_records N*stride bytes, d_hash_prev N uint64 updated in place
 * (caller-owned column; 0 = never seen), d_changed_idx capacity N, d_n_changed one uint32.  Enqueued on
 * `stream`, no synchronisation.  The _device entry points of one shard share ctx-owned scratch: issue them from one
 * stream per shard (select) / one stream per shard (status) at a time. */
int rpk_status_diff_device(rpk_ctx* ctx, int shard, uint32_t N, const uint8_t* d_records, uint32_t stride,
                           uint64_t* d_hash_prev, uint32_t* d_changed_idx, uint32_t* d_n_changed, void* stream);
int rpk_status_diff_device_codes(rpk_ctx* ctx, int shard, uint32_t N, const uint8_t* d_records, uint32_t stride,
                                 uint64_t* d_hash_prev, uint32_t* d_changed_idx, uint16_t* d_changed_code,
                                 uint32_t* d_n_changed, void* stream);

/* Sharded sweep with exchange (one process per GPU): rank `my_rank` sweeps its N slots (global ids idx_base + i) and
 * writes its changed list -- count, ascending global ids, codes -- into region `my_rank` of EVERY rank's exchange buffer
 * d_xchg[0..n_ranks) (peer-mapped like the assignment vectors; each rpk_xchg_bytes(n_ranks, cap) bytes, cap >= any
 * rank's N), straight from the kernel's final copy over NVLink.  Layout of a buffer, in uint32 words:
 *   [0, 8) count per source rank | [8 + r*cap, ...) ids of rank r | then uint16 codes: region r at
 *   ((uint16*)(words + 8 + n_ranks*cap)) + r*cap.
 * With flags bound (rpk_peer_bind) the CTA that finishes last signals the status epoch; rpk_peer_wait(what = 2) on
 * every rank makes all regions readable.  Strides 16 and 32. */
size_t rpk_xchg_bytes(int n_ranks, uint32_t cap);
int rpk_status_diff_device_gather(rpk_ctx* ctx, int shard, uint32_t N, const uint8_t* d_records, uint32_t stride,
                                  uint64_t* d_hash_prev, uint32_t idx_base, int n_ranks, uint32_t* const* d_xchg, uint32_t cap,
                                  int my_rank, uint32_t* d_n_changed, void* stream);

int rpk_stats_get(const rpk_ctx* ctx, rpk_stats* out);

/* number of kernel launches issued by this ctx since creation (bench.py's gpu_launches) */
uint64_t rpk_launch_count(const rpk_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* RPK_H_ */
