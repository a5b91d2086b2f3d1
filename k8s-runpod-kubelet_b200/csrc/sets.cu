// sets.cu -- pod rows restricted to offer sets (rpk_select_sets): rows are partitioned by set id into one contiguous
// bin per set (plus RPK_SET_ALL and out-of-range), every non-empty bin runs the ordinary select against its set's
// sub-table, and the results go back to row order.  Partition: bin histogram -> exclusive scan -> scatter of the row ids
// and the present pod columns (one warp-aggregated cursor bump per distinct bin of a warp).
#include "rpk_internal.cuh"

namespace rpk {

constexpr uint32_t kMaxBins = RPK_MAX_OFFER_SETS + 2;

__device__ __forceinline__ uint32_t set_bin(uint16_t id, uint32_t n_sets) {
    return id == (uint16_t)RPK_SET_ALL ? n_sets : (id < n_sets ? (uint32_t)id : n_sets + 1);
}

__global__ void __launch_bounds__(256) k_set_hist(uint32_t P, uint32_t n_sets, const uint16_t* __restrict__ set_id,
                                                  uint32_t* __restrict__ hist) {
    __shared__ uint32_t sh[kMaxBins];
    const uint32_t nb = n_sets + 2;
    for (uint32_t b = threadIdx.x; b < nb; b += blockDim.x) sh[b] = 0;
    __syncthreads();
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < P; i += gridDim.x * blockDim.x)
        atomicAdd(&sh[set_bin(set_id[i], n_sets)], 1u);
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < nb; b += blockDim.x)
        if (sh[b]) atomicAdd(&hist[b], sh[b]);
}

// exclusive scan of the (<= 258) bin counts into the write cursors
__global__ void k_set_scan(uint32_t nb, uint32_t* __restrict__ hist) {
    if (threadIdx.x != 0) return;
    uint32_t run = 0;
    for (uint32_t b = 0; b < nb; ++b) { hist[nb + b] = run; run += hist[b]; }
}

__global__ void __launch_bounds__(256) k_set_scatter(SetPartitionArgs a) {
    const uint32_t lane = threadIdx.x & 31;
    uint32_t* cursor = a.hist + a.n_sets + 2;
    for (uint32_t base = blockIdx.x * blockDim.x; base < a.P; base += gridDim.x * blockDim.x) {
        const uint32_t i = base + threadIdx.x;  // the whole warp iterates: base is warp-uniform
        const bool valid = i < a.P;
        const uint32_t bin = valid ? set_bin(a.set_id[i], a.n_sets) : 0xFFFFFFFFu;
        const uint32_t peers = __match_any_sync(0xFFFFFFFFu, bin);
        const uint32_t leader = (uint32_t)__ffs(peers) - 1u;
        uint32_t b0 = 0;
        if (valid && lane == leader) b0 = atomicAdd(&cursor[bin], (uint32_t)__popc(peers));
        b0 = __shfl_sync(0xFFFFFFFFu, b0, (int)leader);
        if (!valid) continue;
        const uint32_t pos = b0 + (uint32_t)__popc(peers & ((1u << lane) - 1u));
        a.rows[pos] = i;
        a.o_mem[pos] = a.req_mem[i];
        if (a.req_vcpu) a.o_vcpu[pos] = a.req_vcpu[i];
        if (a.req_ram) a.o_ram[pos] = a.req_ram[i];
        if (a.max_price) a.o_price[pos] = a.max_price[i];
        if (a.cloud) a.o_cloud[pos] = a.cloud[i];
    }
}

__global__ void k_set_unpermute(uint32_t P, const uint32_t* __restrict__ rows, const int32_t* __restrict__ tmp_best,
                                const int32_t* __restrict__ tmp_top5, int32_t* __restrict__ best, int32_t* __restrict__ top5) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const uint32_t r = rows[i];
    best[r] = tmp_best[i];
    if (top5)
        for (int k = 0; k < RPK_TOPK; ++k) top5[(size_t)r * RPK_TOPK + k] = tmp_top5[(size_t)i * RPK_TOPK + k];
}

static uint32_t grid_for(uint32_t P, uint32_t cap) {
    const uint32_t g = (P + 255) / 256;
    return g < 1 ? 1 : g > cap ? cap : g;
}

int launch_set_partition(const SetPartitionArgs& a, cudaStream_t st) {
    const uint32_t nb = a.n_sets + 2;
    k_set_hist<<<grid_for(a.P, 148 * 4), 256, 0, st>>>(a.P, a.n_sets, a.set_id, a.hist);
    k_set_scan<<<1, 32, 0, st>>>(nb, a.hist);
    k_set_scatter<<<grid_for(a.P, 148 * 8), 256, 0, st>>>(a);
    RPK_CUDA(cudaGetLastError());
    return 3;
}

int launch_set_unpermute(uint32_t P, const uint32_t* rows, const int32_t* tmp_best, const int32_t* tmp_top5, int32_t* best,
                         int32_t* top5, cudaStream_t st) {
    k_set_unpermute<<<(P + 255) / 256, 256, 0, st>>>(P, rows, tmp_best, tmp_top5, best, top5);
    RPK_CUDA(cudaGetLastError());
    return 1;
}

}  // namespace rpk
