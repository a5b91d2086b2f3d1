// offers.cu -- offer-table ingest: []GPUType (reference runpod_client.go:83-95) -> two per-cloud views
// sorted by (price, offer index), which is the order sort.Slice + "ties to the lowest index" produces
// (runpod_client.go:497-500; tie contract in DESIGN.md).  Runs once per table refresh, entirely on the
// device: key build -> bitonic sort -> per-column distinct values (rank compression) -> pack.
#include <math_constants.h>

#include "rpk_internal.cuh"

namespace rpk {

using u64 = unsigned long long;
constexpr u64 kKeyMax = ~0ull;

// ---- sort keys -------------------------------------------------------------------------------------
// cloud view c keeps an offer iff cloudCheck && price > 0 (runpod_client.go:469-478; the price < maxPrice
// half of the test is per pod and is applied in the select epilogue).  For price > 0 the IEEE-754 bit
// pattern is monotone in the value, so sorting by it is sorting by price; NaN fails price > 0.
__global__ void k_offer_keys(uint32_t G, uint32_t n, const uint8_t* __restrict__ flags,
                             const double* __restrict__ sp, const double* __restrict__ cp, u64* __restrict__ keys,
                             uint32_t* __restrict__ vals) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u64 k0 = kKeyMax, k1 = kKeyMax;
    uint32_t v = kNone;
    if (i < G) {
        v = i;
        uint8_t f = flags[i];
        double a = sp[i], b = cp[i];
        if ((f & RPK_FLAG_SECURE_CLOUD) && a > 0.0) k0 = (u64)__double_as_longlong(a);
        if ((f & RPK_FLAG_COMMUNITY_CLOUD) && b > 0.0) k1 = (u64)__double_as_longlong(b);
    }
    keys[i] = k0; vals[i] = v;
    keys[n + i] = k1; vals[n + i] = v;
}

__global__ void k_dim_keys(uint32_t G, uint32_t n, const int32_t* __restrict__ col, u64* __restrict__ keys,
                           uint32_t* __restrict__ vals) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = i < G ? (u64)((uint32_t)col[i] ^ 0x80000000u) : kKeyMax;  // order-preserving int32 -> u32
    vals[i] = i;
}

// ---- bitonic sort of (key, val) pairs, ascending lexicographic, n a power of two >= 1024 --------------
__device__ __forceinline__ void cswap(u64& ka, uint32_t& va, u64& kb, uint32_t& vb, bool asc) {
    bool a_gt_b = ka > kb || (ka == kb && va > vb);
    if (a_gt_b == asc) { u64 tk = ka; ka = kb; kb = tk; uint32_t tv = va; va = vb; vb = tv; }
}

template <bool kFullSort>
__global__ void __launch_bounds__(512) k_bitonic_block(u64* __restrict__ keys, uint32_t* __restrict__ vals, uint32_t kk) {
    __shared__ u64 sk[1024];
    __shared__ uint32_t sv[1024];
    const uint32_t base = blockIdx.x * 1024u, t = threadIdx.x;
    sk[t] = keys[base + t]; sv[t] = vals[base + t];
    sk[t + 512] = keys[base + t + 512]; sv[t + 512] = vals[base + t + 512];
    __syncthreads();
    // kFullSort: all stages k = 2..1024; else only the tail j = 512..1 of stage kk
    for (uint32_t k = kFullSort ? 2u : kk; k <= (kFullSort ? 1024u : kk); k <<= 1) {
        for (uint32_t j = (k >> 1) > 512u ? 512u : (k >> 1); j >= 1; j >>= 1) {
            uint32_t i = 2 * t - (t & (j - 1));
            bool asc = ((base + i) & k) == 0;
            cswap(sk[i], sv[i], sk[i + j], sv[i + j], asc);
            __syncthreads();
        }
    }
    keys[base + t] = sk[t]; vals[base + t] = sv[t];
    keys[base + t + 512] = sk[t + 512]; vals[base + t + 512] = sv[t + 512];
}

__global__ void k_bitonic_global(u64* __restrict__ keys, uint32_t* __restrict__ vals, uint32_t n, uint32_t k, uint32_t j) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n / 2) return;
    uint32_t i = 2 * t - (t & (j - 1));
    bool asc = (i & k) == 0;
    u64 ka = keys[i], kb = keys[i + j];
    uint32_t va = vals[i], vb = vals[i + j];
    bool a_gt_b = ka > kb || (ka == kb && va > vb);
    if (a_gt_b == asc) { keys[i] = kb; keys[i + j] = ka; vals[i] = vb; vals[i + j] = va; }
}

static int bitonic_sort(u64* keys, uint32_t* vals, uint32_t n, cudaStream_t st) {
    int launches = 0;
    k_bitonic_block<true><<<n / 1024, 512, 0, st>>>(keys, vals, 0); ++launches;
    for (uint32_t k = 2048; k <= n && k != 0; k <<= 1) {
        for (uint32_t j = k >> 1; j >= 1024; j >>= 1) {
            k_bitonic_global<<<(n / 2 + 255) / 256, 256, 0, st>>>(keys, vals, n, k, j); ++launches;
        }
        k_bitonic_block<false><<<n / 1024, 512, 0, st>>>(keys, vals, k); ++launches;
    }
    return launches;
}

// ---- distinct values of a sorted column (single block, carries a running count) ---------------------
__global__ void __launch_bounds__(1024) k_unique(const u64* __restrict__ keys, uint32_t G, int32_t* __restrict__ distinct,
                                                 uint32_t* __restrict__ count) {
    __shared__ uint32_t warp_sum[32];
    __shared__ uint32_t carry;
    const uint32_t t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < G; base += 1024) {
        uint32_t i = base + t;
        bool head = i < G && (i == 0 || keys[i] != keys[i - 1]);
        uint32_t m = __ballot_sync(0xFFFFFFFFu, head);
        if (lane == 0) warp_sum[w] = __popc(m);
        __syncthreads();
        uint32_t off = 0;
        for (uint32_t x = 0; x < w; ++x) off += warp_sum[x];
        uint32_t total = 0;
        if (t == 0) for (uint32_t x = 0; x < 32; ++x) total += warp_sum[x];
        uint32_t my = carry + off + __popc(m & ((1u << lane) - 1));
        if (head) distinct[my] = (int32_t)((uint32_t)keys[i] ^ 0x80000000u);
        __syncthreads();
        if (t == 0) carry += total;
        __syncthreads();
    }
    if (t == 0) *count = carry;
}

// ---- pack the views ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t lower_bound_i32(const int32_t* __restrict__ a, uint32_t n, int32_t x) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) { uint32_t mid = (lo + hi) >> 1; if (a[mid] < x) lo = mid + 1; else hi = mid; }
    return lo;
}

struct PackArgs {
    uint32_t G, Gpad, n;
    const u64* keys; const uint32_t* vals;  // [2n] sorted, cloud c at c*n
    const int32_t* mem; const int32_t* vcpu; const int32_t* ram;
    const double* sp; const double* cp;
    const int32_t* distinct[3]; uint32_t D[3];
    PackLayout pk;
    uint32_t* packed[2]; int4* wide[2]; double* price[2]; int32_t* perm[2];
};

__global__ void k_offer_pack(PackArgs a) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    int c = blockIdx.y;
    if (s >= a.Gpad) return;
    uint32_t word = a.pk.guard;  // never feasible: mem field 0 < every pod threshold (>= 1)
    int4 w = make_int4(INT32_MIN, INT32_MIN, INT32_MIN, -1);
    double pr = CUDART_NAN;
    int32_t pm = -1;
    if (s < a.G) {
        u64 key = a.keys[(size_t)c * a.n + s];
        uint32_t i = a.vals[(size_t)c * a.n + s];
        if (key != kKeyMax) {
            int32_t m = a.mem[i], v = a.vcpu[i], r = a.ram[i];
            w = make_int4(m, v, r, (int)i);
            pr = c == 0 ? a.sp[i] : a.cp[i];
            pm = (int32_t)i;
            if (a.pk.bits) {
                uint32_t rm = lower_bound_i32(a.distinct[0], a.D[0], m) + 1;
                uint32_t rv = lower_bound_i32(a.distinct[1], a.D[1], v);
                uint32_t rr = lower_bound_i32(a.distinct[2], a.D[2], r);
                word = a.pk.guard | (rm << a.pk.sh_mem) | (rv << a.pk.sh_vcpu) | (rr << a.pk.sh_ram);
            }
        }
    }
    if (a.pk.pos_bits) word |= s & ((1u << a.pk.pos_bits) - 1);  // position inside the 2^pos_bits-offer segment
    a.packed[c][s] = word; a.wide[c][s] = w; a.price[c][s] = pr; a.perm[c][s] = pm;
}

// Bit-sliced view: one warp per 32-offer chunk of a cloud view; lane j holds offer j's ranks and the warp
// ballots one mask per threshold.
struct BitmapArgs {
    uint32_t G, nchunks, nchunks_real;
    const unsigned long long* keys; const uint32_t* vals; uint32_t n;  // sorted (key, offer index), cloud c at c*n
    const int32_t* mem; const int32_t* vcpu; const int32_t* ram;
    const int32_t* distinct[3]; uint32_t D[3];
    uint32_t off_vcpu, off_ram, words, stride;
    uint32_t* bitmap[2];
    uint32_t* bitmapT[2];  // transposed twin for the persistent kernel (zero-filled before this kernel runs)
};

__global__ void __launch_bounds__(256) k_offer_bitmap(BitmapArgs a) {
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int c = blockIdx.y;
    if (warp >= a.nchunks) return;
    const uint32_t s = warp * 32 + lane;
    uint32_t rm = 0, rv = 0, rr = 0;  // rank' of mem (0 = unavailable), ranks of vcpu / ram
    if (s < a.G && a.keys[(size_t)c * a.n + s] != kKeyMax) {
        const uint32_t i = a.vals[(size_t)c * a.n + s];
        rm = lower_bound_i32(a.distinct[0], a.D[0], a.mem[i]) + 1;
        rv = lower_bound_i32(a.distinct[1], a.D[1], a.vcpu[i]);
        rr = lower_bound_i32(a.distinct[2], a.D[2], a.ram[i]);
    }
    uint32_t* row = a.bitmap[c] + (size_t)warp * a.stride;
    for (uint32_t w = 0; w < a.stride; ++w) {
        bool bit = false;
        if (w < a.off_vcpu) bit = rm >= w + 1;                       // mem threshold t' = w+1
        else if (w < a.off_ram) bit = rm != 0 && rv >= w - a.off_vcpu;  // vcpu threshold t = w - off
        else if (w < a.words) bit = rm != 0 && rr >= w - a.off_ram;
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, bit);
        if (lane == 0) {
            row[w] = m;
            if (w < a.words && warp < a.nchunks_real)
                a.bitmapT[c][((size_t)(warp / kSubChunks) * a.words + w) * kSubStride + (warp % kSubChunks)] = m;
        }
    }
}

static uint32_t bitlen(uint32_t x) { uint32_t b = 0; while (x) { ++b; x >>= 1; } return b ? b : 1; }

int launch_offer_ingest(DeviceState& ds, OfferTable& t, const OfferIngest& in, cudaStream_t st) {
    int launches = 0;
    const uint32_t G = in.G;
    uint32_t n = 1024;
    while (n < G) n <<= 1;
    // padded length: whole kChunk multiples plus one spare segment so a CTA's bulk copy never runs off the end
    const uint32_t Gpad = ((G + kChunk - 1) / kChunk) * kChunk + kSegPacked;
    ds.sort_keys.reserve((size_t)3 * n);
    ds.sort_vals.reserve((size_t)3 * n);
    for (int c = 0; c < 2; ++c) {
        t.v_bitmap[c].reserve((size_t)(Gpad / 32) * kBmMaxStride);
        t.v_bitmapT[c].reserve((size_t)(((G + 31) / 32 + kSubChunks - 1) / kSubChunks + 1) * kBmMaxStride * kSubStride);
        t.v_packed[c].reserve(Gpad); t.v_wide[c].reserve(Gpad); t.v_price[c].reserve(Gpad); t.v_perm[c].reserve(Gpad);
    }
    for (int d = 0; d < 3; ++d) t.distinct[d].reserve(G ? G : 1);
    ds.dcount.reserve(4);
    u64* keys = ds.sort_keys.p;
    uint32_t* vals = ds.sort_vals.p;

    k_offer_keys<<<(n + 255) / 256, 256, 0, st>>>(G, n, in.flags, in.secure_price, in.community_price, keys, vals); ++launches;
    launches += bitonic_sort(keys, vals, n, st);
    launches += bitonic_sort(keys + n, vals + n, n, st);
    const int32_t* cols[3] = {in.mem, in.vcpu, in.ram};
    for (int d = 0; d < 3; ++d) {
        k_dim_keys<<<(n + 255) / 256, 256, 0, st>>>(G, n, cols[d], keys + 2 * (size_t)n, vals + 2 * (size_t)n); ++launches;
        launches += bitonic_sort(keys + 2 * (size_t)n, vals + 2 * (size_t)n, n, st);
        k_unique<<<1, 1024, 0, st>>>(keys + 2 * (size_t)n, G, t.distinct[d].p, ds.dcount.p + d); ++launches;
    }
    uint32_t D[3] = {0, 0, 0};
    RPK_CUDA(cudaMemcpyAsync(D, ds.dcount.p, sizeof(D), cudaMemcpyDeviceToHost, st));
    RPK_CUDA(cudaStreamSynchronize(st));
    // field widths: mem holds rank'+1 in [0, D0] and thresholds in [1, D0+1]; the others ranks in [0, D-1], thresholds in [0, D]
    uint32_t b1 = bitlen(D[0] + 1), b2 = bitlen(D[1]), b3 = bitlen(D[2]);
    PackLayout pk = {};
    if (b1 + b2 + b3 + 3 <= 32) {
        pk.bits = b1 + b2 + b3 + 3;
        pk.pos_bits = pk.bits + kPosBits <= 32 ? kPosBits : 0;
        pk.sh_ram = pk.pos_bits;
        pk.sh_vcpu = pk.sh_ram + b3 + 1;
        pk.sh_mem = pk.sh_vcpu + b2 + 1;
        pk.guard = (1u << (pk.sh_ram + b3)) | (1u << (pk.sh_vcpu + b2)) | (1u << (pk.sh_mem + b1));
    }
    const uint32_t bm_words = (D[0] + 1) + (D[1] + 1) + (D[2] + 1);
    if (bm_words <= kBmMaxStride) {
        pk.bm_words = bm_words; pk.bm_off_vcpu = D[0] + 1; pk.bm_off_ram = D[0] + 1 + D[1] + 1;
        pk.bm_stride = bm_words <= 32 ? 32 : 64;
    }
    if (ds.force_kind == 5 || ds.force_kind == 6) pk.no_fused = 1;
    if (ds.force_kind == 6) pk.no_persist = 1;
    if (ds.force_kind == 1) { pk.bits = 0; pk.pos_bits = 0; pk.bm_words = 0; }
    if (ds.force_kind == 2) { pk.pos_bits = 0; pk.bm_words = 0; }
    if (ds.force_kind == 3) pk.bm_words = 0;
    if (ds.force_kind == 2 && pk.bits) {  // re-derive the shifts without the position field
        pk.sh_ram = 0; pk.sh_vcpu = b3 + 1; pk.sh_mem = pk.sh_vcpu + b2 + 1;
        pk.guard = (1u << b3) | (1u << (pk.sh_vcpu + b2)) | (1u << (pk.sh_mem + b1));
    }
    t.nsub = 0;
    if (pk.bm_words) {
        BitmapArgs ba;
        ba.G = G; ba.nchunks = Gpad / 32; ba.keys = keys; ba.vals = vals; ba.n = n;
        ba.mem = in.mem; ba.vcpu = in.vcpu; ba.ram = in.ram;
        for (int d = 0; d < 3; ++d) { ba.distinct[d] = t.distinct[d].p; ba.D[d] = D[d]; }
        ba.off_vcpu = pk.bm_off_vcpu; ba.off_ram = pk.bm_off_ram; ba.words = pk.bm_words; ba.stride = pk.bm_stride;
        ba.nchunks_real = (G + 31) / 32;
        t.nsub = (ba.nchunks_real + kSubChunks - 1) / kSubChunks;
        for (int c = 0; c < 2; ++c) {
            ba.bitmap[c] = t.v_bitmap[c].p; ba.bitmapT[c] = t.v_bitmapT[c].p;
            RPK_CUDA(cudaMemsetAsync(t.v_bitmapT[c].p, 0, (size_t)(t.nsub ? t.nsub : 1) * pk.bm_words * kSubStride * sizeof(uint32_t), st));
        }
        k_offer_bitmap<<<dim3((ba.nchunks * 32 + 255) / 256, 2), 256, 0, st>>>(ba); ++launches;
    }
    PackArgs pa;
    pa.G = G; pa.Gpad = Gpad; pa.n = n; pa.keys = keys; pa.vals = vals;
    pa.mem = in.mem; pa.vcpu = in.vcpu; pa.ram = in.ram; pa.sp = in.secure_price; pa.cp = in.community_price;
    for (int d = 0; d < 3; ++d) { pa.distinct[d] = t.distinct[d].p; pa.D[d] = D[d]; }
    pa.pk = pk;
    for (int c = 0; c < 2; ++c) { pa.packed[c] = t.v_packed[c].p; pa.wide[c] = t.v_wide[c].p; pa.price[c] = t.v_price[c].p; pa.perm[c] = t.v_perm[c].p; }
    k_offer_pack<<<dim3((Gpad + 255) / 256, 2), 256, 0, st>>>(pa); ++launches;
    RPK_CUDA(cudaGetLastError());
    t.G = G; t.Gpad = Gpad; t.pk = pk;
    for (int d = 0; d < 3; ++d) t.D[d] = D[d];
    return launches;
}

// ---- offer sets ------------------------------------------------------------------------------------------
// A set is a sub-table: its members, gathered in ascending global order, go through the same ingest as the resident
// table.  Within the sub-table the (price, row) order is then the global (price, offer index) order, so the tie
// contract holds, and one remap of perm / wide.w to global ids lets every select kernel emit global indices.

// one block per set: popcount of each membership word, block-wide exclusive scan, each word's set bits written in
// ascending order from its offset (bits >= G are ignored)
__global__ void __launch_bounds__(1024) k_set_compact(const uint32_t* __restrict__ words, uint32_t W, uint32_t G,
                                                      const uint32_t* __restrict__ set_off, uint32_t* __restrict__ members) {
    __shared__ uint32_t warp_sum[32];
    __shared__ uint32_t carry;
    const uint32_t s = blockIdx.x, t = threadIdx.x, lane = t & 31, w = t >> 5;
    const uint32_t* sw = words + (size_t)s * W;
    uint32_t* out = members + set_off[s];
    if (t == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < W; base += 1024) {
        const uint32_t i = base + t;
        uint32_t m = i < W ? sw[i] : 0u;
        if (i < W && (i + 1) * 32 > G) m &= (1u << (G - i * 32)) - 1u;  // last word: 0 < G - 32 i < 32
        const uint32_t c = __popc(m);
        uint32_t incl = c;  // warp-inclusive scan of the counts
        for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= (uint32_t)d) incl += v; }
        if (lane == 31) warp_sum[w] = incl;
        __syncthreads();
        uint32_t off = 0, total = 0;
        for (uint32_t x = 0; x < 32; ++x) { const uint32_t v = warp_sum[x]; if (x < w) off += v; total += v; }
        uint32_t pos = carry + off + incl - c;
        while (m) { out[pos++] = i * 32 + (uint32_t)(__ffs(m) - 1); m &= m - 1; }
        __syncthreads();
        if (t == 0) carry += total;
        __syncthreads();
    }
}

// the six raw columns of the members (sub-table row j = offer members[j])
__global__ void k_set_gather(uint32_t n, const uint32_t* __restrict__ members, const int32_t* __restrict__ mem,
                             const int32_t* __restrict__ vcpu, const int32_t* __restrict__ ram, const double* __restrict__ sp,
                             const double* __restrict__ cp, const uint8_t* __restrict__ flags, int32_t* __restrict__ o_mem,
                             int32_t* __restrict__ o_vcpu, int32_t* __restrict__ o_ram, double* __restrict__ o_sp,
                             double* __restrict__ o_cp, uint8_t* __restrict__ o_flags) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t g = members[j];
    o_mem[j] = mem[g]; o_vcpu[j] = vcpu[g]; o_ram[j] = ram[g]; o_sp[j] = sp[g]; o_cp[j] = cp[g]; o_flags[j] = flags[g];
}

// sub-table row -> global offer id in both views (-1 = unavailable / padding stays -1)
__global__ void k_set_remap(uint32_t Gpad, const uint32_t* __restrict__ members, int32_t* perm0, int32_t* perm1, int4* wide0,
                            int4* wide1) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= Gpad) return;
    int32_t* perm = blockIdx.y ? perm1 : perm0;
    int4* wide = blockIdx.y ? wide1 : wide0;
    const int32_t p = perm[s];
    if (p >= 0) perm[s] = (int32_t)members[p];
    const int32_t w = wide[s].w;
    if (w >= 0) wide[s].w = (int32_t)members[w];
}

int launch_offer_sets_build(DeviceState& ds, uint32_t n_sets, const uint32_t* d_words, const uint32_t* counts, cudaStream_t st) {
    int launches = 0;
    const uint32_t G = ds.main.G, W = (G + 31) / 32;
    std::vector<uint32_t> off((size_t)n_sets + 1, 0);
    uint32_t gmax = 0;
    for (uint32_t s = 0; s < n_sets; ++s) { off[s + 1] = off[s] + counts[s]; gmax = counts[s] > gmax ? counts[s] : gmax; }
    ds.set_members.reserve((size_t)off[n_sets] + n_sets + 1);  // member lists, then the n_sets offsets
    uint32_t* d_off = ds.set_members.p + off[n_sets];
    RPK_CUDA(cudaMemcpyAsync(d_off, off.data(), (size_t)n_sets * 4, cudaMemcpyHostToDevice, st));
    if (n_sets && W) { k_set_compact<<<n_sets, 1024, 0, st>>>(d_words, W, G, d_off, ds.set_members.p); ++launches; }
    const size_t cap = gmax ? gmax : 1;
    ds.set_mem.reserve(cap); ds.set_vcpu.reserve(cap); ds.set_ram.reserve(cap);
    ds.set_sp.reserve(cap); ds.set_cp.reserve(cap); ds.set_flags.reserve(cap);
    for (uint32_t s = 0; s < n_sets; ++s) {
        OfferTable& t = ds.sets[s];
        const uint32_t n = counts[s];
        if (n == 0) { t.G = 0; continue; }  // an empty set never reaches a select kernel
        const uint32_t* mem = ds.set_members.p + off[s];
        k_set_gather<<<(n + 255) / 256, 256, 0, st>>>(n, mem, ds.raw_mem.p, ds.raw_vcpu.p, ds.raw_ram.p, ds.raw_sp.p, ds.raw_cp.p,
                                                      ds.raw_flags.p, ds.set_mem.p, ds.set_vcpu.p, ds.set_ram.p, ds.set_sp.p,
                                                      ds.set_cp.p, ds.set_flags.p);
        ++launches;
        OfferIngest in{n, ds.set_mem.p, ds.set_vcpu.p, ds.set_ram.p, ds.set_sp.p, ds.set_cp.p, ds.set_flags.p};
        launches += launch_offer_ingest(ds, t, in, st);  // synchronises st once (distinct-value counts)
        k_set_remap<<<dim3((t.Gpad + 255) / 256, 2), 256, 0, st>>>(t.Gpad, mem, t.v_perm[0].p, t.v_perm[1].p, t.v_wide[0].p, t.v_wide[1].p);
        ++launches;
    }
    RPK_CUDA(cudaGetLastError());
    return launches;
}

}  // namespace rpk
