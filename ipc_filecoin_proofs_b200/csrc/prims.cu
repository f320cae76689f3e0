// prims.cu — scan / bitmap compaction / radix sort kernels (see prims.cuh).
#include "prims.cuh"

namespace ipcfp {

// ------------------------------------------------------------------------------------------ scan
static constexpr int SCAN_THREADS = 512;
static constexpr int SCAN_ITEMS = 4;
static constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

struct LoadIdentity { __device__ __forceinline__ uint32_t operator()(const uint32_t* in, uint64_t i) const { return in[i]; } };
struct LoadPopc { __device__ __forceinline__ uint32_t operator()(const uint32_t* in, uint64_t i) const { return (uint32_t)__popc(in[i]); } };

__device__ __forceinline__ uint64_t block_exclusive_scan(uint64_t v, uint64_t* total) {
    __shared__ uint64_t warp_sums[SCAN_THREADS / 32];
    __shared__ uint64_t block_total;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint64_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint64_t s = lane < SCAN_THREADS / 32 ? warp_sums[lane] : 0;
        uint64_t t = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint64_t y = __shfl_up_sync(0xffffffffu, t, o);
            if (lane >= o) t += y;
        }
        if (lane < SCAN_THREADS / 32) warp_sums[lane] = t - s;
        if (lane == 31) block_total = t;
    }
    __syncthreads();
    uint64_t res = warp_sums[warp] + x - v;
    if (total) *total = block_total;
    __syncthreads();
    return res;
}

template <class Load> __global__ void __launch_bounds__(SCAN_THREADS) k_scan_reduce(const uint32_t* in, uint64_t n, uint64_t* block_sums, Load load) {
    uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
    uint64_t s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) if (base + k < n) s += load(in, base + k);
    uint64_t tot;
    block_exclusive_scan(s, &tot);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = tot;
}
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_block_sums(uint64_t* block_sums, uint64_t nblocks, uint64_t* total_dev) {
    uint64_t carry = 0;
    for (uint64_t base = 0; base < nblocks; base += SCAN_THREADS) {
        uint64_t i = base + threadIdx.x;
        uint64_t v = i < nblocks ? block_sums[i] : 0;
        uint64_t tot;
        uint64_t ex = block_exclusive_scan(v, &tot);
        if (i < nblocks) block_sums[i] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0 && total_dev) *total_dev = carry;
}
template <class Load> __global__ void __launch_bounds__(SCAN_THREADS) k_scan_final(const uint32_t* in, uint64_t* out, uint64_t n, const uint64_t* block_sums, Load load) {
    uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    uint64_t s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) { v[k] = base + k < n ? load(in, base + k) : 0; s += v[k]; }
    uint64_t ex = block_exclusive_scan(s, nullptr) + block_sums[blockIdx.x];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) { if (base + k < n) out[base + k] = ex; ex += v[k]; }
}

// The whole scan in one CTA (n ≤ SCAN_SMALL): tiles in sequence with a running carry — one launch instead of three.
static constexpr uint64_t SCAN_SMALL = 8 * SCAN_TILE;
template <class Load> __global__ void __launch_bounds__(SCAN_THREADS) k_scan_small(const uint32_t* in, uint64_t* out, uint64_t n, uint64_t* total_dev, Load load) {
    uint64_t carry = 0;
    for (uint64_t tile = 0; tile < n; tile += SCAN_TILE) {
        uint64_t base = tile + (uint64_t)threadIdx.x * SCAN_ITEMS;
        uint32_t v[SCAN_ITEMS];
        uint64_t s = 0;
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; k++) { v[k] = base + k < n ? load(in, base + k) : 0; s += v[k]; }
        uint64_t tot;
        uint64_t ex = block_exclusive_scan(s, &tot) + carry;
#pragma unroll
        for (int k = 0; k < SCAN_ITEMS; k++) { if (base + k < n) out[base + k] = ex; ex += v[k]; }
        carry += tot;
    }
    if (threadIdx.x == 0 && total_dev) *total_dev = carry;
}
// Second kernel of the two-launch scan: every CTA first adds up the tile sums of the tiles before it (≤ SCAN_FUSED_BLOCKS
// values, L2-resident) instead of waiting for a separate single-CTA pass over them.
static constexpr unsigned SCAN_FUSED_BLOCKS = 8192;
template <class Load> __global__ void __launch_bounds__(SCAN_THREADS) k_scan_final_fused(const uint32_t* in, uint64_t* out, uint64_t n, const uint64_t* block_sums,
                                                                                        uint64_t* total_dev, Load load) {
    uint64_t mine = 0;
    for (uint32_t i = threadIdx.x; i < blockIdx.x; i += SCAN_THREADS) mine += block_sums[i];
    uint64_t prefix;
    block_exclusive_scan(mine, &prefix);
    uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS];
    uint64_t s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) { v[k] = base + k < n ? load(in, base + k) : 0; s += v[k]; }
    uint64_t tot;
    uint64_t ex = block_exclusive_scan(s, &tot) + prefix;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) { if (base + k < n) out[base + k] = ex; ex += v[k]; }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0 && total_dev) *total_dev = prefix + tot;
}

size_t scan_scratch_elems(uint64_t n) { return (size_t)div_up(n, SCAN_TILE) + 1; }

template <class Load> static void scan_impl(const uint32_t* in, uint64_t* out, uint64_t n, uint64_t* total_dev, uint64_t* scratch, cudaStream_t st, Load load,
                                            bool fixed_launches) {
    if (n == 0) {
        if (total_dev) IPCFP_CUDA(cudaMemsetAsync(total_dev, 0, 8, st));
        return;
    }
    if (n <= SCAN_SMALL && !fixed_launches) { k_scan_small<<<1, SCAN_THREADS, 0, st>>>(in, out, n, total_dev, load); IPCFP_LAUNCH_CHECK(); return; }
    unsigned nb = div_up(n, SCAN_TILE);
    k_scan_reduce<<<nb, SCAN_THREADS, 0, st>>>(in, n, scratch, load); IPCFP_LAUNCH_CHECK();
    if (nb <= SCAN_FUSED_BLOCKS) { k_scan_final_fused<<<nb, SCAN_THREADS, 0, st>>>(in, out, n, scratch, total_dev, load); IPCFP_LAUNCH_CHECK(); return; }
    k_scan_block_sums<<<1, SCAN_THREADS, 0, st>>>(scratch, nb, total_dev); IPCFP_LAUNCH_CHECK();
    k_scan_final<<<nb, SCAN_THREADS, 0, st>>>(in, out, n, scratch, load); IPCFP_LAUNCH_CHECK();
}
void exclusive_scan_u32(const uint32_t* in, uint64_t* out, uint64_t n, uint64_t* total_dev, uint64_t* scratch, cudaStream_t st, bool fixed_launches) {
    scan_impl(in, out, n, total_dev, scratch, st, LoadIdentity(), fixed_launches);
}

// ------------------------------------------------------------------------------------------ bitmap → indices
__global__ void k_bitmap_scatter(const uint32_t* bits, uint64_t nwords, const uint64_t* word_prefix, uint32_t* out) {
    uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwords) return;
    uint32_t x = bits[w];
    uint64_t o = word_prefix[w];
    while (x) {
        int b = __ffs((int)x) - 1;
        out[o++] = (uint32_t)(w * 32 + (uint64_t)b);
        x &= x - 1;
    }
}
void bitmap_to_indices(const uint32_t* bits, uint64_t nbits, uint32_t* out, uint64_t* total_dev, uint64_t* word_prefix, uint64_t* scratch,
                       cudaStream_t st, bool fixed_launches) {
    uint64_t nwords = (nbits + 31) / 32;
    scan_impl(bits, word_prefix, nwords, total_dev, scratch, st, LoadPopc(), fixed_launches);
    if (nwords == 0) return;
    k_bitmap_scatter<<<div_up(nwords, 256), 256, 0, st>>>(bits, nwords, word_prefix, out); IPCFP_LAUNCH_CHECK();
}

// ------------------------------------------------------------------------------------------ radix sort
static constexpr int RS_THREADS = 256;
static constexpr int RS_WARPS = RS_THREADS / 32;
static constexpr int RS_CHUNKS = 8;                        // 32-key chunks per warp
static constexpr int RS_TILE = RS_THREADS * RS_CHUNKS;     // 2048 keys per block

unsigned radix_blocks(uint64_t n) { return n ? div_up(n, RS_TILE) : 1; }

__global__ void __launch_bounds__(RS_THREADS) k_radix_count(const uint32_t* keys, uint64_t n, int shift, uint32_t* ghist, unsigned nblocks) {
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    uint64_t base = (uint64_t)blockIdx.x * RS_TILE;
#pragma unroll
    for (int c = 0; c < RS_CHUNKS; c++) {
        uint64_t i = base + (uint64_t)c * RS_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&h[(keys[i] >> shift) & 255], 1u);
    }
    __syncthreads();
    ghist[(uint64_t)threadIdx.x * nblocks + blockIdx.x] = h[threadIdx.x];
}

__global__ void __launch_bounds__(RS_THREADS) k_radix_scatter(const uint32_t* keys, const uint32_t* vals, uint32_t* okeys, uint32_t* ovals,
                                                              uint64_t n, int shift, const uint64_t* ghist_scanned, unsigned nblocks) {
    __shared__ uint32_t wh[RS_WARPS][256];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < RS_WARPS * 256; i += RS_THREADS) (&wh[0][0])[i] = 0;
    __syncthreads();
    // each warp owns a CONTIGUOUS run of RS_CHUNKS*32 keys so that warp order == key order
    uint64_t wbase = (uint64_t)blockIdx.x * RS_TILE + (uint64_t)warp * (RS_CHUNKS * 32);
    uint32_t k[RS_CHUNKS];
#pragma unroll
    for (int c = 0; c < RS_CHUNKS; c++) {
        uint64_t i = wbase + (uint64_t)c * 32 + lane;
        k[c] = i < n ? keys[i] : 0;
        if (i < n) atomicAdd(&wh[warp][(k[c] >> shift) & 255], 1u);
    }
    __syncthreads();
    {
        int d = threadIdx.x;  // 256 threads ↔ 256 digits
        uint32_t run = (uint32_t)ghist_scanned[(uint64_t)d * nblocks + blockIdx.x];
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++) { uint32_t t = wh[w][d]; wh[w][d] = run; run += t; }
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < RS_CHUNKS; c++) {
        uint64_t i = wbase + (uint64_t)c * 32 + lane;
        bool valid = i < n;
        unsigned active = __ballot_sync(0xffffffffu, valid);
        if (valid) {
            uint32_t d = (k[c] >> shift) & 255;
            unsigned m = __match_any_sync(active, d);
            uint32_t rank = (uint32_t)__popc(m & ((1u << lane) - 1));
            uint32_t pos = wh[warp][d] + rank;
            okeys[pos] = k[c];
            ovals[pos] = vals[i];
            __syncwarp(active);
            if (rank == 0) wh[warp][d] += (uint32_t)__popc(m);
        }
        __syncwarp();
    }
}

void radix_sort_pairs(uint32_t* keys, uint32_t* vals, uint32_t* keys_alt, uint32_t* vals_alt, uint64_t n, int nbits, uint32_t* hist,
                      uint64_t* scan_tmp, uint64_t* scratch, cudaStream_t st) {
    if (n <= 1) return;
    unsigned nb = radix_blocks(n);
    uint32_t *ki = keys, *vi = vals, *ko = keys_alt, *vo = vals_alt;
    int passes = (nbits + 7) / 8;
    for (int p = 0; p < passes; p++) {
        k_radix_count<<<nb, RS_THREADS, 0, st>>>(ki, n, 8 * p, hist, nb); IPCFP_LAUNCH_CHECK();
        exclusive_scan_u32(hist, scan_tmp, (uint64_t)256 * nb, nullptr, scratch, st);
        k_radix_scatter<<<nb, RS_THREADS, 0, st>>>(ki, vi, ko, vo, n, 8 * p, scan_tmp, nb); IPCFP_LAUNCH_CHECK();
        uint32_t* t;
        t = ki; ki = ko; ko = t;
        t = vi; vi = vo; vo = t;
    }
    if (ki != keys) {
        IPCFP_CUDA(cudaMemcpyAsync(keys, ki, n * 4, cudaMemcpyDeviceToDevice, st));
        IPCFP_CUDA(cudaMemcpyAsync(vals, vi, n * 4, cudaMemcpyDeviceToDevice, st));
    }
}

}  // namespace ipcfp
