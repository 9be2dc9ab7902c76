// scatter.cu -- deterministic scatter-add through an index: inverse index (CSR) + pull.
//
// The backward of every gather (grouping, index_points, 3-NN interpolation, the chamfer nearest points) adds the rows of an
// upstream gradient into the rows named by an index.  The default kernels (train.cu) do that with fp32 atomics, so the order
// of the additions into one destination row, and with it the rounding, changes from run to run.  Here the index is inverted
// first -- destination -> its slots in ascending slot order -- and one warp per destination row then adds its slots in that
// order, sequentially in fp32 starting from 0: the sum np.add.at computes.
//
//   pn_csr_build     key(slot) = batch * n_dst + clamp(idx[slot]); a STABLE least-significant-digit radix sort of the keys
//                    (8-bit digits, as many passes as the largest key needs) leaves the slots of each key in ascending order;
//                    the offsets are the first position of each key.  No atomics but the integer digit histograms, no size
//                    limit on a segment (a padded ball repeats its first hit, so a point can own many slots).
//   pn_csr_pull_f32  out[d, c] = sum over the slots s of d, in order, of (weight ? weight[s] : 1) * src[(s / div) * ld + col0 + c].
#include "common.cuh"

namespace pn {
namespace csr {

constexpr int THREADS = 256, ITEMS = 8, TILE = THREADS * ITEMS, RADIX = 256, SCAN_THREADS = 1024;

__global__ void keys_kernel(const void* __restrict__ idx, int idx64, int64_t n, int64_t per_batch, int n_dst,
                            uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t j = idx64 ? static_cast<const int64_t*>(idx)[i] : (int64_t) static_cast<const int32_t*>(idx)[i];
        j = j < 0 ? 0 : (j >= n_dst ? n_dst - 1 : j);
        keys[i] = (uint32_t)((i / per_batch) * n_dst + j);
        vals[i] = (uint32_t)i;
    }
}

// hist[d * tiles + t] = number of keys of tile t whose digit is d (digit-major, so that one exclusive scan gives every tile's
// first output position per digit in tile order).
__global__ void __launch_bounds__(THREADS)
hist_kernel(const uint32_t* __restrict__ keys, int64_t n, int shift, int tiles, uint32_t* __restrict__ hist) {
    __shared__ uint32_t h[RADIX];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * TILE;
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
        const int64_t e = base + i * THREADS + threadIdx.x;
        if (e < n) atomicAdd(&h[(keys[e] >> shift) & (RADIX - 1)], 1u);
    }
    __syncthreads();
    hist[(int64_t)threadIdx.x * tiles + blockIdx.x] = h[threadIdx.x];
}

__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t x, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    return x;
}

// In-place exclusive scan of a[0, n) by one CTA.
__global__ void __launch_bounds__(SCAN_THREADS) scan_kernel(uint32_t* __restrict__ a, int64_t n) {
    __shared__ uint32_t wsum[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t carry = 0;
    for (int64_t base = 0; base < n; base += SCAN_THREADS) {
        const int64_t e = base + threadIdx.x;
        const uint32_t v = e < n ? a[e] : 0u;
        const uint32_t x = warp_incl_scan(v, lane);
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        if (warp == 0) wsum[lane] = warp_incl_scan(wsum[lane], lane);
        __syncthreads();
        if (e < n) a[e] = carry + (warp ? wsum[warp - 1] : 0u) + x - v;
        carry += wsum[31];
        __syncthreads();
    }
}

// One stable pass: the keys of a tile keep their order among equal digits (ranked 256 at a time: within a warp by
// __match_any_sync, across the warps by the per-warp digit counts, across the steps by the running per-digit position).
__global__ void __launch_bounds__(THREADS)
scatter_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in, int64_t n, int shift, int tiles,
               const uint32_t* __restrict__ offs, uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out) {
    __shared__ uint32_t run[RADIX];
    __shared__ uint32_t wcnt[THREADS / 32][RADIX];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    run[tid] = offs[(int64_t)tid * tiles + blockIdx.x];
    const int64_t base = (int64_t)blockIdx.x * TILE;
    for (int i = 0; i < ITEMS; ++i) {
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) wcnt[w][tid] = 0;
        __syncthreads();
        const int64_t e = base + i * THREADS + tid;
        const bool ok = e < n;
        const uint32_t k = ok ? keys_in[e] : 0u;
        const uint32_t d = ok ? (k >> shift) & (RADIX - 1) : (uint32_t)RADIX;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const unsigned below = peers & ((1u << lane) - 1u);
        if (ok && below == 0) wcnt[warp][d] = __popc(peers);
        __syncthreads();
        if (ok) {
            uint32_t pos = run[d] + __popc(below);
            for (int w = 0; w < warp; ++w) pos += wcnt[w][d];
            keys_out[pos] = k;
            vals_out[pos] = vals_in[e];
        }
        __syncthreads();
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) t += wcnt[w][tid];
        run[tid] += t;
    }
}

// off[k] = the first position of the sorted keys holding a key >= k, for k in [0, n_keys]; off[n_keys] = n.
__global__ void offsets_kernel(const uint32_t* __restrict__ keys, int64_t n, int64_t n_keys, int32_t* __restrict__ off) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i <= n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t lo = i == 0 ? 0 : (int64_t)keys[i - 1] + 1;
        const int64_t hi = i == n ? n_keys : (int64_t)keys[i];
        for (int64_t k = lo; k <= hi; ++k) off[k] = (int32_t)i;
    }
}

__global__ void __launch_bounds__(256)
pull_kernel(const float* __restrict__ src, int64_t ld, int col0, int D, int div, const float* __restrict__ weight,
            const int32_t* __restrict__ off, const int32_t* __restrict__ slots, int64_t n_dst, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t d = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); d < n_dst; d += warps) {
        const int s0 = off[d], s1 = off[d + 1];
        for (int c = lane; c < D; c += 32) {
            float acc = 0.0f;
            for (int s = s0; s < s1; ++s) {
                const int slot = slots[s];
                float v = src[(int64_t)(slot / div) * ld + col0 + c];
                if (weight) v = __fmul_rn(v, weight[slot]);
                acc = __fadd_rn(acc, v);
            }
            out[d * D + c] = acc;
        }
    }
}

struct Plan {
    int64_t tiles, hist_words;
    int passes;
    size_t bytes;
};

static Plan plan(int64_t n, int64_t n_keys) {
    Plan p;
    p.tiles = ceil_div(n > 0 ? n : 1, TILE);
    p.hist_words = RADIX * p.tiles;
    int bits = 0;
    while (bits < 32 && ((uint64_t)(n_keys - 1) >> bits) != 0) ++bits;
    p.passes = bits <= 8 ? 1 : (bits + 7) / 8;
    p.bytes = sizeof(uint32_t) * (size_t)(4 * n + p.hist_words);
    return p;
}

static inline unsigned grid_for(int64_t n, int threads) {
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
    const int64_t want = ceil_div(n > 0 ? n : 1, threads), cap = (int64_t)sms * 16;
    return (unsigned)(want > cap ? cap : want);
}

}  // namespace csr

int csr_pull(const float* src, int64_t ld, int col0, int D, int div, const float* weight, const int32_t* offsets,
             const int32_t* slots, int64_t n_dst, float* out, cudaStream_t stream) {
    csr::pull_kernel<<<csr::grid_for(n_dst * 32, 256), 256, 0, stream>>>(src, ld, col0, D, div, weight, offsets, slots, n_dst, out);
    return finish_launch("pn_csr_pull_f32");
}

}  // namespace pn

using namespace pn;

PN_EXPORT size_t pn_csr_workspace_bytes(int64_t n_slots, int64_t n_keys) {
    if (n_slots <= 0 || n_keys <= 0 || n_slots >= ((int64_t)1 << 31) || n_keys >= ((int64_t)1 << 31)) return 0;
    return csr::plan(n_slots, n_keys).bytes;
}

PN_EXPORT int pn_csr_build(const void* idx, int idx_bits, int64_t n_slots, int64_t slots_per_batch, int n_dst, int B,
                           void* workspace, size_t workspace_bytes, int32_t* offsets, int32_t* slots, pn_stream_t stream) {
    PN_REQUIRE(idx && workspace && offsets && slots, PN_ERR_BAD_ARG, "pn_csr_build: null pointer");
    PN_REQUIRE(idx_bits == 32 || idx_bits == 64, PN_ERR_BAD_ARG, "pn_csr_build: idx_bits must be 32 or 64");
    PN_REQUIRE(B > 0 && n_dst > 0 && slots_per_batch > 0 && n_slots == (int64_t)B * slots_per_batch, PN_ERR_BAD_ARG,
               "pn_csr_build: bad shape (n_slots must be B * slots_per_batch)");
    const int64_t n_keys = (int64_t)B * n_dst;
    PN_REQUIRE(n_slots < ((int64_t)1 << 31) && n_keys < ((int64_t)1 << 31), PN_ERR_UNSUPPORTED,
               "pn_csr_build: fewer than 2^31 slots and destinations");
    const csr::Plan p = csr::plan(n_slots, n_keys);
    PN_REQUIRE(workspace_bytes >= p.bytes, PN_ERR_BAD_ARG, "pn_csr_build: workspace of %zu bytes, need %zu", workspace_bytes,
               p.bytes);
    PN_REQUIRE(((uintptr_t)workspace & 3) == 0, PN_ERR_BAD_ARG, "pn_csr_build: workspace must be 4-byte aligned");
    PN_REQUIRE(p.tiles <= 65535 * 32, PN_ERR_UNSUPPORTED, "pn_csr_build: too many slots");
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t* w = static_cast<uint32_t*>(workspace);
    uint32_t *keys[2] = {w, w + n_slots}, *vals[2] = {w + 2 * n_slots, w + 3 * n_slots};
    uint32_t* hist = w + 4 * n_slots;
    csr::keys_kernel<<<csr::grid_for(n_slots, 256), 256, 0, st>>>(idx, idx_bits == 64, n_slots, slots_per_batch, n_dst, keys[0],
                                                                  vals[0]);
    for (int pass = 0; pass < p.passes; ++pass) {
        const int in = pass & 1, out = in ^ 1;
        uint32_t* vout = pass == p.passes - 1 ? reinterpret_cast<uint32_t*>(slots) : vals[out];
        csr::hist_kernel<<<(unsigned)p.tiles, csr::THREADS, 0, st>>>(keys[in], n_slots, 8 * pass, (int)p.tiles, hist);
        csr::scan_kernel<<<1, csr::SCAN_THREADS, 0, st>>>(hist, p.hist_words);
        csr::scatter_kernel<<<(unsigned)p.tiles, csr::THREADS, 0, st>>>(keys[in], vals[in], n_slots, 8 * pass, (int)p.tiles, hist,
                                                                        keys[out], vout);
    }
    csr::offsets_kernel<<<csr::grid_for(n_slots + 1, 256), 256, 0, st>>>(keys[p.passes & 1], n_slots, n_keys, offsets);
    return finish_launch("pn_csr_build");
}

PN_EXPORT int pn_csr_pull_f32(const float* src, int64_t ld, int col0, int D, int div, const float* weight, const int32_t* offsets,
                              const int32_t* slots, int64_t n_dst, float* out, pn_stream_t stream) {
    PN_REQUIRE(src && offsets && slots && out, PN_ERR_BAD_ARG, "pn_csr_pull_f32: null pointer");
    PN_REQUIRE(n_dst > 0 && D > 0 && div > 0 && col0 >= 0 && ld >= col0 + D, PN_ERR_BAD_ARG, "pn_csr_pull_f32: bad shape");
    return csr_pull(src, ld, col0, D, div, weight, offsets, slots, n_dst, out, (cudaStream_t)stream);
}
