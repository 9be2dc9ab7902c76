// three_nn.cu -- the 3-NN search of PointNetFeaturePropagation (reference: model/pointnet_util.py:295-300) as an exact
// branch-and-bound over spatial blocks of the coarse cloud, for the levels where the brute-force scan of group.cu
// (N x S distance evaluations: 197 M at N = 24000, S = 1024, B = 8 -- 117 us of the whole GPU) would compete with the
// critical path of the forward.
//
//   build  (one CTA per cloud, S <= 8192): Morton-sort the coarse points (10 bits per axis inside the bounding box) and
//          cut the sorted sequence into blocks of BP = 8 / 16 / 32 points (at most 256 blocks) with their bounding boxes.
//          The points are stored in PAIRS, (x0, x1, y0, y1) (z0, z1, |p0|^2, |p1|^2), the operand layout of the packed
//          f32x2 arithmetic of the search.
//   search (one warp per 32 fine points, which should be spatial neighbours: the caller passes the bucket order of
//          the fine cloud): the warp's query box is tested against every block box, blocks are visited nearest first, and
//          the search stops when the nearest unvisited block is farther than the worst third-neighbour distance of the
//          warp.  Two candidates per instruction (mul / fma / add .f32x2 round each half exactly like the scalar forms);
//          ONE warp-uniform branch per pair decides whether any lane's top three changes, and the insertion itself is
//          branch-free.  (ncu on the first version, one divergent branch per candidate: 14 instructions per candidate on
//          the reject path, 6 of them BSSY / BSYNC / WARPSYNC / register moves, and 20 % of the candidates in the insert path.)
//
// The result is exactly the brute-force result: distances are the reference's expansion formula (common.cuh), the
// three neighbours are ordered by (distance, index), and a block is skipped only if its box distance exceeds the
// bound by more than the rounding slack of that formula.
#include <math_constants.h>
#include <stdlib.h>

#include "common.cuh"

namespace pn {

constexpr int kNbMaxS = 8192;
constexpr int kNbBuildThreads = 1024;
constexpr int kNbHdrFloats = 16;   // [0] = max |p|^2 over the cloud's bounding box
constexpr int kNbPadIndex = 0x7fffffff;

// points per block: at most 256 blocks (8 per lane of the searching warp)
static int nb_block_points(int S) {
    static const int forced = [] { const char* e = getenv("PN12_NN_BLOCK"); return e ? atoi(e) : 0; }();   // tuning hook
    // 16 measured best at S = 1024 (fp1 of the segmentation nets; search alone 54 / 54 / 62 us for 8 / 16 / 32 at C2)
    const int least = S <= 2048 ? 8 : (S <= 4096 ? 16 : 32), preferred = S <= 4096 ? 16 : 32;
    return (forced == 8 || forced == 16 || forced == 32) && forced >= least ? forced : preferred;
}
__host__ __device__ inline int nb_padded(int S) { return (S + 31) / 32 * 32; }
__host__ __device__ inline size_t nb_cloud_bytes(int S, int BP) {
    const size_t Sp = (size_t)nb_padded(S);
    // header | pairs: float4 (x0, x1, y0, y1), float4 (z0, z1, w0, w1) [Sp / 2] | int index [Sp] | boxes float[8] per block
    return (size_t)kNbHdrFloats * 4 + Sp * 16 + Sp * 4 + Sp / BP * 32;
}

__device__ __forceinline__ unsigned spread10(unsigned v) {   // 10 bits -> every third bit
    v &= 0x3FFu;
    v = (v | (v << 16)) & 0x030000FFu;
    v = (v | (v << 8)) & 0x0300F00Fu;
    v = (v | (v << 4)) & 0x030C30C3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}

__global__ void __launch_bounds__(kNbBuildThreads, 1)
nn_blocks_build_kernel(const float* __restrict__ xyz, int64_t xB, int64_t xN, int64_t xC, int S, int Spad, int BP,
                       unsigned char* __restrict__ ws_all, size_t ws_stride) {
    extern __shared__ unsigned long long keys[];   // Spad (power of two) composite keys: morton << 32 | index
    __shared__ float red[6][kNbBuildThreads / 32];
    __shared__ float box[6];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* __restrict__ p = xyz + (int64_t)b * xB;
    unsigned char* ws = ws_all + (size_t)b * ws_stride;

    float mn[3] = {3.0e38f, 3.0e38f, 3.0e38f}, mx[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
    for (int i = tid; i < S; i += kNbBuildThreads) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float v = p[(int64_t)i * xN + a * xC];
            mn[a] = fminf(mn[a], v);
            mx[a] = fmaxf(mx[a], v);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
            mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
        }
        if (lane == 0) {
            red[a][warp] = mn[a];
            red[3 + a][warp] = mx[a];
        }
    }
    __syncthreads();
    if (tid < 3) {
        float l = red[tid][0], h = red[3 + tid][0];
        for (int w = 1; w < kNbBuildThreads / 32; ++w) {
            l = fminf(l, red[tid][w]);
            h = fmaxf(h, red[3 + tid][w]);
        }
        if (!(l <= h)) { l = 0.0f; h = 0.0f; }
        box[tid] = l;
        box[3 + tid] = h;
    }
    __syncthreads();
    float sc[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float ext = box[3 + a] - box[a];
        sc[a] = ext > 0.0f ? 1023.999f / ext : 0.0f;
    }
    for (int i = tid; i < Spad; i += kNbBuildThreads) {
        unsigned long long k = ~0ull;
        if (i < S) {
            unsigned q[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const float t = (p[(int64_t)i * xN + a * xC] - box[a]) * sc[a];
                q[a] = (unsigned)fminf(fmaxf(t, 0.0f), 1023.0f);   // NaN -> 0
            }
            const unsigned m = spread10(q[0]) | (spread10(q[1]) << 1) | (spread10(q[2]) << 2);
            k = ((unsigned long long)m << 32) | (unsigned)i;
        }
        keys[i] = k;
    }
    __syncthreads();
    // bitonic sort, ascending
    for (int k = 2; k <= Spad; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < Spad; i += kNbBuildThreads) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = keys[i], c = keys[ixj];
                    const bool up = (i & k) == 0;
                    if ((a > c) == up) {
                        keys[i] = c;
                        keys[ixj] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
    const int Sp = nb_padded(S);
    float* __restrict__ pts = reinterpret_cast<float*>(ws + kNbHdrFloats * 4);
    int* __restrict__ index = reinterpret_cast<int*>(ws + kNbHdrFloats * 4 + (size_t)Sp * 16);
    float* __restrict__ boxes = reinterpret_cast<float*>(ws + kNbHdrFloats * 4 + (size_t)Sp * 20);
    for (int pos = tid; pos < Sp; pos += kNbBuildThreads) {       // (Sp is a multiple of 32: whole warps)
        float lo[3] = {3.0e38f, 3.0e38f, 3.0e38f}, hi[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
        float x = 0.0f, y = 0.0f, z = 0.0f, w = CUDART_INF_F;       // padding: distance +inf, index never "better"
        int i = kNbPadIndex;
        if (pos < S) {
            i = (int)(keys[pos] & 0xFFFFFFFFull);
            x = p[(int64_t)i * xN];
            y = p[(int64_t)i * xN + xC];
            z = p[(int64_t)i * xN + 2 * xC];
            w = sqnorm3(x, y, z);
            lo[0] = hi[0] = x;
            lo[1] = hi[1] = y;
            lo[2] = hi[2] = z;
        }
        float* pr = pts + (size_t)(pos >> 1) * 8 + (pos & 1);
        pr[0] = x;
        pr[2] = y;
        pr[4] = z;
        pr[6] = w;
        index[pos] = i;
#pragma unroll
        for (int a = 0; a < 3; ++a)
            for (int o = BP >> 1; o; o >>= 1) {
                lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
                hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
            }
        const int c = pos & (BP - 1);
        if (c < 3) {
            boxes[(pos / BP) * 8 + c] = c == 0 ? lo[0] : (c == 1 ? lo[1] : lo[2]);
            boxes[(pos / BP) * 8 + 4 + c] = c == 0 ? hi[0] : (c == 1 ? hi[1] : hi[2]);
        }
    }
    if (tid == 0) {
        float m2 = 0.0f;
        for (int a = 0; a < 3; ++a) {
            const float m = fmaxf(fabsf(box[a]), fabsf(box[3 + a]));
            m2 += m * m;
        }
        reinterpret_cast<float*>(ws)[0] = m2;
    }
}

// ------------------------------------------------------------------------------------------------ search
constexpr int kNbWarps = 4;

__device__ __forceinline__ bool nn_better(float d, int i, float dk, int ik) { return d < dk || (d == dk && i < ik); }

// monotone map float -> unsigned (for REDUX max over possibly negative distances) and back
__device__ __forceinline__ unsigned nn_ordered(float f) {
    const unsigned u = __float_as_uint(f);
    return u ^ ((unsigned)((int)u >> 31) | 0x80000000u);
}
__device__ __forceinline__ float nn_unordered(unsigned k) {
    return __uint_as_float(k ^ ((k & 0x80000000u) ? 0x80000000u : 0xFFFFFFFFu));
}

// (d, jj) into the lane's sorted top three, branch-free; lanes whose candidate is not better keep their state
__device__ __forceinline__ void nn_insert(float d, int jj, float& d0, float& d1, float& d2, int& i0, int& i1, int& i2) {
    const bool b2 = nn_better(d, jj, d2, i2), b1 = nn_better(d, jj, d1, i1), b0 = nn_better(d, jj, d0, i0);
    d2 = b1 ? d1 : (b2 ? d : d2);
    i2 = b1 ? i1 : (b2 ? jj : i2);
    d1 = b0 ? d0 : (b1 ? d : d1);
    i1 = b0 ? i0 : (b1 ? jj : i1);
    d0 = b0 ? d : d0;
    i0 = b0 ? jj : i0;
}

template <int BP, int NSLOT>
__global__ void __launch_bounds__(kNbWarps * 32)
three_nn_blocks_kernel(const float* __restrict__ xyz1, int64_t aB, int64_t aN, int64_t aC, const int* __restrict__ order,
                       int64_t order_es, int64_t order_bs, const unsigned char* __restrict__ ws_all, size_t ws_stride, int N,
                       int S, int64_t* __restrict__ idx, float* __restrict__ weight) {
    extern __shared__ __align__(16) unsigned char nb_smem[];   // pairs [Sp / 2][2] float4 | int index[Sp] | float boxes[nblk * 8]
    const int Sp = nb_padded(S), nblk = Sp / BP;
    const float4* spts = reinterpret_cast<const float4*>(nb_smem);
    const int* sidx = reinterpret_cast<const int*>(nb_smem + (size_t)Sp * 16);
    const float* sbox = reinterpret_cast<const float*>(nb_smem + (size_t)Sp * 20);
    const int b = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned char* ws = ws_all + (size_t)b * ws_stride;
    {   // stage the cloud's blocks (the three regions are contiguous in the workspace, 16-byte granular)
        const uint4* src = reinterpret_cast<const uint4*>(ws + kNbHdrFloats * 4);
        uint4* dst = reinterpret_cast<uint4*>(nb_smem);
        const int n16 = (int)((nb_cloud_bytes(S, BP) - kNbHdrFloats * 4) / 16);
        for (int i = threadIdx.x; i < n16; i += kNbWarps * 32) dst[i] = src[i];
    }
    const float m2c = reinterpret_cast<const float*>(ws)[0];
    __syncthreads();

    // (a capped grid -- background mode -- walks several groups of kNbWarps * 32 fine points per CTA)
    for (int r0 = blockIdx.x * kNbWarps * 32; r0 < N; r0 += gridDim.x * kNbWarps * 32) {
        const int r = r0 + warp * 32 + lane;   // position in the processing order
        const bool ok = r < N;
        int n = ok ? r : 0;
        if (ok && order) {
            n = order[(int64_t)b * order_bs + (int64_t)r * order_es];
            n = n < 0 ? 0 : (n >= N ? N - 1 : n);
        }
        const float* a = xyz1 + (int64_t)b * aB + (int64_t)n * aN;
        const float ax = a[0], ay = a[aC], az = a[2 * aC];
        const float sa = sqnorm3(ax, ay, az);
        // the warp's query box
        float qlo[3] = {ok ? ax : 3.0e38f, ok ? ay : 3.0e38f, ok ? az : 3.0e38f};
        float qhi[3] = {ok ? ax : -3.0e38f, ok ? ay : -3.0e38f, ok ? az : -3.0e38f};
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                qlo[c] = fminf(qlo[c], __shfl_xor_sync(0xffffffffu, qlo[c], o));
                qhi[c] = fmaxf(qhi[c], __shfl_xor_sync(0xffffffffu, qhi[c], o));
            }
        float m2q = 0.0f;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float m = fmaxf(fabsf(qlo[c]), fabsf(qhi[c]));
            m2q += m * m;
        }
        const float slack = (m2q + m2c) * (1.0f / 131072.0f);   // 2^-17 (|a|^2 + |b|^2)  >>  rounding of the expansion formula
        // box-to-box lower bounds, block k + 32 j in slot j of lane k
        float lb[NSLOT];
#pragma unroll
        for (int j = 0; j < NSLOT; ++j) {
            const int blk = lane + 32 * j;
            lb[j] = CUDART_INF_F;
            if (blk < nblk) {
                float s2 = 0.0f;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float g = fmaxf(fmaxf(sbox[blk * 8 + c] - qhi[c], qlo[c] - sbox[blk * 8 + 4 + c]), 0.0f);
                    s2 += g * g;
                }
                lb[j] = s2;
            }
        }
        float d0 = CUDART_INF_F, d1 = CUDART_INF_F, d2 = CUDART_INF_F;
        int i0 = kNbPadIndex, i1 = kNbPadIndex, i2 = kNbPadIndex;
        const bool any_ok = __any_sync(0xffffffffu, ok);
        const unsigned long long ax2 = pack2(ax, ax), ay2 = pack2(ay, ay), az2 = pack2(az, az), sa2 = pack2(sa, sa),
                                 minus2 = pack2(-2.0f, -2.0f);
        for (int visited = 0; any_ok && visited < nblk; ++visited) {
            // nearest unvisited block of this lane, then of the warp
            float mine = lb[0];
            int slot = 0;
#pragma unroll
            for (int j = 1; j < NSLOT; ++j)
                if (lb[j] < mine) {
                    mine = lb[j];
                    slot = j;
                }
            const unsigned mbits = __reduce_min_sync(0xffffffffu, __float_as_uint(mine));   // lower bounds are >= 0
            const float nearest = __uint_as_float(mbits);
            // the warp's worst third-neighbour distance (inf while any live lane has fewer than three)
            const float worst = nn_unordered(__reduce_max_sync(0xffffffffu, ok ? nn_ordered(d2) : 0u));
            if (!(nearest <= worst * 1.001f + slack)) break;
            const int owner = __ffs(__ballot_sync(0xffffffffu, __float_as_uint(mine) == mbits)) - 1;
            const int blk = __shfl_sync(0xffffffffu, lane + 32 * slot, owner);
            if (lane == owner) {
#pragma unroll
                for (int j = 0; j < NSLOT; ++j)
                    if (j == slot) lb[j] = CUDART_INF_F;
            }
            const float4* pp = spts + (size_t)blk * BP;        // BP / 2 pairs of two float4
            const int* pi = sidx + (size_t)blk * BP;
#pragma unroll
            for (int q = 0; q < BP / 2; ++q) {
                const float4 A = pp[2 * q], Bv = pp[2 * q + 1];
                // dot = fma(az,bz, fma(ay,by, ax*bx));  d = fma(-2, dot, |a|^2) + |b|^2   (sqdist_expand, two candidates at once)
                unsigned long long t = mul2(ax2, pack2(A.x, A.y));
                t = fma2(ay2, pack2(A.z, A.w), t);
                t = fma2(az2, pack2(Bv.x, Bv.y), t);
                t = add2(fma2(minus2, t, sa2), pack2(Bv.z, Bv.w));
                float e0, e1;
                unpack2(t, e0, e1);
                if (!__any_sync(0xffffffffu, !(e0 > d2) || !(e1 > d2))) continue;        // the common case, warp-uniform
                if (__any_sync(0xffffffffu, !(e0 > d2))) nn_insert(e0, pi[2 * q], d0, d1, d2, i0, i1, i2);
                if (__any_sync(0xffffffffu, !(e1 > d2))) nn_insert(e1, pi[2 * q + 1], d0, d1, d2, i0, i1, i2);
            }
        }
        if (!ok) continue;
        // dists[dists < 1e-10] = 1e-10 ; weight = 1/d ; weight /= sum(weight)   (pointnet_util.py:298-300)
        const float c0 = d0 < 1e-10f ? 1e-10f : d0, c1 = d1 < 1e-10f ? 1e-10f : d1, c2 = d2 < 1e-10f ? 1e-10f : d2;
        const float w0 = __fdiv_rn(1.0f, c0), w1 = __fdiv_rn(1.0f, c1), w2 = __fdiv_rn(1.0f, c2);
        const float norm = __fadd_rn(__fadd_rn(w0, w1), w2);
        const int64_t o = ((int64_t)b * N + n) * 3;
        idx[o] = i0;
        idx[o + 1] = i1;
        idx[o + 2] = i2;
        weight[o] = __fdiv_rn(w0, norm);
        weight[o + 1] = __fdiv_rn(w1, norm);
        weight[o + 2] = __fdiv_rn(w2, norm);
    }
}

}  // namespace pn

PN_EXPORT size_t pn_three_nn_blocks_bytes(int B, int S) {
    if (B <= 0 || S <= 0) return 0;
    return (size_t)B * pn::nb_cloud_bytes(S, pn::nb_block_points(S));
}

PN_EXPORT int pn_three_nn_blocks_build_f32(const float* xyz2, int64_t bB, int64_t bN, int64_t bC, int B, int S, void* blocks,
                                           size_t blocks_bytes, pn_stream_t stream) {
    using namespace pn;
    PN_REQUIRE(xyz2 && blocks, PN_ERR_BAD_ARG, "pn_three_nn_blocks_build_f32: null pointer");
    PN_REQUIRE(B > 0 && S >= 3, PN_ERR_BAD_ARG, "pn_three_nn_blocks_build_f32: need B > 0 and S >= 3 (got %d, %d)", B, S);
    PN_REQUIRE(S <= kNbMaxS, PN_ERR_UNSUPPORTED, "pn_three_nn_blocks_build_f32: S=%d exceeds %d", S, kNbMaxS);
    PN_REQUIRE(((uintptr_t)blocks & 15) == 0, PN_ERR_ALIGNMENT, "pn_three_nn_blocks_build_f32: blocks must be 16-byte aligned");
    PN_REQUIRE(blocks_bytes >= pn_three_nn_blocks_bytes(B, S), PN_ERR_BAD_ARG,
               "pn_three_nn_blocks_build_f32: buffer holds %zu bytes, %zu needed", blocks_bytes, pn_three_nn_blocks_bytes(B, S));
    int Spad = 32;
    while (Spad < S) Spad <<= 1;
    const size_t smem = (size_t)Spad * sizeof(unsigned long long);
    auto kern = nn_blocks_build_kernel;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("pn_three_nn_blocks_build_f32: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
        return (int)e;
    }
    const int BP = nb_block_points(S);
    kern<<<B, kNbBuildThreads, smem, (cudaStream_t)stream>>>(xyz2, bB, bN, bC, S, Spad, BP, static_cast<unsigned char*>(blocks),
                                                            nb_cloud_bytes(S, BP));
    return finish_launch("pn_three_nn_blocks_build_f32");
}

PN_EXPORT int pn_three_nn_blocks_f32(const float* xyz1, int64_t aB, int64_t aN, int64_t aC, const int32_t* order,
                                     int64_t order_es, int64_t order_bs, const void* blocks, size_t blocks_bytes, int B, int N,
                                     int S, int background, int64_t* idx, float* weight, pn_stream_t stream) {
    using namespace pn;
    PN_REQUIRE(xyz1 && blocks && idx && weight, PN_ERR_BAD_ARG, "pn_three_nn_blocks_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && S >= 3, PN_ERR_BAD_ARG, "pn_three_nn_blocks_f32: need B, N > 0 and S >= 3 (got %d, %d, %d)", B, N, S);
    PN_REQUIRE(S <= kNbMaxS && B <= 65535, PN_ERR_UNSUPPORTED, "pn_three_nn_blocks_f32: S=%d exceeds %d or B=%d exceeds 65535", S,
               kNbMaxS, B);
    PN_REQUIRE(blocks_bytes >= pn_three_nn_blocks_bytes(B, S), PN_ERR_BAD_ARG,
               "pn_three_nn_blocks_f32: buffer holds %zu bytes, %zu needed", blocks_bytes, pn_three_nn_blocks_bytes(B, S));
    const int BP = nb_block_points(S);
    const size_t smem = nb_cloud_bytes(S, BP) - kNbHdrFloats * 4;
    // background: at most ~3 CTAs (12 warps, 15 K registers, 65 KB of shared memory) per SM, so that kernels of a concurrent
    // stream still find room on every SM (an 8-warp streaming CTA of the chains: 25 K registers, 110 KB); the search then
    // takes longer but stays out of their way
    int64_t gx = ceil_div(N, kNbWarps * 32);
    if (background) {
        const int64_t cap = ceil_div(148 * 3, B);
        gx = gx < cap ? gx : cap;
    }
    const dim3 grid((unsigned)gx, (unsigned)B);
    auto launch = [&](auto kern) -> int {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_error("pn_three_nn_blocks_f32: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
            return (int)e;
        }
        kern<<<grid, kNbWarps * 32, smem, (cudaStream_t)stream>>>(xyz1, aB, aN, aC, order, order_es, order_bs,
                                                                 static_cast<const unsigned char*>(blocks), nb_cloud_bytes(S, BP), N,
                                                                 S, idx, weight);
        return finish_launch("pn_three_nn_blocks_f32");
    };
    const int slots = (nb_padded(S) / BP + 31) / 32;      // blocks per lane: <= 8
#define PN_NN_CASE(bp)                                                   \
    if (BP == bp) {                                                      \
        if (slots <= 1) return launch(three_nn_blocks_kernel<bp, 1>);    \
        if (slots <= 2) return launch(three_nn_blocks_kernel<bp, 2>);    \
        if (slots <= 4) return launch(three_nn_blocks_kernel<bp, 4>);    \
        return launch(three_nn_blocks_kernel<bp, 8>);                    \
    }
    PN_NN_CASE(8)
    PN_NN_CASE(16)
    PN_NN_CASE(32)
#undef PN_NN_CASE
    return PN_ERR_UNSUPPORTED;
}
