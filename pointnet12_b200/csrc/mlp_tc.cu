// mlp_tc.cu -- fused shared-MLP chains on the 5th-generation tensor cores (tcgen05 + TMEM), fp32 parity
// through a 3-pass split-bf16 product ("bf16x3": a = a_hi + a_lo, w = w_hi + w_lo, a*w ~ a_hi*w_hi + a_hi*w_lo +
// a_lo*w_hi with fp32 accumulation in TMEM; the dropped a_lo*w_lo term is ~2^-18 relative).
//
// One kernel runs a whole chain  rows -> [linear + bias (+ReLU)] x L -> {rows | max over groups | log_softmax}
// for a tile of 128 rows (points) per CTA:
//   reference                                                   here
//   gather + recentre + concat   pointnet_util.py:127-131,:243-247   producer: each thread builds ITS row
//   3-NN interpolate + concat    pointnet_util.py:301-307            producer: weighted gather of 3 coarse rows
//   conv1x1 + BN + ReLU chain    pointnet_util.py:195-197,:310-312   tcgen05.mma, BN folded into W and bias
//   max over nsample             pointnet_util.py:199                warp REDUX over the 32 rows of a group
//   conv2 + log_softmax          pointnet2.py:172-175                in-thread over the row's classes
//
// Orientation: D[128 rows x N channels] = A[128 rows x K] * W[N x K]^T.  TMEM lanes are rows (thread t owns row t
// of the tile), TMEM columns are channels.  The activations NEVER touch shared memory: a layer's accumulator is
// read back with tcgen05.ld by the thread that owns the row, gets bias + ReLU, is split into bf16 hi/lo, packed two
// per 32-bit cell and written with tcgen05.st into the TMEM region the next layer's MMAs read their A operand
// from (tcgen05.mma with A in TMEM).  Shared memory only holds weight tiles: pre-packed on the device into the
// exact UMMA K-major core-matrix image (8 rows x 16 bytes, no swizzle), streamed per 64-wide K slice with one
// cp.async.bulk (TMA engine) each into a 2-stage ring, completion on mbarriers (complete_tx), stage release by
// tcgen05.commit.  The PTX and its conventions (descriptor fields, A packing, TMEM addressing) come from tcgen05.cuh.
#include <cuda_bf16.h>
#include <math_constants.h>

#include "common.cuh"
#include "tcgen05.cuh"

namespace pn {

constexpr int kTcThreads = 256;  // 8 warps: warp w owns TMEM lanes 32*(w%4).., column half w/4 of every 64 columns
constexpr int kTcMaxLayers = PN_MLP_MAX_LAYERS;
constexpr int kTcKSub = 32;     // K values per streamed weight slice
constexpr int kTcMaxStages = 8; // ring depth limit of the streaming kernel
constexpr int kTcAChunk = 256;  // K values resident in TMEM as the A operand (128 columns hi + 128 columns lo)
constexpr int kTcNPass = 256;   // output channels per accumulation pass (TMEM D columns)

struct TcLayer {
    int k_real, k_pad, n_real, n_pad, relu;
    unsigned w_off;  // byte offset of the layer's weight images in the blob
    unsigned b_off;  // float offset of the layer's bias in the bias table
};
struct TcChain {
    int nlayers, stage_bytes, tmem_cols, x_cols, a_lo_off, bias_floats;
    int nstages;        // ring depth of the streaming kernel (set at launch)
    int pass_w;         // output channels per accumulation pass of the streaming kernel: kTcNPass, or the N-slice width
    int probe;          // timing probes of the resident kernel (results invalid): 1 = producer only, 2 = one group only, 4 = no producer
    int split;          // 1 = all three products a_hi*w_hi + a_hi*w_lo + a_lo*w_hi (fp32 parity); 0 = a_hi*w_hi only (plain bf16)
    unsigned bias_off;  // byte offset of the bias table in the blob
    unsigned blob_bytes;
    TcLayer L[kTcMaxLayers];
};

static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

// Plans the chain: padded sizes, blob layout, TMEM columns, ring stage size.  Returns false if unsupported.
static bool plan_chain(const pn_mlp_desc* d, TcChain* c, const char** why) {
    *why = "";
    if (!d || d->nlayers < 1 || d->nlayers > kTcMaxLayers) { *why = "nlayers must be in [1, 6]"; return false; }
    c->nlayers = d->nlayers;
    c->probe = 0;
    unsigned off = 0;
    int bias_floats = 0, stage = 0, x_cols = 0, a_k = 0;
    for (int l = 0; l < d->nlayers; ++l) {
        TcLayer& L = c->L[l];
        if (d->cin[l] < 1 || d->cout[l] < 1) { *why = "channel counts must be positive"; return false; }
        if (l > 0 && d->cin[l] != d->cout[l - 1]) { *why = "cin[l] must equal cout[l-1]"; return false; }
        L.k_real = d->cin[l];
        L.n_real = d->cout[l];
        L.relu = d->relu[l];
        L.n_pad = round_up(L.n_real, 32);
        L.k_pad = l == 0 ? round_up(L.k_real, 32) : c->L[l - 1].n_pad;
        if (l + 1 < d->nlayers && L.n_pad > kTcNPass) { *why = "hidden layers are limited to 256 channels"; return false; }
        if (L.n_pad > 1024 || L.k_pad > 4096) { *why = "layer too wide"; return false; }
        L.w_off = off;
        off += (unsigned)L.n_pad * (unsigned)L.k_pad * 4u;  // hi + lo bf16 images
        L.b_off = (unsigned)bias_floats;
        bias_floats += L.n_pad;
        const int rows_p = L.n_pad < kTcNPass ? L.n_pad : kTcNPass;
        const int kw = L.k_pad < kTcKSub ? L.k_pad : kTcKSub;
        stage = stage > rows_p * kw * 4 ? stage : rows_p * kw * 4;
        x_cols = x_cols > rows_p ? x_cols : rows_p;
        const int ak = L.k_pad < kTcAChunk ? L.k_pad : kTcAChunk;
        a_k = a_k > ak ? a_k : ak;
    }
    c->bias_off = off;
    c->bias_floats = bias_floats;
    c->blob_bytes = off + (unsigned)bias_floats * 4u;
    c->stage_bytes = stage;
    c->x_cols = x_cols;
    c->a_lo_off = a_k / 2;
    int cols = x_cols + a_k, p2 = 32;
    while (p2 < cols) p2 <<= 1;
    if (p2 > 512) { *why = "chain needs more than 512 TMEM columns"; return false; }
    c->tmem_cols = p2;
    return true;
}

// ------------------------------------------------------------------------------------------------ packing
// Weight image of one (pass, K slice): element (n, k) at (n/8)*SBO + (k/8)*128 + (n%8)*16 + (k%8)*2 bytes,
// SBO = (kw/8)*128; hi image first, lo image right after it.
// Element (n, k) of the layer's weight is w[n*sn + k*sk]: (sn, sk) = (k_real, 1) for a row-major [n, k] matrix, (1, n_real)
// for the TRANSPOSE of a row-major [k, n] matrix (the input-gradient GEMM dx = dy W of the training step reads W^T).
__global__ void tc_pack_layer_kernel(const float* __restrict__ w, const float* __restrict__ bias, int k_real, int k_pad,
                                     int n_real, int n_pad, int sn, int sk, unsigned char* __restrict__ img,
                                     float* __restrict__ bias_out) {
    const int total = n_pad * k_pad;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int n = e / k_pad, k = e % k_pad;
        const float v = (n < n_real && k < k_real) ? w[(size_t)n * sn + (size_t)k * sk] : 0.0f;
        const __nv_bfloat16 hi = __float2bfloat16_rn(v);
        const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
        const int p = n / kTcNPass, np = n % kTcNPass;
        const int rows_p = min(kTcNPass, n_pad - p * kTcNPass);
        const int s = k / kTcKSub, ks = k % kTcKSub;
        const int kw = min(kTcKSub, k_pad - s * kTcKSub);
        // offset of (pass p, slice s): passes are [rows_p x k_pad] blocks, slices inside a pass are consecutive
        size_t off = (size_t)p * kTcNPass * k_pad * 4 + (size_t)rows_p * (s * kTcKSub) * 4;
        const size_t in_img = (size_t)(np / 8) * (kw / 8) * 128 + (size_t)(ks / 8) * 128 + (np % 8) * 16 + (ks % 8) * 2;
        *reinterpret_cast<__nv_bfloat16*>(img + off + in_img) = hi;
        *reinterpret_cast<__nv_bfloat16*>(img + off + (size_t)rows_p * kw * 2 + in_img) = lo;
    }
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < n_pad; n += gridDim.x * blockDim.x)
        bias_out[n] = (bias && n < n_real) ? bias[n] : 0.0f;
}

// ------------------------------------------------------------------------------------------------ device helpers
// order-preserving float <-> uint key (for REDUX max over possibly negative values)
__device__ __forceinline__ unsigned tc_key(float f) {
    const unsigned b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float tc_unkey(unsigned k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

// Column-wise max over the 32 rows (= lanes) of a warp for 32 columns held one row per lane (a butterfly: 31 shuffles and
// max per lane instead of 32 REDUX instructions, which the hardware serialises).  Afterwards lane j holds the max of column j.
__device__ __forceinline__ float tc_colmax32(float (&v)[32], int lane) {
    tc::col_butterfly<16, 1>(v, lane, [](float x, float y) { return fmaxf(x, y); });
    return v[0];
}
// The same over the 16 rows of each half-warp for the 16 columns in v[0..15]: lane j holds column j % 16 of its half.
__device__ __forceinline__ float tc_colmax16(float (&v)[32], int lane) {
    tc::col_butterfly<8, 1>(v, lane, [](float x, float y) { return fmaxf(x, y); });
    return v[0];
}
// Max-pool epilogue for groups of 16 rows (two groups per warp): 32 accumulator columns in r -> y[group, c0 .. c0+31]
__device__ __forceinline__ void tc_store_max16(const unsigned (&r)[32], const float* bias, int relu, bool valid, int64_t row,
                                               int lane, int c0, int n_real, float* y, int64_t ldy) {
    const unsigned half_mask = (lane & 16) ? 0xffff0000u : 0x0000ffffu;
    const bool any_valid = (__ballot_sync(0xffffffffu, valid) & half_mask) != 0u;
    const int64_t g = __shfl_sync(0xffffffffu, row / 16, lane & 16);   // the group of this half-warp (its first lane)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        float v[32];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = valid ? __uint_as_float(r[h * 16 + j]) : -CUDART_INF_F;
        const int n = c0 + h * 16 + (lane & 15);
        float m = tc_colmax16(v, lane) + bias[n];      // (max first: bias + ReLU are monotone, the result is bit-identical)
        if (relu) m = fmaxf(m, 0.0f);
        if (any_valid && n < n_real) y[g * ldy + n] = m;
    }
}

// ------------------------------------------------------------------------------------------------ row producers
enum { TC_IN_ROWS = 0, TC_IN_SA = 1, TC_IN_FP = 2 };
enum { TC_OUT_ROWS = 0, TC_OUT_MAX = 1, TC_OUT_LOGSOFTMAX = 2 };

struct TcIo {
    // rows are organised in `nseg` segments of `seg_rows` rows; a tile never straddles two segments
    int64_t nseg, seg_rows;
    // TC_IN_ROWS
    const float* x; int64_t ldx;
    // TC_IN_SA: row = (b, s, k)
    const float* xyz; int64_t xB, xN, xC;
    const float* feat; int64_t fB, fN, fC; int D;
    const float* qxyz; int64_t qB, qN, qC;
    const int64_t* idx; int N, S, K, msg_order;
    // TC_IN_FP: row = (b, n)
    const float* p1; int64_t p1B, p1N, p1C; int D1;
    const float* p2; int64_t p2B, p2N, p2C; int D2; int S2;
    const int64_t* idx3; const float* w3;
    const int* order; int64_t order_es, order_bs;   // TC_IN_FP: optional processing order (row r of cloud b handles point order[b*bs + r*es])
    int relu_in;   // TC_IN_FP: ReLU applied to the interpolated channels (layer 1 was folded into the coarse level)
    // output
    int out_mode; float* y; int64_t ldy; int group;
    const float* res; int64_t ldr;   // optional per-row term added to layer 0's pre-activation: res[row * ldr + channel]
    int quad_fp;      // TC_IN_FP: all channel runs are float4-addressable -> coalesced quad producer (fp_quad_producer)
    long long* dbg;   // optional timeline (pn_launch_opts.mlp_debug): CTA 0 records clock64() per phase
    unsigned* tile_ctr;   // resident kernel: zeroed counter the 128-row tiles are handed out through (NULL: static round-robin)
};

template <int IN>
struct RowCtx {
    bool valid;
    int64_t row;      // global row index
    // SA
    const float* xyz_j; const float* feat_j; float cx, cy, cz;
    // FP
    const float* p1row; const float* r0; const float* r1; const float* r2; float w0, w1, w2;
    // ROWS
    const float* xrow;
};

template <int IN>
__device__ __forceinline__ void row_setup(const TcIo& io, RowCtx<IN>& c) {   // may remap c.row (TC_IN_FP with an order)
    if (!c.valid) return;
    if constexpr (IN == TC_IN_ROWS) {
        c.xrow = io.x + c.row * io.ldx;
    } else if constexpr (IN == TC_IN_SA) {
        const int64_t bs = c.row / io.K;
        const int64_t b = bs / io.S, s = bs % io.S;
        int64_t j = io.idx[c.row];
        j = j < 0 ? 0 : (j >= io.N ? io.N - 1 : j);
        c.xyz_j = io.xyz + b * io.xB + j * io.xN;
        c.feat_j = io.feat ? io.feat + b * io.fB + j * io.fN : nullptr;
        const float* q = io.qxyz + b * io.qB + s * io.qN;
        c.cx = q[0];
        c.cy = q[io.qC];
        c.cz = q[2 * io.qC];
    } else {
        const int64_t b = c.row / io.seg_rows;
        int64_t n = c.row % io.seg_rows;
        if (io.order) {   // spatially sorted processing order: the rows of a warp share their coarse neighbours
            n = io.order[b * io.order_bs + n * io.order_es];
            n = n < 0 ? 0 : (n >= io.seg_rows ? io.seg_rows - 1 : n);
            c.row = b * io.seg_rows + n;
        }
        c.p1row = io.p1 ? io.p1 + b * io.p1B + n * io.p1N : nullptr;
        int64_t j0 = io.idx3[c.row * 3], j1 = io.idx3[c.row * 3 + 1], j2 = io.idx3[c.row * 3 + 2];
        const int64_t hi = io.S2 - 1;
        j0 = j0 < 0 ? 0 : (j0 > hi ? hi : j0);
        j1 = j1 < 0 ? 0 : (j1 > hi ? hi : j1);
        j2 = j2 < 0 ? 0 : (j2 > hi ? hi : j2);
        c.r0 = io.p2 + b * io.p2B + j0 * io.p2N;
        c.r1 = io.p2 + b * io.p2B + j1 * io.p2N;
        c.r2 = io.p2 + b * io.p2B + j2 * io.p2N;
        c.w0 = io.w3[c.row * 3];
        c.w1 = io.w3[c.row * 3 + 1];
        c.w2 = io.w3[c.row * 3 + 2];
    }
}

// value of input channel k of this thread's row (0 beyond the real channels / rows)
template <int IN>
__device__ __forceinline__ float row_value(const TcIo& io, const RowCtx<IN>& c, int k, int k_real) {
    if (!c.valid || k >= k_real) return 0.0f;
    if constexpr (IN == TC_IN_ROWS) {
        return c.xrow[k];
    } else if constexpr (IN == TC_IN_SA) {
        const int kx = io.msg_order ? k - io.D : k;   // channel inside the recentred-xyz block if 0 <= kx < 3
        if (kx >= 0 && kx < 3) {
            const float p = c.xyz_j[kx * io.xC];
            return __fsub_rn(p, kx == 0 ? c.cx : (kx == 1 ? c.cy : c.cz));
        }
        return c.feat_j[(io.msg_order ? k : k - 3) * io.fC];
    } else {
        if (k < io.D1) return c.p1row[k * io.p1C];
        const int d = k - io.D1;
        const float v = __fadd_rn(__fadd_rn(__fmul_rn(c.r0[d * io.p2C], c.w0), __fmul_rn(c.r1[d * io.p2C], c.w1)),
                                  __fmul_rn(c.r2[d * io.p2C], c.w2));
        return io.relu_in ? fmaxf(v, 0.0f) : v;
    }
}

// 32 consecutive input channels starting at k0 (vectorised fast paths for contiguous rows)
template <int IN>
__device__ __forceinline__ void row_load32(const TcIo& io, const RowCtx<IN>& c, int k0, int k_real, float (&v)[32]) {
    if constexpr (IN == TC_IN_ROWS) {
        if (c.valid && k0 + 32 <= k_real && ((reinterpret_cast<uintptr_t>(c.xrow + k0) & 15) == 0)) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 t = *reinterpret_cast<const float4*>(c.xrow + k0 + 4 * j);
                v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
            }
            return;
        }
    }
    if constexpr (IN == TC_IN_FP) {
        const int d0 = k0 - io.D1;
        if (c.valid && d0 >= 0 && k0 + 32 <= k_real && io.p2C == 1 &&
            (((reinterpret_cast<uintptr_t>(c.r0 + d0) | reinterpret_cast<uintptr_t>(c.r1 + d0) |
               reinterpret_cast<uintptr_t>(c.r2 + d0)) & 15) == 0)) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 a = *reinterpret_cast<const float4*>(c.r0 + d0 + 4 * j);
                const float4 b = *reinterpret_cast<const float4*>(c.r1 + d0 + 4 * j);
                const float4 e = *reinterpret_cast<const float4*>(c.r2 + d0 + 4 * j);
                v[4 * j] = __fadd_rn(__fadd_rn(__fmul_rn(a.x, c.w0), __fmul_rn(b.x, c.w1)), __fmul_rn(e.x, c.w2));
                v[4 * j + 1] = __fadd_rn(__fadd_rn(__fmul_rn(a.y, c.w0), __fmul_rn(b.y, c.w1)), __fmul_rn(e.y, c.w2));
                v[4 * j + 2] = __fadd_rn(__fadd_rn(__fmul_rn(a.z, c.w0), __fmul_rn(b.z, c.w1)), __fmul_rn(e.z, c.w2));
                v[4 * j + 3] = __fadd_rn(__fadd_rn(__fmul_rn(a.w, c.w0), __fmul_rn(b.w, c.w1)), __fmul_rn(e.w, c.w2));
            }
            if (io.relu_in) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.0f);
            }
            return;
        }
        if (c.valid && k0 + 32 <= io.D1 && io.p1C == 1 && ((reinterpret_cast<uintptr_t>(c.p1row + k0) & 15) == 0)) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 t = *reinterpret_cast<const float4*>(c.p1row + k0 + 4 * j);
                v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
            }
            return;
        }
    }
    if constexpr (IN == TC_IN_SA) {
        if (io.msg_order && k0 == io.D) {   // the chunk that starts at the recentred coordinates: [dx, dy, dz, padding], no branches
            const float px = c.valid ? c.xyz_j[0] : 0.0f, py = c.valid ? c.xyz_j[io.xC] : 0.0f, pz = c.valid ? c.xyz_j[2 * io.xC] : 0.0f;
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = 0.0f;
            if (c.valid) {
                v[0] = __fsub_rn(px, c.cx);
                v[1] = __fsub_rn(py, c.cy);
                v[2] = __fsub_rn(pz, c.cz);
            }
            return;
        }
        const int f0 = io.msg_order ? k0 : k0 - 3;   // first feature channel covered if the block is all features
        const bool all_feat = io.msg_order ? (k0 + 32 <= io.D) : (k0 >= 3 && k0 + 32 <= k_real);
        if (c.valid && all_feat && io.fC == 1 && ((reinterpret_cast<uintptr_t>(c.feat_j + f0) & 15) == 0)) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 t = *reinterpret_cast<const float4*>(c.feat_j + f0 + 4 * j);
                v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
            }
            return;
        }
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = row_value<IN>(io, c, k0 + j, k_real);
}

// Fast path of the set-abstraction producer for levels whose whole input row fits one 32-channel chunk with at most four
// feature channels (sa1 of every net: xyz alone or xyz + reflectance / normals).  The generic path (row_setup + row_value per
// channel) branches per element, and every branch ends a basic block: index -> centroid -> coordinates -> features became a
// chain of dependent round trips (the producer was half of sa1's tile time).  Here the index is the only dependency: the
// point's coordinates, its features and the centroid are loaded unconditionally (a row beyond the end is clamped to row 0
// and zeroed afterwards) right after it, in one round trip.  Channel order: [features (D), xyz - centroid (3)], i.e.
// msg_order = 1, which is how every SA chain is packed (FoldedLayers.chain(xyz_last=True)).
__device__ __forceinline__ void sa_small_row(const TcIo& io, bool valid, int64_t row, float (&v)[32]) {
    const int64_t r = valid ? row : 0;
    const int64_t bs = r / io.K;
    const int64_t b = bs / io.S, s = bs % io.S;
    int64_t j = io.idx[r];
    j = j < 0 ? 0 : (j >= io.N ? io.N - 1 : j);
    const float* pj = io.xyz + b * io.xB + j * io.xN;
    const float* q = io.qxyz + b * io.qB + s * io.qN;
    const float* fj = io.feat ? io.feat + b * io.fB + j * io.fN : pj;
    const int64_t fc = io.feat ? io.fC : 0;
    const float f0 = fj[0], f1 = fj[io.D > 1 ? fc : 0], f2 = fj[io.D > 2 ? 2 * fc : 0], f3 = fj[io.D > 3 ? 3 * fc : 0];
    const float dx = __fsub_rn(pj[0], q[0]), dy = __fsub_rn(pj[io.xC], q[io.qC]), dz = __fsub_rn(pj[2 * io.xC], q[2 * io.qC]);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = 0.0f;
    if (valid) {
        switch (io.D) {     // warp-uniform; no loads inside
            case 0: v[0] = dx; v[1] = dy; v[2] = dz; break;
            case 1: v[0] = f0; v[1] = dx; v[2] = dy; v[3] = dz; break;
            case 2: v[0] = f0; v[1] = f1; v[2] = dx; v[3] = dy; v[4] = dz; break;
            case 3: v[0] = f0; v[1] = f1; v[2] = f2; v[3] = dx; v[4] = dy; v[5] = dz; break;
            default: v[0] = f0; v[1] = f1; v[2] = f2; v[3] = f3; v[4] = dx; v[5] = dy; v[6] = dz; break;
        }
    }
}

// ------------------------------------------------------------------------------------------------ quad producer
// tcgen05.st.16x256b.x1: the warp stores a 16-lane x 8-column block; thread t provides {row t/4: columns 2(t%4),
// 2(t%4)+1; row t/4 + 8: the same columns} (pinned on hardware with tools/probes/st_shape_probe.cu).  With packed
// bf16 pairs two columns are four consecutive channels = one float4, so the four threads of a quad read 64
// CONTIGUOUS bytes of a source row and a warp-wide load touches 8 rows instead of 32: the row-per-thread producer
// is bound by L1 tag lookups (32 distinct lines per load instruction), this one needs a quarter of them.
__device__ __forceinline__ void tc_split4(const float4 v, unsigned& h0, unsigned& h1, unsigned& l0, unsigned& l1) {
    tc::split_bf16x2(v.x, v.y, h0, l0);
    tc::split_bf16x2(v.z, v.w, h1, l1);
}

// log_softmax over the first n_real (<= 32) accumulator columns of the 16 TMEM lanes at `taddr`, quad layout: the four
// threads of a quad share a row (8 classes each), so the row max / sum are two xor-shuffles, one TMEM read instead
// of three, and a warp-wide store touches 8 output rows instead of 32.  rowA / rowB: output rows (or -1) of the two
// rows this thread serves (lanes t/4 and t/4 + 8 of the block).
__device__ __forceinline__ void tc_logsoftmax_quad(unsigned taddr, const float* bias, int n_real, int lane, int64_t rowA,
                                                   int64_t rowB, float* y, int64_t ldy) {
    unsigned r[16];
    tc::ld_16x256_x4(taddr, r);
    const int qd = lane & 3;
    float v[2][8];
    float mx[2] = {-CUDART_INF_F, -CUDART_INF_F};
#pragma unroll
    for (int m = 0; m < 4; ++m)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const int col = 8 * m + 2 * qd + c;
            const float b = bias[col];
#pragma unroll
            for (int rb = 0; rb < 2; ++rb) {
                const float f = col < n_real ? __uint_as_float(r[4 * m + 2 * rb + c]) + b : -CUDART_INF_F;
                v[rb][2 * m + c] = f;
                mx[rb] = fmaxf(mx[rb], f);
            }
        }
#pragma unroll
    for (int rb = 0; rb < 2; ++rb) {
        mx[rb] = fmaxf(mx[rb], __shfl_xor_sync(0xffffffffu, mx[rb], 1));
        mx[rb] = fmaxf(mx[rb], __shfl_xor_sync(0xffffffffu, mx[rb], 2));
    }
    float sm[2] = {0.0f, 0.0f};
#pragma unroll
    for (int rb = 0; rb < 2; ++rb)
#pragma unroll
        for (int i = 0; i < 8; ++i) sm[rb] += __expf(v[rb][i] - mx[rb]);     // exp(-inf) = 0 for the padding classes
#pragma unroll
    for (int rb = 0; rb < 2; ++rb) {
        sm[rb] += __shfl_xor_sync(0xffffffffu, sm[rb], 1);
        sm[rb] += __shfl_xor_sync(0xffffffffu, sm[rb], 2);
    }
#pragma unroll
    for (int rb = 0; rb < 2; ++rb) {
        const int64_t row = rb ? rowB : rowA;
        if (row < 0) continue;
        const float ls = __logf(sm[rb]);
        float* dst = y + row * ldy;
#pragma unroll
        for (int m = 0; m < 4; ++m)
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int col = 8 * m + 2 * qd + c;
                if (col < n_real) dst[col] = (v[rb][2 * m + c] - mx[rb]) - ls;
            }
    }
}

struct FpQuadRow {   // one of the four rows a thread serves
    const float* p1row; const float* r0; const float* r1; const float* r2;
    float w0, w1, w2;
    bool valid;
};

__device__ __forceinline__ void fp_quad_row_setup(const TcIo& io, int64_t seg, int64_t r_in_seg, FpQuadRow& q) {
    q.valid = r_in_seg < io.seg_rows;
    q.p1row = nullptr;
    q.r0 = q.r1 = q.r2 = io.p2;
    q.w0 = q.w1 = q.w2 = 0.0f;
    if (!q.valid) return;
    int64_t n = r_in_seg;
    if (io.order) {
        n = io.order[seg * io.order_bs + n * io.order_es];
        n = n < 0 ? 0 : (n >= io.seg_rows ? io.seg_rows - 1 : n);
    }
    const int64_t row = seg * io.seg_rows + n;
    if (io.p1) q.p1row = io.p1 + seg * io.p1B + n * io.p1N;
    int64_t j0 = io.idx3[row * 3], j1 = io.idx3[row * 3 + 1], j2 = io.idx3[row * 3 + 2];
    const int64_t hi = io.S2 - 1;
    j0 = j0 < 0 ? 0 : (j0 > hi ? hi : j0);
    j1 = j1 < 0 ? 0 : (j1 > hi ? hi : j1);
    j2 = j2 < 0 ? 0 : (j2 > hi ? hi : j2);
    q.r0 = io.p2 + seg * io.p2B + j0 * io.p2N;
    q.r1 = io.p2 + seg * io.p2B + j1 * io.p2N;
    q.r2 = io.p2 + seg * io.p2B + j2 * io.p2N;
    q.w0 = io.w3[row * 3];
    q.w1 = io.w3[row * 3 + 1];
    q.w2 = io.w3[row * 3 + 2];
}

// channels [k, k+4) of the row: skip features, interpolated features (same fp32 operation order as row_value) or zero padding
__device__ __forceinline__ float4 fp_quad_value(const TcIo& io, const FpQuadRow& q, int k, int k_real) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!q.valid || k >= k_real) return v;
    if (k < io.D1) return *reinterpret_cast<const float4*>(q.p1row + k);
    const int d = k - io.D1;
    const float4 a = *reinterpret_cast<const float4*>(q.r0 + d);
    const float4 b = *reinterpret_cast<const float4*>(q.r1 + d);
    const float4 e = *reinterpret_cast<const float4*>(q.r2 + d);
    v.x = __fadd_rn(__fadd_rn(__fmul_rn(a.x, q.w0), __fmul_rn(b.x, q.w1)), __fmul_rn(e.x, q.w2));
    v.y = __fadd_rn(__fadd_rn(__fmul_rn(a.y, q.w0), __fmul_rn(b.y, q.w1)), __fmul_rn(e.y, q.w2));
    v.z = __fadd_rn(__fadd_rn(__fmul_rn(a.z, q.w0), __fmul_rn(b.z, q.w1)), __fmul_rn(e.z, q.w2));
    v.w = __fadd_rn(__fadd_rn(__fmul_rn(a.w, q.w0), __fmul_rn(b.w, q.w1)), __fmul_rn(e.w, q.w2));
    if (io.relu_in) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
    return v;
}

// The warp fills its 32 TMEM lanes (tile rows row0 .. row0+31 of segment `seg`) of the A region for the channel
// groups cg = cg0, cg0 + cgstep, ... of 16 channels each of the chunk [kbase, kbase + kchunk).  t_ahi / t_alo: the warp's
// lane-0 addresses of the regions.
__device__ __forceinline__ void fp_quad_producer(const TcIo& io, int64_t seg, int64_t row0, int lane, int kbase, int kchunk,
                                                 int k_real, int cg0, int cgstep, unsigned t_ahi, unsigned t_alo) {
    const int qd = lane & 3, rq = lane >> 2;
    FpQuadRow R[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) fp_quad_row_setup(io, seg, row0 + rq + 8 * i, R[i]);
    for (int cg = cg0; cg * 16 < kchunk; cg += cgstep) {   // channels [kbase, kbase + kchunk) -> A columns [0, kchunk / 2)
        const int k = kbase + cg * 16 + qd * 4;
        float4 v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = fp_quad_value(io, R[i], k, k_real);
#pragma unroll
        for (int blk = 0; blk < 2; ++blk) {
            unsigned ha0, ha1, la0, la1, hb0, hb1, lb0, lb1;
            tc_split4(v[2 * blk], ha0, ha1, la0, la1);
            tc_split4(v[2 * blk + 1], hb0, hb1, lb0, lb1);
            const unsigned off = ((unsigned)(blk * 16) << 16) + (unsigned)cg * 8;
            tc::st_16x256(t_ahi + off, ha0, ha1, hb0, hb1);
            tc::st_16x256(t_alo + off, la0, la1, lb0, lb1);
        }
    }
}

// Fast path of the quad producer for levels WITHOUT skip input whose channel count fills whole 16-channel groups (fp1 of the
// segmentation nets: 24000 rows per cloud, the hot case).  The generic path above decides per row and per channel group
// (valid? skip or interpolated? padding?), and every such branch ends a basic block: ptxas then issues a row's loads, waits
// for them and only then turns to the next row -- ~26 dependent L2 round trips per tile (measured: 11.3 k cycles per 128-row
// tile, the same for one warp group as for two: pure latency).  Here nothing branches: invalid rows are clamped to the last
// valid row and given zero weights, so the 24 index / weight loads of a thread's four rows are issued back to back, and so are
// the twelve 16-byte row loads of every channel group.
__device__ __forceinline__ void fp_quad_producer_fast(const TcIo& io, int64_t seg, int64_t row0, int lane, int kchunk, int cg0,
                                                      int cgstep, unsigned t_ahi, unsigned t_alo, long long* stamps = nullptr) {
    const int qd = lane & 3, rq = lane >> 2;
    const float* src[4][3];
    float wgt[4][3];
    const int64_t hi = io.S2 - 1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t r_in_seg = row0 + rq + 8 * i;
        const bool valid = r_in_seg < io.seg_rows;
        const int64_t row = seg * io.seg_rows + (valid ? r_in_seg : io.seg_rows - 1);
        const int64_t* ip = io.idx3 + row * 3;
        const float* wp = io.w3 + row * 3;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            int64_t j = ip[k];
            j = j < 0 ? 0 : (j > hi ? hi : j);
            src[i][k] = io.p2 + seg * io.p2B + j * io.p2N + qd * 4;
            const float w = wp[k];
            wgt[i][k] = valid ? w : 0.0f;
        }
    }
    const float floor_v = io.relu_in ? 0.0f : -CUDART_INF_F;   // relu(v) = max(v, 0); identity = max(v, -inf)
    if (stamps) { if (wgt[0][0] + wgt[1][1] + wgt[2][2] + wgt[3][0] > -1.0f && src[0][0] != nullptr && src[3][2] != nullptr) *stamps++ = clock64(); }
    for (int cg = cg0; cg * 16 < kchunk; cg += cgstep) {
        float4 a[4][3];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 3; ++k) a[i][k] = *reinterpret_cast<const float4*>(src[i][k] + cg * 16);
        float4 v[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {   // same fp32 operation order as row_value / fp_quad_value
            v[i].x = fmaxf(__fadd_rn(__fadd_rn(__fmul_rn(a[i][0].x, wgt[i][0]), __fmul_rn(a[i][1].x, wgt[i][1])), __fmul_rn(a[i][2].x, wgt[i][2])), floor_v);
            v[i].y = fmaxf(__fadd_rn(__fadd_rn(__fmul_rn(a[i][0].y, wgt[i][0]), __fmul_rn(a[i][1].y, wgt[i][1])), __fmul_rn(a[i][2].y, wgt[i][2])), floor_v);
            v[i].z = fmaxf(__fadd_rn(__fadd_rn(__fmul_rn(a[i][0].z, wgt[i][0]), __fmul_rn(a[i][1].z, wgt[i][1])), __fmul_rn(a[i][2].z, wgt[i][2])), floor_v);
            v[i].w = fmaxf(__fadd_rn(__fadd_rn(__fmul_rn(a[i][0].w, wgt[i][0]), __fmul_rn(a[i][1].w, wgt[i][1])), __fmul_rn(a[i][2].w, wgt[i][2])), floor_v);
        }
#pragma unroll
        for (int blk = 0; blk < 2; ++blk) {
            unsigned ha0, ha1, la0, la1, hb0, hb1, lb0, lb1;
            tc_split4(v[2 * blk], ha0, ha1, la0, la1);
            tc_split4(v[2 * blk + 1], hb0, hb1, lb0, lb1);
            const unsigned off = ((unsigned)(blk * 16) << 16) + (unsigned)cg * 8;
            tc::st_16x256(t_ahi + off, ha0, ha1, hb0, hb1);
            tc::st_16x256(t_alo + off, la0, la1, lb0, lb1);
        }
        if (stamps) *stamps++ = clock64();
    }
}

// ------------------------------------------------------------------------------------------------ the kernel
// THREADS = 256 (8 warps, two CTAs per SM) or 512 (16 warps, one CTA per SM: used when the grid has at most one CTA per
// SM anyway -- twice the warps halve the latency-bound producer and epilogue phases of the small levels).
template <int IN, int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? 2 : 1)
mlp_tc_kernel(const __grid_constant__ TcChain ch, const unsigned char* __restrict__ blob, const __grid_constant__ TcIo io) {
    extern __shared__ __align__(128) unsigned char smem[];
    // layout: [stage 0 .. nstages-1][bias table][barriers: full[8] empty[8] done][tmem ptr]
    const int NS = ch.nstages;
    float* sbias = reinterpret_cast<float*>(smem + NS * ch.stage_bytes);
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + NS * ch.stage_bytes + ((ch.bias_floats * 4 + 15) & ~15));
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 2 * kTcMaxStages + 1);
    const unsigned bar_full0 = tc::smem_u32(&bars[0]), bar_empty0 = tc::smem_u32(&bars[kTcMaxStages]);   // stage st: + 8 st bytes
    const unsigned bar_done = tc::smem_u32(&bars[2 * kTcMaxStages]);
    const unsigned stage0 = tc::smem_u32(smem);

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler: MMA operands stay in uniform registers
    if (warp == 0) tc::tmem_alloc(tmem_slot, ch.tmem_cols);
    if (tid == 0) {
        for (int st = 0; st < NS; ++st) {
            tc::mbar_init(bar_full0 + 8 * st, 1);
            tc::mbar_init(bar_empty0 + 8 * st, 1);
        }
        tc::mbar_init(bar_done, 1);
        tc::mbar_init_fence();
    }
    {
        const float* gb = reinterpret_cast<const float*>(blob + ch.bias_off);
        for (int i = tid; i < ch.bias_floats; i += THREADS) sbias[i] = gb[i];
    }
    tc::fence_before();
    __syncthreads();
    tc::fence_after();
    const unsigned tbase = __shfl_sync(0xffffffffu, *tmem_slot, 0);
    constexpr int HALVES = THREADS / 128, CSTEP = 32 * HALVES;
    const int wl = warp & 3, half = warp >> 2;                      // lane quarter / column slice (of HALVES) of this warp
    const unsigned tlane = tbase + ((unsigned)(wl * 32) << 16);      // this warp's 32 TMEM lanes
    const unsigned t_x = tlane;                                      // accumulator columns
    const unsigned t_ahi = tlane + ch.x_cols, t_alo = t_ahi + ch.a_lo_off;
    const unsigned a_hi_col = tbase + ch.x_cols, a_lo_col = a_hi_col + ch.a_lo_off;   // lane 0 addresses for the MMA

    // ring bookkeeping: `fill` lives in the copy thread (warp 4, lane 0), `use` in the MMA thread (warp 0, lane 0); both walk
    // the same static schedule of (tile, layer, pass, chunk, slice), so slice number i always sits in stage i % NS
    unsigned fill = 0, use = 0, fill_st = 0, use_st = 0, done_phase = 0;
    int nlog = 0;
    auto stamp = [&](int tag) {   // pn_launch_opts.mlp_debug: flat (tag, clock) log of CTA 0, thread 0
        if (io.dbg != nullptr && blockIdx.x == 0 && tid == 0 && nlog < 500) {
            io.dbg[1 + 2 * nlog] = tag;
            io.dbg[2 + 2 * nlog] = clock64();
            io.dbg[0] = ++nlog;
        }
    };

    const int64_t tiles_per_seg = (io.seg_rows + 127) / 128;
    const int64_t ntiles = io.nseg * tiles_per_seg;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t seg = tile / tiles_per_seg;
        const int64_t r_in_seg = (tile % tiles_per_seg) * 128 + wl * 32 + lane;
        RowCtx<IN> rc;
        rc.valid = r_in_seg < io.seg_rows;
        rc.row = seg * io.seg_rows + r_in_seg;
        stamp(1);
        row_setup<IN>(io, rc);

        for (int l = 0; l < ch.nlayers; ++l) {
            const TcLayer& L = ch.L[l];
            const bool last = l + 1 == ch.nlayers;
            // output channels are produced in passes of PW columns; with gridDim.y > 1 (single-layer chains on few row
            // tiles) the passes of a tile are spread over the CTAs (tile, y): N-slicing fills the GPU when rows are scarce
            const int PW = ch.pass_w;
            const int npass = (L.n_pad + PW - 1) / PW;
            const int nchunk = (L.k_pad + kTcAChunk - 1) / kTcAChunk;   // > 1 only for a wide first layer
            for (int p = blockIdx.y; p < npass; p += gridDim.y) {
                const int n0 = p * PW;                                   // first output channel of the pass
                const int rows_p = min(PW, L.n_pad - n0);
                for (int a = 0; a < nchunk; ++a) {
                    const int kbase = a * kTcAChunk;
                    const int kchunk = min(kTcAChunk, L.k_pad - kbase);
                    if (l == 0) {
                        // ---- producer: channels [kbase, kbase + kchunk) of the tile's rows -> TMEM A region
                        bool quad = false;
                        if constexpr (IN == TC_IN_FP) quad = io.quad_fp != 0;
                        if (quad) {
                            fp_quad_producer(io, seg, (tile % tiles_per_seg) * 128 + wl * 32, lane, kbase, kchunk, L.k_real, half, HALVES,
                                             t_ahi, t_alo);
                        } else {
                            for (int k0 = half * 32; k0 < kchunk; k0 += CSTEP) {   // this thread's row
                                float v[32];
                                row_load32<IN>(io, rc, kbase + k0, L.k_real, v);
                                tc::store_split32(t_ahi + k0 / 2, t_alo + k0 / 2, v);
                            }
                        }
                        tc::wait_st();
                        tc::fence_before();
                        __syncthreads();
                        stamp(2);
                    }
                    const int s0 = kbase / kTcKSub, ns = (kchunk + kTcKSub - 1) / kTcKSub;
                    if (warp == 4) {
                        // ---- copy warp (all lanes walk the loop, one elected lane issues): the weight slices of this chunk, one
                        // or two cp.async.bulk (TMA engine) each, running up to NS slices ahead of the tensor core; a stage is
                        // reused once the MMAs that read it have completed.
                        // The blob stores 256-row blocks: [block P][slice][hi image | lo image]; rows [r0, r0 + rows_p) of a
                        // slice image are contiguous (8-row groups are the outer dimension of the core-matrix layout).
                        const int P = n0 / kTcNPass, r0 = n0 % kTcNPass;
                        const int rows_P = min(kTcNPass, L.n_pad - P * kTcNPass);
                        const unsigned char* wpass = blob + L.w_off + (size_t)P * kTcNPass * L.k_pad * 4;
                        for (int s = 0; s < ns; ++s) {
                            const int kw = min(kTcKSub, L.k_pad - (s0 + s) * kTcKSub);
                            const unsigned bytes = (unsigned)rows_p * kw * 4;
                            const unsigned char* src = wpass + (size_t)rows_P * ((s0 + s) * kTcKSub) * 4 + (size_t)r0 * kw * 2;
                            const unsigned dst = stage0 + fill_st * (unsigned)ch.stage_bytes;
                            const unsigned full = bar_full0 + 8 * fill_st;
                            tc::mbar_wait(bar_empty0 + 8 * fill_st, ((fill / NS) & 1) ^ 1);
                            if (tc::elect()) {
                                tc::mbar_arrive_expect_tx(full, bytes);
                                if (rows_p == rows_P) {   // hi and lo images are adjacent: one copy
                                    tc::bulk_load(dst, src, bytes, full);
                                } else {
                                    tc::bulk_load(dst, src, bytes / 2, full);
                                    tc::bulk_load(dst + bytes / 2, src + (size_t)rows_P * kw * 2, bytes / 2, full);
                                }
                            }
                            __syncwarp();
                            ++fill;
                            fill_st = fill_st + 1 == (unsigned)NS ? 0u : fill_st + 1;
                        }
                    }
                    if (warp == 0) {
                        // ---- MMA warp (same scheme): the MMAs of a slice are issued as soon as it has landed
                        tc::fence_after();
                        const unsigned idesc = tc::idesc_bf16_f32(128, rows_p);
                        for (int s = 0; s < ns; ++s) {
                            const int kw = min(kTcKSub, L.k_pad - (s0 + s) * kTcKSub);
                            tc::mbar_wait(bar_full0 + 8 * use_st, (use / NS) & 1);
                            tc::fence_after();
                            stamp(6);
                            const unsigned b_hi = stage0 + use_st * (unsigned)ch.stage_bytes, b_lo = b_hi + (unsigned)rows_p * kw * 2;
                            const unsigned long long dbase = tc::sdesc_base(((unsigned)kw / 8) * 128u);
                            if (tc::elect()) {
                                for (int t = 0; t < kw / 16; ++t) {
                                    const unsigned kcol = (unsigned)(s * kTcKSub + t * 16) / 2;   // A columns of this K step
                                    const unsigned long long dh = tc::sdesc(dbase, b_hi + t * 256), dl = tc::sdesc(dbase, b_lo + t * 256);
                                    const unsigned acc0 = (a > 0 || s > 0 || t > 0) ? 1u : 0u;
                                    tc::mma_bf16x3(tbase, a_hi_col + kcol, a_lo_col + kcol, dh, dl, idesc, acc0, ch.split);
                                }
                                tc::commit(bar_empty0 + 8 * use_st);
                                if (s + 1 == ns) tc::commit(bar_done);
                            }
                            __syncwarp();
                            stamp(7);
                            ++use;
                            use_st = use_st + 1 == (unsigned)NS ? 0u : use_st + 1;
                        }
                        stamp(3);
                    }
                    // ---- everyone waits for this chunk's MMAs (the A region / accumulator are then free to touch)
                    tc::mbar_wait(bar_done, done_phase);
                    done_phase ^= 1;
                    tc::fence_after();
                    stamp(4);
                }
                // ---- epilogue of pass p: accumulator columns [0, rows_p)
                const float* bias = sbias + L.b_off + n0;
                if (!last) {
                    for (int c0 = half * 32; c0 < rows_p; c0 += CSTEP) {
                        unsigned r[32];
                        tc::ld32(t_x + c0, r);
                        float v[32];
                        if (l == 0 && io.res != nullptr) {   // the skip half of the layer, computed beforehand per row
                            const float4* rr = reinterpret_cast<const float4*>(io.res + (rc.valid ? rc.row : 0) * io.ldr + n0 + c0);
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const float4 t = rr[j];
                                r[4 * j] = __float_as_uint(__uint_as_float(r[4 * j]) + t.x);
                                r[4 * j + 1] = __float_as_uint(__uint_as_float(r[4 * j + 1]) + t.y);
                                r[4 * j + 2] = __float_as_uint(__uint_as_float(r[4 * j + 2]) + t.z);
                                r[4 * j + 3] = __float_as_uint(__uint_as_float(r[4 * j + 3]) + t.w);
                            }
                        }
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float f = __uint_as_float(r[j]) + bias[c0 + j];
                            v[j] = L.relu ? fmaxf(f, 0.0f) : f;
                        }
                        tc::store_split32(t_ahi + c0 / 2, t_alo + c0 / 2, v);
                    }
                    tc::wait_st();
                    tc::fence_before();
                    __syncthreads();
                } else if (io.out_mode == TC_OUT_ROWS) {
                    for (int c0 = half * 32; c0 < rows_p; c0 += CSTEP) {
                        unsigned r[32];
                        tc::ld32(t_x + c0, r);
                        if (rc.valid) {
                            float* dst = io.y + rc.row * io.ldy + n0 + c0;
                            const int nleft = L.n_real - (n0 + c0);
                            const bool vec = nleft >= 32 && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0);
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                float4 o;
                                o.x = __uint_as_float(r[j]) + bias[c0 + j];
                                o.y = __uint_as_float(r[j + 1]) + bias[c0 + j + 1];
                                o.z = __uint_as_float(r[j + 2]) + bias[c0 + j + 2];
                                o.w = __uint_as_float(r[j + 3]) + bias[c0 + j + 3];
                                if (L.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                                if (vec) {
                                    *reinterpret_cast<float4*>(dst + j) = o;
                                } else {
                                    if (j < nleft) dst[j] = o.x;
                                    if (j + 1 < nleft) dst[j + 1] = o.y;
                                    if (j + 2 < nleft) dst[j + 2] = o.z;
                                    if (j + 3 < nleft) dst[j + 3] = o.w;
                                }
                            }
                        }
                    }
                    tc::fence_before();
                    __syncthreads();
                } else if (io.out_mode == TC_OUT_MAX) {
                    // group = 32 consecutive rows = this warp: REDUX max per channel, lane j keeps channel c0 + j
                    const int64_t grp = rc.row / 32;   // warp-uniform when the warp has any valid row
                    const bool any_valid = __any_sync(0xffffffffu, rc.valid);
                    const int64_t g = __shfl_sync(0xffffffffu, grp, 0);
                    for (int c0 = half * 32; c0 < rows_p; c0 += CSTEP) {
                        unsigned r[32];
                        tc::ld32(t_x + c0, r);
                        if (io.group == 16) {
                            tc_store_max16(r, bias, L.relu, rc.valid, rc.row, lane, c0, L.n_real - n0, io.y + n0, io.ldy);
                            continue;
                        }
                        // max first, bias + ReLU on the one survivor: x -> relu(fl(x + b)) is monotone, so the result is bit-identical
                        float v[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = rc.valid ? __uint_as_float(r[j]) : -CUDART_INF_F;
                        float mine = tc_colmax32(v, lane) + bias[c0 + lane];
                        if (L.relu) mine = fmaxf(mine, 0.0f);
                        const int n = n0 + c0 + lane;
                        if (any_valid && n < L.n_real) io.y[g * io.ldy + n] = mine;
                    }
                    tc::fence_before();
                    __syncthreads();
                } else {   // TC_OUT_LOGSOFTMAX over the n_real (<= 64) classes of the row: column-half 0 warps only
                    if (half == 0) {
                        float m = -CUDART_INF_F, ssum = 0.0f;
                        for (int c0 = 0; c0 < rows_p; c0 += 32) {
                            unsigned r[32];
                            tc::ld32(t_x + c0, r);
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (c0 + j < L.n_real) m = fmaxf(m, __uint_as_float(r[j]) + bias[c0 + j]);
                        }
                        for (int c0 = 0; c0 < rows_p; c0 += 32) {
                            unsigned r[32];
                            tc::ld32(t_x + c0, r);
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (c0 + j < L.n_real) ssum += __expf((__uint_as_float(r[j]) + bias[c0 + j]) - m);
                        }
                        const float ls = __logf(ssum);
                        for (int c0 = 0; c0 < rows_p; c0 += 32) {
                            unsigned r[32];
                            tc::ld32(t_x + c0, r);
                            if (rc.valid) {
                                float* dst = io.y + rc.row * io.ldy + c0;
#pragma unroll
                                for (int j = 0; j < 32; ++j)
                                    if (c0 + j < L.n_real) dst[j] = ((__uint_as_float(r[j]) + bias[c0 + j]) - m) - ls;
                            }
                        }
                    }
                    tc::fence_before();
                    __syncthreads();
                }
                stamp(5);
            }
        }
    }
    tc::fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tbase, ch.tmem_cols);
}

// ------------------------------------------------------------------------------------------------ resident kernel
// Chains whose packed weights fit in shared memory (<= ~225 KB: sa1, sa2, fp1 + segmentation head, the PointNet
// per-point chains) do not stream anything: the whole blob (weight images + bias table) is brought in ONCE per CTA
// with cp.async.bulk and stays resident; the CTA is persistent over row tiles.  512 threads form GROUPS independent
// warp groups, each owning its own 128-row tile and its own slice of TMEM (512 / GROUPS columns: accumulator + A
// operand); while one group waits for its MMAs the others run producers / epilogues, so the tensor pipe and the
// issue slots overlap without any hand-written software pipeline.  Groups synchronise on named barriers.
//   WPG = 8: 2 groups, warp gw owns TMEM lanes 32*(gw%4).. and column half gw/4     (x_cols + a_k <= 256)
//   WPG = 4: 4 groups, a thread handles every column of its row                      (x_cols + a_k <= 128)
constexpr int kResThreads = 512;

__device__ __forceinline__ void tc_group_bar(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <int IN, int WPG>
__global__ void __launch_bounds__(kResThreads, 1)
mlp_tc_res_kernel(const __grid_constant__ TcChain ch, const unsigned char* __restrict__ blob, const __grid_constant__ TcIo io) {
    constexpr int GROUPS = 16 / WPG, GTHREADS = WPG * 32, HALVES = WPG / 4, GCOLS = 512 / GROUPS, CSTEP = 32 * HALVES;
    extern __shared__ __align__(128) unsigned char smem[];
    // layout: [blob: weight images | bias table][barriers: weights, done[GROUPS]][tmem ptr][next tile of every group]
    const float* sbias = reinterpret_cast<const float*>(smem + ch.bias_off);
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + ((ch.blob_bytes + 15u) & ~15u));
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 1 + GROUPS);
    volatile unsigned* tile_slot = reinterpret_cast<volatile unsigned*>(bars + 6);   // [GROUPS <= 4]
    unsigned* mma_lock = reinterpret_cast<unsigned*>(bars + 8);
    const unsigned bar_w = tc::smem_u32(&bars[0]);
    const unsigned smem_w = tc::smem_u32(smem);

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler: MMA operands stay in uniform registers
    const int g = warp / WPG, gw = warp % WPG;
    const unsigned bar_done = tc::smem_u32(&bars[1 + g]);
    const int64_t tiles_per_seg = (io.seg_rows + 127) / 128;
    const int64_t ntiles = io.nseg * tiles_per_seg;
    // Dynamic tile scheduling (io.tile_ctr): every group draws its tiles from one global counter, so a CTA whose SM was
    // held by another stream's kernel when the launch began only takes what is left when it finally starts.  Every group
    // draws until its first out-of-range ticket: ntiles + gridDim.x * GROUPS draws in total, and whoever receives the
    // last ticket resets the counter for the next launch that is handed the same word.
    const bool dyn = io.tile_ctr != nullptr;
    const unsigned last_ticket = (unsigned)ntiles + gridDim.x * GROUPS - 1u;
    if (warp == 0) tc::tmem_alloc(tmem_slot, 512);
    if (tid == 0) {
        *mma_lock = 0u;
        tc::mbar_init(bar_w, 1);
        for (int i = 0; i < GROUPS; ++i) tc::mbar_init(tc::smem_u32(&bars[1 + i]), 1);
        tc::mbar_init_fence();
        bool any = true;
        if (dyn) {
            any = false;
            for (int i = 0; i < GROUPS; ++i) {
                const unsigned t = atomicAdd(io.tile_ctr, 1u);
                if (t == last_ticket) atomicExch(io.tile_ctr, 0u);
                tile_slot[i] = t;
                any = any || (int64_t)t < ntiles;
            }
        }
        if (any) {   // (a CTA that arrives after the last tile was taken must not leave with a copy in flight)
            tc::bulk_load_pieces(smem_w, blob, ch.blob_bytes, bar_w);     // the whole blob
        }
    }
    tc::fence_before();
    __syncthreads();
    tc::fence_after();
    const unsigned tbase = __shfl_sync(0xffffffffu, *tmem_slot, 0) + (unsigned)(g * GCOLS);
    const int wl = gw & 3, half = gw >> 2;                           // lane quarter (== warp % 4) / column half
    const unsigned tlane = tbase + ((unsigned)(wl * 32) << 16);      // this warp's 32 TMEM lanes
    const unsigned t_x = tlane;                                      // accumulator columns
    const unsigned t_ahi = tlane + ch.x_cols, t_alo = t_ahi + ch.a_lo_off;
    const unsigned a_hi_col = tbase + ch.x_cols, a_lo_col = a_hi_col + ch.a_lo_off;   // lane 0 addresses for the MMA
    unsigned done_phase = 0;
    bool w_ready = false;

    const bool leader = gw == 0 && lane == 0;   // draws the group's tickets (and issues its MMAs)
    int round = 0;
    for (int64_t tile = dyn ? (int64_t)tile_slot[g] : (int64_t)blockIdx.x * GROUPS + g; tile < ntiles; ++round) {
        if ((ch.probe & 2) && g > 0) break;
        // the NEXT tile's ticket is drawn now and only looked at when this tile is finished: the atomic's latency hides
        unsigned next_ticket = 0u;
        if (dyn && leader) next_ticket = atomicAdd(io.tile_ctr, 1u);
        const int64_t seg = tile / tiles_per_seg;
        const int64_t r_in_seg = (tile % tiles_per_seg) * 128 + wl * 32 + lane;
        RowCtx<IN> rc;
        rc.valid = r_in_seg < io.seg_rows;
        rc.row = seg * io.seg_rows + r_in_seg;
        const bool rec = io.dbg != nullptr && blockIdx.x == 0 && gw == 0 && lane == 0;
        long long* drow = io.dbg + (g * 64 + round % 64) * 32;
        int dcol = 0;
        if (rec) drow[dcol++] = clock64();
        bool sa_small = false;
        if constexpr (IN == TC_IN_SA) sa_small = ch.L[0].k_pad == 32 && io.D <= 4 && io.msg_order != 0 && !(ch.probe & 16);
        if (!sa_small) row_setup<IN>(io, rc);

        for (int l = 0; l < ch.nlayers; ++l) {
            const TcLayer& L = ch.L[l];
            const bool last = l + 1 == ch.nlayers;
            if (l == 0 && !(ch.probe & 4)) {
                // ---- producer: rows -> TMEM A region
                bool quad = false;
                if constexpr (IN == TC_IN_FP) quad = io.quad_fp != 0;
                if (quad && io.quad_fp == 2) {
                    fp_quad_producer_fast(io, seg, (tile % tiles_per_seg) * 128 + wl * 32, lane, L.k_pad, half, HALVES, t_ahi, t_alo,
                                          rec ? drow + 22 : nullptr);
                } else if (quad) {
                    fp_quad_producer(io, seg, (tile % tiles_per_seg) * 128 + wl * 32, lane, 0, L.k_pad, L.k_real, half, HALVES,
                                     t_ahi, t_alo);
                } else if (sa_small) {
                    if (half == 0) {
                        float v[32];
                        sa_small_row(io, rc.valid, rc.row, v);
                        tc::store_split32(t_ahi, t_alo, v);
                    }
                } else {
                    for (int k0 = half * 32; k0 < L.k_pad; k0 += CSTEP) {   // this thread's row
                        float v[32];
                        row_load32<IN>(io, rc, k0, L.k_real, v);
                        tc::store_split32(t_ahi + k0 / 2, t_alo + k0 / 2, v);
                    }
                }
                tc::wait_st();
                if (rec) drow[dcol++] = clock64();
                tc::fence_before();
                tc_group_bar(1 + g, GTHREADS);
            }
            if (ch.probe & 1) break;
            if (rec) drow[dcol++] = clock64();
            if (gw == 0) {
                // ---- MMA issue.  The whole warp walks the (warp-uniform) loop and one elected lane issues: every operand of
                // tcgen05.mma then lives in a uniform register.  (Issued from inside an `if (lane == 0)` branch the same loop
                // costs an ELECT + 3 x R2UR.BROADCAST waterfall per MMA, ~90 cycles against the 64 the tensor pipe needs.)
                if (!w_ready) tc::mbar_wait(bar_w, 0);
                // One group issues a whole layer at a time.  Without the lock the groups interleave their MMAs in the tensor
                // queue, both layers complete together and the groups stay in lock-step: MMA phases with idle CUDA cores, then
                // epilogue phases with an idle tensor pipe.  With it the first group's accumulator is ready after one layer's
                // worth of MMAs and its epilogue runs under the second group's: the groups settle half a phase apart.
                // (Two groups only: with four groups of small layers -- sa1 -- the MMAs are too short to be worth serialising and
                // three spinning lanes cost more than they save: 44.0 vs 41.9 us.)
                const bool use_lock = GROUPS == 2 && ch.probe != 8;
                if (use_lock) {
                    if (lane == 0) while (atomicCAS(mma_lock, 0u, 1u) != 0u) {}
                    __syncwarp();
                }
                tc::fence_after();
                const unsigned wl_base = smem_w + L.w_off;
                const unsigned idesc = tc::idesc_bf16_f32(128, L.n_pad);
                const int ns = L.k_pad / kTcKSub;                    // k_pad is a multiple of 32: every slice is 32 wide
                // shared-memory descriptor: LBO = 128 B (next 8 K values), SBO = 512 B (next 8 rows), version bit 46; the
                // start-address field (bits 0-13, 16-byte units) advances by 16 per 16-wide K step, n_pad * 8 per slice,
                // and the lo image of a slice sits n_pad * 4 units after its hi image
                const unsigned d_hi32 = tc::sdesc_hi32((32u / 8) * 128u);
                unsigned d_lo32 = tc::sdesc_lo32(wl_base);
                const unsigned lo_img = (unsigned)L.n_pad * 4u, slice = (unsigned)L.n_pad * 8u;
                const bool issuer = tc::elect();
                unsigned kcol = 0;
                for (int s = 0; s < ns; ++s) {
#pragma unroll
                    for (int t = 0; t < 2; ++t) {
                        const unsigned long long dh = ((unsigned long long)d_hi32 << 32) | (unsigned long long)(d_lo32 + 16u * t);
                        const unsigned long long dl = dh + lo_img;
                        if (issuer)
                            tc::mma_bf16x3(tbase, a_hi_col + kcol, a_lo_col + kcol, dh, dl, idesc, (s > 0 || t > 0) ? 1u : 0u, ch.split);
                        kcol += 8;
                    }
                    d_lo32 += slice;
                }
                if (issuer) tc::commit(bar_done);
                __syncwarp();
                if (use_lock && lane == 0) atomicExch(mma_lock, 0u);
                if (rec) drow[dcol++] = clock64();
            }
            tc::mbar_wait(bar_done, done_phase);
            done_phase ^= 1;
            if (rec) drow[dcol++] = clock64();
            if (!w_ready) {     // the bias table arrived with the weights: every reader observes the barrier once
                tc::mbar_wait(bar_w, 0);
                w_ready = true;
            }
            tc::fence_after();

            // ---- epilogue: accumulator columns [0, n_pad)
            const float* bias = sbias + L.b_off;
            if (!last) {
                for (int c0 = half * 32; c0 < L.n_pad; c0 += CSTEP) {
                    unsigned r[32];
                    tc::ld32(t_x + c0, r);
                    float v[32];
                    if (l == 0 && io.res != nullptr) {   // the skip half of the layer, computed beforehand per row
                        const float4* rr = reinterpret_cast<const float4*>(io.res + (rc.valid ? rc.row : 0) * io.ldr + c0);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float4 t = rr[j];
                            r[4 * j] = __float_as_uint(__uint_as_float(r[4 * j]) + t.x);
                            r[4 * j + 1] = __float_as_uint(__uint_as_float(r[4 * j + 1]) + t.y);
                            r[4 * j + 2] = __float_as_uint(__uint_as_float(r[4 * j + 2]) + t.z);
                            r[4 * j + 3] = __float_as_uint(__uint_as_float(r[4 * j + 3]) + t.w);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float f = __uint_as_float(r[j]) + bias[c0 + j];
                        v[j] = L.relu ? fmaxf(f, 0.0f) : f;
                    }
                    tc::store_split32(t_ahi + c0 / 2, t_alo + c0 / 2, v);
                }
                tc::wait_st();
            } else if (io.out_mode == TC_OUT_ROWS) {
                for (int c0 = half * 32; c0 < L.n_pad; c0 += CSTEP) {
                    unsigned r[32];
                    tc::ld32(t_x + c0, r);
                    if (rc.valid) {
                        float* dst = io.y + rc.row * io.ldy + c0;
                        const int nleft = L.n_real - c0;
                        const bool vec = nleft >= 32 && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0);
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            float4 o;
                            o.x = __uint_as_float(r[j]) + bias[c0 + j];
                            o.y = __uint_as_float(r[j + 1]) + bias[c0 + j + 1];
                            o.z = __uint_as_float(r[j + 2]) + bias[c0 + j + 2];
                            o.w = __uint_as_float(r[j + 3]) + bias[c0 + j + 3];
                            if (L.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                            if (vec) {
                                *reinterpret_cast<float4*>(dst + j) = o;
                            } else {
                                if (j < nleft) dst[j] = o.x;
                                if (j + 1 < nleft) dst[j + 1] = o.y;
                                if (j + 2 < nleft) dst[j + 2] = o.z;
                                if (j + 3 < nleft) dst[j + 3] = o.w;
                            }
                        }
                    }
                }
            } else if (io.out_mode == TC_OUT_MAX) {
                // group = 32 consecutive rows = this warp: REDUX max per channel, lane j keeps channel c0 + j
                const int64_t grp = rc.row / 32;
                const bool any_valid = __any_sync(0xffffffffu, rc.valid);
                const int64_t gi = __shfl_sync(0xffffffffu, grp, 0);
                for (int c0 = half * 32; c0 < L.n_pad; c0 += CSTEP) {
                    unsigned r[32];
                    tc::ld32(t_x + c0, r);
                    if (io.group == 16) {
                        tc_store_max16(r, bias, L.relu, rc.valid, rc.row, lane, c0, L.n_real, io.y, io.ldy);
                        continue;
                    }
                    // max first, bias + ReLU on the one survivor: x -> relu(fl(x + b)) is monotone, so the result is bit-identical
                    float v[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = rc.valid ? __uint_as_float(r[j]) : -CUDART_INF_F;
                    float mine = tc_colmax32(v, lane) + bias[c0 + lane];
                    if (L.relu) mine = fmaxf(mine, 0.0f);
                    const int n = c0 + lane;
                    if (any_valid && n < L.n_real) io.y[gi * io.ldy + n] = mine;
                }
            } else if (L.n_pad == 32) {   // TC_OUT_LOGSOFTMAX, up to 32 classes: quad layout, every warp takes part
                const int64_t orow = rc.valid ? rc.row : -1;
#pragma unroll
                for (int blk = 0; blk < 2; ++blk) {
                    // (shuffles are executed by the whole warp; with two column-half warps each takes one 16-lane block)
                    const int64_t rowA = __shfl_sync(0xffffffffu, orow, blk * 16 + (lane >> 2));
                    const int64_t rowB = __shfl_sync(0xffffffffu, orow, blk * 16 + (lane >> 2) + 8);
                    if (HALVES == 1 || half == blk)
                        tc_logsoftmax_quad(t_x + ((unsigned)(blk * 16) << 16), bias, L.n_real, lane, rowA, rowB, io.y, io.ldy);
                }
            } else {   // TC_OUT_LOGSOFTMAX over the n_real (<= 64) classes of the row: column-half 0 warps only
                if (half == 0) {
                    float m = -CUDART_INF_F, ssum = 0.0f;
                    for (int c0 = 0; c0 < L.n_pad; c0 += 32) {
                        unsigned r[32];
                        tc::ld32(t_x + c0, r);
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (c0 + j < L.n_real) m = fmaxf(m, __uint_as_float(r[j]) + bias[c0 + j]);
                    }
                    for (int c0 = 0; c0 < L.n_pad; c0 += 32) {
                        unsigned r[32];
                        tc::ld32(t_x + c0, r);
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (c0 + j < L.n_real) ssum += __expf((__uint_as_float(r[j]) + bias[c0 + j]) - m);
                    }
                    const float ls = __logf(ssum);
                    for (int c0 = 0; c0 < L.n_pad; c0 += 32) {
                        unsigned r[32];
                        tc::ld32(t_x + c0, r);
                        if (rc.valid) {
                            float* dst = io.y + rc.row * io.ldy + c0;
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (c0 + j < L.n_real) dst[j] = ((__uint_as_float(r[j]) + bias[c0 + j]) - m) - ls;
                        }
                    }
                }
            }
            if (rec) drow[dcol++] = clock64();
            if (last && dyn && leader) {   // published before the group's closing barrier, read by everyone after it
                if (next_ticket == last_ticket) atomicExch(io.tile_ctr, 0u);
                tile_slot[g] = next_ticket;
            }
            tc::fence_before();
            tc_group_bar(1 + g, GTHREADS);
        }
        if (rec) drow[dcol++] = clock64();
        tile = dyn ? (int64_t)tile_slot[g] : tile + (int64_t)gridDim.x * GROUPS;
    }
    if (ch.probe && tid == 0) tc::mbar_wait(bar_w, 0);   // (probe modes may skip every reader of the weights)
    tc::fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(*tmem_slot, 512);
}

static size_t tc_res_smem_bytes(const TcChain& c) { return (size_t)((c.blob_bytes + 15u) & ~15u) + 9 * 8 + 16; }

// Per-call launch options (pn_launch_opts), decoded.
struct TcOpts {
    int engine = 0;             // 0 = automatic (resident when the chain fits), 1 = always stream (mlp_tc_kernel), 2 = resident or fail
    int quad = 1;               // mlp_engine | 4 disables the coalesced quad producer
    int nslice = 1;             // mlp_engine | 8 disables N-slicing of single-layer chains
    int wide = 1;               // mlp_engine | 16 disables the 16-warp streaming CTAs
    int reserved = 0;           // reserved_sms
    int split = 1;              // mlp_passes: 1 = bf16x3 (fp32 parity), 0 = single-pass bf16
    int probe = 0;              // (mlp_engine >> 5) & 7: timing probes (results invalid)
    int engine_bits = 0;        // the raw mlp_engine flags (+256: generic quad producer even where the fast path applies; +512: no MMA issue lock)
    long long* dbg = nullptr;   // mlp_debug
    unsigned* tile_ctr = nullptr;
};

static int tc_opts_from(const pn_launch_opts* o, TcOpts* t, const char* what) {
    if (!o) return PN_OK;
    PN_REQUIRE(o->mlp_passes == 0 || o->mlp_passes == 1 || o->mlp_passes == 3, PN_ERR_BAD_ARG,
               "%s: pn_launch_opts.mlp_passes must be 3 (or 0: split bf16, fp32 parity) or 1 (plain bf16)", what);
    const int engine = o->mlp_engine;
    PN_REQUIRE(engine >= 0 && (engine & 3) <= 2 && engine < 1024, PN_ERR_BAD_ARG,
               "%s: pn_launch_opts.mlp_engine: 0 = automatic, 1 = streaming, 2 = resident; +4 = row-per-thread producers only; "
               "+8 = no N-slicing; +16 = 8-warp streaming CTAs only", what);
    PN_REQUIRE(o->reserved_sms >= 0 && o->reserved_sms < 148, PN_ERR_BAD_ARG, "%s: pn_launch_opts.reserved_sms must be in [0, 148)", what);
    PN_REQUIRE(((uintptr_t)o->tile_counter & 3) == 0, PN_ERR_ALIGNMENT, "%s: pn_launch_opts.tile_counter must be 4-byte aligned", what);
    t->split = o->mlp_passes == 1 ? 0 : 1;
    t->engine = engine & 3;
    t->quad = (engine & 4) ? 0 : 1;
    t->nslice = (engine & 8) ? 0 : 1;
    t->wide = (engine & 16) ? 0 : 1;
    t->probe = ((engine >> 5) & 7) | ((engine & 256) ? 16 : 0);   // +256 also selects the generic SA producer
    t->engine_bits = engine;
    t->reserved = o->reserved_sms;
    t->dbg = static_cast<long long*>(o->mlp_debug);
    t->tile_ctr = o->tile_counter;
    return PN_OK;
}

// Resident kernel usable?  Returns warps per group (8 or 4), or 0.
static int tc_resident_wpg(const TcChain& c) {
    if (tc_res_smem_bytes(c) > 227 * 1024) return 0;
    int a_k = 2 * c.a_lo_off;
    for (int l = 0; l < c.nlayers; ++l)
        if (c.L[l].k_pad > kTcAChunk || c.L[l].n_pad > kTcNPass) return 0;
    if (c.x_cols + a_k <= 128) return 4;
    if (c.x_cols + a_k <= 256) return 8;
    return 0;
}

static size_t tc_smem_bytes(const TcChain& c, int nstages) {
    return (size_t)nstages * c.stage_bytes + ((c.bias_floats * 4 + 15) & ~15) + (2 * kTcMaxStages + 1) * 8 + 16;
}

template <int IN>
static int tc_launch(const TcChain& ch, const void* blob, const TcIo& io, const TcOpts& to, cudaStream_t stream, const char* what) {
    const int64_t ntiles_all = io.nseg * ((io.seg_rows + 127) / 128);
    // single-layer chains on few row tiles: slice the output channels over gridDim.y so that the launch fills the GPU
    int pass_w = kTcNPass;
    if (ch.nlayers == 1 && to.nslice && io.out_mode != TC_OUT_LOGSOFTMAX && ntiles_all * ((ch.L[0].n_pad + kTcNPass - 1) / kTcNPass) < 148) {
        pass_w = 128;
        while (pass_w > 32 && ntiles_all * ((ch.L[0].n_pad + pass_w - 1) / pass_w) < 148) pass_w /= 2;
    }
    const int wpg = (to.engine == 1 || (pass_w != kTcNPass && to.engine != 2)) ? 0 : tc_resident_wpg(ch);
    PN_REQUIRE(to.engine != 2 || wpg != 0, PN_ERR_UNSUPPORTED, "%s: chain does not fit the resident kernel", what);
    if (wpg != 0) {
        const size_t rsmem = tc_res_smem_bytes(ch);
        auto launch_res = [&](auto rkern, int groups) -> int {
            cudaError_t e = cudaFuncSetAttribute(rkern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rsmem);
            if (e != cudaSuccess) {
                cudaGetLastError();
                set_error("%s: cudaFuncSetAttribute failed: %s", what, cudaGetErrorString(e));
                return (int)e;
            }
            // one persistent CTA per SM; SMs held by kernels of other streams are left out (a CTA that had to wait for
            // its SM would start its full static share of tiles late and stretch the whole launch)
            const int64_t want = (ntiles_all + groups - 1) / groups;
            const int64_t sms = 148 - to.reserved > 1 ? 148 - to.reserved : 1;
            const unsigned grid = (unsigned)(want < sms ? want : sms);
            TcIo io2 = io;
            io2.dbg = to.dbg;
            io2.tile_ctr = to.tile_ctr;
            TcChain chr = ch;
            chr.split = to.split;
            chr.probe = (to.engine_bits & 512) ? 8 : to.probe;
            e = launch_kernel(rkern, dim3(grid), dim3(kResThreads), rsmem, stream, chr, static_cast<const unsigned char*>(blob), io2);
            if (e != cudaSuccess) {
                cudaGetLastError();
                set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
                return (int)e;
            }
            return PN_OK;
        };
        return wpg == 8 ? launch_res(mlp_tc_res_kernel<IN, 8>, 2) : launch_res(mlp_tc_res_kernel<IN, 4>, 4);
    }
    // ring depth: what fits in ~110 KB (two CTAs can share an SM), at least 2, at most kTcMaxStages
    TcChain chs = ch;
    chs.pass_w = pass_w;
    chs.split = to.split;
    if (pass_w != kTcNPass) {   // re-plan the per-CTA resources for the narrower pass
        const TcLayer& L0 = ch.L[0];
        const int xw = L0.n_pad < pass_w ? L0.n_pad : pass_w;
        const int a_k = 2 * ch.a_lo_off;
        chs.x_cols = xw;
        chs.stage_bytes = xw * (L0.k_pad < kTcKSub ? L0.k_pad : kTcKSub) * 4;
        int p2 = 32;
        while (p2 < xw + a_k) p2 <<= 1;
        chs.tmem_cols = p2;
    }
    {
        const int by_tmem = 512 / chs.tmem_cols;
        (void)by_tmem;
        const size_t budget = 110 * 1024;   // deeper rings bought nothing (the MMAs, not the copies, pace a chunk); a modest
                                            // footprint lets background kernels of other streams share the SM
        const size_t fixed = tc_smem_bytes(chs, 0);
        int ns = (int)((budget - fixed) / (size_t)chs.stage_bytes);
        ns = ns < 2 ? 2 : (ns > kTcMaxStages ? kTcMaxStages : ns);
        chs.nstages = ns;
    }
    const size_t smem = tc_smem_bytes(chs, chs.nstages);
    PN_REQUIRE(smem <= 227 * 1024, PN_ERR_UNSUPPORTED, "%s: chain needs %zu bytes of shared memory", what, smem);
    // (only the FP producer / epilogues gained from 16 warps; the SA levels did not, and their 8-warp CTAs fit beside the
    // background 3-NN search that runs at the same time)
    const bool wide = to.wide && IN == TC_IN_FP && (int64_t)ntiles_all * (pass_w != kTcNPass ? (ch.L[0].n_pad + pass_w - 1) / pass_w : 1) <= 148;
    auto kern = wide ? mlp_tc_kernel<IN, 512> : mlp_tc_kernel<IN, 256>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("%s: cudaFuncSetAttribute failed: %s", what, cudaGetErrorString(e));
        return (int)e;
    }
    const int64_t ntiles = io.nseg * ((io.seg_rows + 127) / 128);
    // co-resident CTAs per SM: limited by TMEM columns (512) and shared memory
    int per_sm = 512 / chs.tmem_cols;
    const int by_smem = (int)((227 * 1024) / (smem + 1024));
    per_sm = per_sm < by_smem ? per_sm : by_smem;
    per_sm = per_sm < 1 ? 1 : (per_sm > 2 ? 2 : per_sm);   // __launch_bounds__(256, 2): registers allow two CTAs per SM
    const int64_t cap = 148LL * per_sm;
    const unsigned ny = (unsigned)((ch.L[ch.nlayers - 1].n_pad + pass_w - 1) / pass_w);
    const dim3 grid((unsigned)(ntiles < cap ? ntiles : cap), pass_w != kTcNPass ? ny : 1u);
    TcIo io2 = io;
    io2.dbg = to.dbg;
    e = launch_kernel(kern, grid, dim3(wide ? 512 : 256), smem, stream, chs, static_cast<const unsigned char*>(blob), io2);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
        return (int)e;
    }
    return PN_OK;
}

}  // namespace pn

// ------------------------------------------------------------------------------------------------ C ABI
PN_EXPORT int pn_mlp_resident_groups(const pn_mlp_desc* desc) {
    pn::TcChain ch;
    const char* why;
    if (!pn::plan_chain(desc, &ch, &why)) return 0;
    const int wpg = pn::tc_resident_wpg(ch);
    return wpg ? 16 / wpg : 0;
}

PN_EXPORT size_t pn_mlp_blob_bytes(const pn_mlp_desc* desc) {
    pn::TcChain ch;
    const char* why;
    if (!pn::plan_chain(desc, &ch, &why)) {
        pn::set_error("pn_mlp_blob_bytes: %s", why);
        return 0;
    }
    return ch.blob_bytes;
}

static int tc_pack(const pn_mlp_desc* desc, const float* const* w, const float* const* bias, const int* transposed, void* blob,
                   pn_stream_t stream);

PN_EXPORT int pn_mlp_pack_bf16x3(const pn_mlp_desc* desc, const float* const* w, const float* const* bias, void* blob,
                                 pn_stream_t stream) {
    return tc_pack(desc, w, bias, nullptr, blob, stream);
}

PN_EXPORT int pn_mlp_pack_t_bf16x3(const pn_mlp_desc* desc, const float* const* w, const float* const* bias,
                                   const int* transposed, void* blob, pn_stream_t stream) {
    return tc_pack(desc, w, bias, transposed, blob, stream);
}

static int tc_pack(const pn_mlp_desc* desc, const float* const* w, const float* const* bias, const int* transposed, void* blob,
                   pn_stream_t stream) {
    using namespace pn;
    TcChain ch;
    const char* why;
    PN_REQUIRE(plan_chain(desc, &ch, &why), PN_ERR_UNSUPPORTED, "pn_mlp_pack_bf16x3: %s", why);
    PN_REQUIRE(w && blob, PN_ERR_BAD_ARG, "pn_mlp_pack_bf16x3: null pointer");
    PN_REQUIRE(((uintptr_t)blob & 127) == 0, PN_ERR_ALIGNMENT, "pn_mlp_pack_bf16x3: blob must be 128-byte aligned");
    for (int l = 0; l < ch.nlayers; ++l) {
        const TcLayer& L = ch.L[l];
        PN_REQUIRE(w[l], PN_ERR_BAD_ARG, "pn_mlp_pack_bf16x3: weight pointer %d is null", l);
        unsigned char* img = static_cast<unsigned char*>(blob) + L.w_off;
        float* bo = reinterpret_cast<float*>(static_cast<unsigned char*>(blob) + ch.bias_off) + L.b_off;
        const int total = L.n_pad * L.k_pad;
        const bool tr = transposed && transposed[l];
        tc_pack_layer_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w[l], bias ? bias[l] : nullptr, L.k_real,
                                                                                    L.k_pad, L.n_real, L.n_pad, tr ? 1 : L.k_real,
                                                                                    tr ? L.n_real : 1, img, bo);
    }
    return finish_launch("pn_mlp_pack_bf16x3");
}

static int tc_common_checks(const pn_mlp_desc* desc, const void* blob, pn::TcChain* ch, int out_mode, const char* what) {
    using namespace pn;
    const char* why;
    PN_REQUIRE(plan_chain(desc, ch, &why), PN_ERR_UNSUPPORTED, "%s: %s", what, why);
    PN_REQUIRE(blob && ((uintptr_t)blob & 127) == 0, PN_ERR_ALIGNMENT, "%s: blob must be a 128-byte aligned device pointer", what);
    PN_REQUIRE(out_mode >= 0 && out_mode <= 2, PN_ERR_BAD_ARG, "%s: out_mode must be 0 (rows), 1 (max) or 2 (log_softmax)", what);
    const TcLayer& last = ch->L[ch->nlayers - 1];
    PN_REQUIRE(out_mode != TC_OUT_LOGSOFTMAX || last.n_real <= 64, PN_ERR_UNSUPPORTED, "%s: log_softmax head is limited to 64 classes", what);
    return PN_OK;
}

PN_EXPORT int pn_mlp_rows_bf16x3(const pn_mlp_desc* desc, const void* blob, const float* x, int64_t ldx, int64_t rows,
                                 int out_mode, float* y, int64_t ldy, const pn_launch_opts* opts, pn_stream_t stream) {
    using namespace pn;
    TcChain ch;
    int rc = tc_common_checks(desc, blob, &ch, out_mode, "pn_mlp_rows_bf16x3");
    if (rc) return rc;
    TcOpts to;
    if ((rc = tc_opts_from(opts, &to, "pn_mlp_rows_bf16x3"))) return rc;
    PN_REQUIRE(x && y && rows > 0 && ldx >= desc->cin[0], PN_ERR_BAD_ARG, "pn_mlp_rows_bf16x3: bad arguments");
    PN_REQUIRE(out_mode != TC_OUT_MAX || rows % 32 == 0, PN_ERR_UNSUPPORTED, "pn_mlp_rows_bf16x3: max-pool needs rows %% 32 == 0");
    TcIo io = {};
    io.nseg = 1;
    io.seg_rows = rows;
    io.x = x;
    io.ldx = ldx;
    io.out_mode = out_mode;
    io.y = y;
    io.ldy = ldy;
    io.group = 32;
    return tc_launch<TC_IN_ROWS>(ch, blob, io, to, (cudaStream_t)stream, "pn_mlp_rows_bf16x3");
}

PN_EXPORT int pn_sa_mlp_max_bf16x3(const pn_mlp_desc* desc, const void* blob, const float* xyz, int64_t xB, int64_t xN,
                                   int64_t xC, const float* feat, int64_t fB, int64_t fN, int64_t fC, int D,
                                   const float* new_xyz, int64_t qB, int64_t qN, int64_t qC, const int64_t* idx, int B, int N,
                                   int S, int K, int msg_order, float* out, int64_t ldo, const pn_launch_opts* opts,
                                   pn_stream_t stream) {
    return pn_sa_mlp_bf16x3(desc, blob, xyz, xB, xN, xC, feat, fB, fN, fC, D, new_xyz, qB, qN, qC, idx, B, N, S, K, msg_order,
                            PN_MLP_OUT_MAX32, out, ldo, opts, stream);
}

PN_EXPORT int pn_sa_mlp_bf16x3(const pn_mlp_desc* desc, const void* blob, const float* xyz, int64_t xB, int64_t xN,
                               int64_t xC, const float* feat, int64_t fB, int64_t fN, int64_t fC, int D,
                               const float* new_xyz, int64_t qB, int64_t qN, int64_t qC, const int64_t* idx, int B, int N,
                               int S, int K, int msg_order, int out_mode, float* out, int64_t ldo, const pn_launch_opts* opts,
                               pn_stream_t stream) {
    using namespace pn;
    TcChain ch;
    int rc = tc_common_checks(desc, blob, &ch, out_mode, "pn_sa_mlp_max_bf16x3");
    if (rc) return rc;
    TcOpts to;
    if ((rc = tc_opts_from(opts, &to, "pn_sa_mlp_bf16x3"))) return rc;
    PN_REQUIRE(out_mode == TC_OUT_MAX || out_mode == TC_OUT_ROWS, PN_ERR_BAD_ARG,
               "pn_sa_mlp_bf16x3: out_mode must be 0 (rows) or 1 (max over nsample)");
    PN_REQUIRE(xyz && new_xyz && idx && out, PN_ERR_BAD_ARG, "pn_sa_mlp_max_bf16x3: null pointer");
    PN_REQUIRE((feat != nullptr) == (D > 0) && desc->cin[0] == 3 + D, PN_ERR_BAD_ARG,
               "pn_sa_mlp_max_bf16x3: first layer expects %d channels, grouping provides 3 + %d", desc->cin[0], D);
    PN_REQUIRE(K == 16 || K % 32 == 0 || out_mode == TC_OUT_ROWS, PN_ERR_UNSUPPORTED,
               "pn_sa_mlp_bf16x3: nsample must be 16 or a multiple of 32 for the pooled output (got %d)", K);
    PN_REQUIRE(B > 0 && N > 0 && S > 0 && ldo >= desc->cout[desc->nlayers - 1], PN_ERR_BAD_ARG, "pn_sa_mlp_max_bf16x3: bad sizes");
    TcIo io = {};
    io.nseg = 1;
    io.seg_rows = (int64_t)B * S * K;
    io.xyz = xyz; io.xB = xB; io.xN = xN; io.xC = xC;
    io.feat = feat; io.fB = fB; io.fN = fN; io.fC = fC; io.D = D;
    io.qxyz = new_xyz; io.qB = qB; io.qN = qN; io.qC = qC;
    io.idx = idx; io.N = N; io.S = S; io.K = K; io.msg_order = msg_order;
    io.out_mode = out_mode;
    io.y = out;
    io.ldy = ldo;
    io.group = K == 16 ? 16 : 32;   // pooled output: one row per 16 / 32 grouped rows (K > 32: the caller reduces the K/32 partial rows)
    return tc_launch<TC_IN_SA>(ch, blob, io, to, (cudaStream_t)stream, "pn_sa_mlp_max_bf16x3");
}

PN_EXPORT int pn_fp_mlp_bf16x3(const pn_mlp_desc* desc, const void* blob, const float* points1, int64_t p1B, int64_t p1N,
                               int64_t p1C, int D1, const float* points2, int64_t p2B, int64_t p2N, int64_t p2C, int D2,
                               int S, const int64_t* idx, const float* weight, int relu_in, const int32_t* order,
                               int64_t order_es, int64_t order_bs, const float* residual, int64_t ldr, int B, int N,
                               int out_mode, float* out, int64_t ldo, const pn_launch_opts* opts, pn_stream_t stream) {
    using namespace pn;
    TcChain ch;
    int rc = tc_common_checks(desc, blob, &ch, out_mode, "pn_fp_mlp_bf16x3");
    if (rc) return rc;
    TcOpts to;
    if ((rc = tc_opts_from(opts, &to, "pn_fp_mlp_bf16x3"))) return rc;
    PN_REQUIRE(points2 && idx && weight && out, PN_ERR_BAD_ARG, "pn_fp_mlp_bf16x3: null pointer");
    PN_REQUIRE((points1 != nullptr) == (D1 > 0) && desc->cin[0] == D1 + D2, PN_ERR_BAD_ARG,
               "pn_fp_mlp_bf16x3: first layer expects %d channels, inputs provide %d + %d", desc->cin[0], D1, D2);
    PN_REQUIRE(out_mode != TC_OUT_MAX, PN_ERR_BAD_ARG, "pn_fp_mlp_bf16x3: out_mode must be 0 (rows) or 2 (log_softmax)");
    PN_REQUIRE(!relu_in || D1 == 0, PN_ERR_BAD_ARG, "pn_fp_mlp_bf16x3: relu_in needs points1 == NULL");
    PN_REQUIRE(residual == nullptr || (desc->nlayers >= 2 && !relu_in && ((uintptr_t)residual & 15) == 0 && (ldr % 4) == 0 &&
                                       ldr >= ((desc->cout[0] + 31) / 32) * 32),
               PN_ERR_BAD_ARG,
               "pn_fp_mlp_bf16x3: residual needs a chain of >= 2 layers, 16-byte aligned rows and ldr >= cout[0] rounded up to 32");
    PN_REQUIRE(B > 0 && N > 0 && S > 0 && ldo >= desc->cout[desc->nlayers - 1], PN_ERR_BAD_ARG, "pn_fp_mlp_bf16x3: bad sizes");
    TcIo io = {};
    io.nseg = B;
    io.seg_rows = N;
    io.p1 = points1; io.p1B = p1B; io.p1N = p1N; io.p1C = p1C; io.D1 = D1;
    io.p2 = points2; io.p2B = p2B; io.p2N = p2N; io.p2C = p2C; io.D2 = D2; io.S2 = S;
    io.idx3 = idx; io.w3 = weight;
    io.relu_in = relu_in;
    io.order = order; io.order_es = order_es; io.order_bs = order_bs;
    io.res = residual; io.ldr = ldr;
    {
        auto al16 = [](const void* p) { return ((uintptr_t)p & 15) == 0; };
        bool ok = p2C == 1 && (p2N % 4) == 0 && (p2B % 4) == 0 && (D2 % 4) == 0 && al16(points2);
        if (D1 > 0) ok = ok && p1C == 1 && (p1N % 4) == 0 && (p1B % 4) == 0 && (D1 % 4) == 0 && al16(points1);
        io.quad_fp = (ok && to.quad) ? 1 : 0;
        // 2 = the branch-free fast path: no skip input, no processing order, every 16-channel group is full
        if (io.quad_fp && D1 == 0 && order == nullptr && (D2 % 16) == 0 && desc->cin[0] == D2 && !(to.engine_bits & 256)) io.quad_fp = 2;
    }
    io.out_mode = out_mode;
    io.y = out;
    io.ldy = ldo;
    io.group = 32;
    return tc_launch<TC_IN_FP>(ch, blob, io, to, (cudaStream_t)stream, "pn_fp_mlp_bf16x3");
}
