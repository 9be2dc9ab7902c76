// gemm_tc.cu -- the training step's layer GEMM on the tensor cores with BatchNorm fused on both sides
// (SURVEY.md section 8 row f-1; reference: F.relu(bn(conv(x))) of model/pointnet_util.py:195-197, :310-312 and
// pointnet2.py:172 in train() mode, and the input-gradient half of their autograd backward).
//
//     y[r, n] = sum_k f(x[r, k]) * W[n, k] + bias[n]          f(v) = relu(v * in_scale[k] + in_shift[k])   (optional)
//     col_sum[n] += sum_r y[r, n],  col_sumsq[n] += sum_r y[r, n]^2                                         (optional, fp64)
//
// In train() mode BatchNorm needs the statistics of a layer's WHOLE output before the next layer can start, so the
// forward cannot be one chain; unfused it costs three passes per layer (GEMM writes y, a reduction re-reads y, the
// normalise+ReLU pass re-reads y and writes z: 20 bytes per element).  Here the statistics are accumulated in the GEMM's
// epilogue and the normalise+ReLU of the PREVIOUS layer is applied while this GEMM loads its operand, so a layer costs one
// read and one write (8 bytes per element) and the activated tensor z never exists; the backward recomputes what it needs
// from y (pn_grad_weight_bf16x3 applies the same f to its x operand).
//
// Structure: persistent CTAs (up to two per SM).  The weights (<= 128 KB as bf16 hi + lo) are converted once per call by a
// small pre-pass into the UMMA K-major layout, fetched by every CTA with bulk copies (cp.async.bulk + mbarrier) and stay
// resident in shared memory; the x operand streams through a 2-stage ring of 128-row x
// 32-column chunks that the four PRODUCER warps fill (thread = row: fp32 -> f() -> bf16 hi/lo, 16-byte stores straight into
// the K-major layout, register double buffer across chunks and tiles); an elected lane of warp 0 issues hi*hi + hi*lo +
// lo*hi per 16 columns (tcgen05.mma kind::f16, both operands from shared memory) into one of TWO fp32 accumulators of
// 128 x cout in TMEM; the four EPILOGUE warps read a finished accumulator back (thread = row), add the bias, store y and
// reduce the column sums with a shuffle butterfly in fp64 -- while the producers and the tensor core work on the next tile.
// W can be given transposed (w[k, n]): the input-gradient GEMM dx = dy W of the backward pass reads W that way.
#include <stdlib.h>

#include "common.cuh"
#include "tcgen05.cuh"

namespace pn {
namespace gemm {

constexpr int TM = 128, KC = 32, THREADS = 256;
constexpr int NS_MAX = 4, NA_MAX = 4;          // operand ring stages / TMEM accumulators: chosen per layer by the host (Args::ns, ::na)
constexpr int A_IMG = TM * KC * 2;            // one bf16 image of a 128 x 32 chunk: 8 KB
constexpr int A_STAGE = 2 * A_IMG;            // hi + lo
constexpr int W_MAX_BYTES = 128 * 1024;       // resident weights (hi + lo)
constexpr int PF = 6;                         // L2 prefetch distance of the operand stream, in 32-column chunks

struct Args {
    const float* x; int64_t ldx; int64_t rows; int cin;
    const float* in_scale; const float* in_shift; int in_relu;
    const float* w; int w_transposed; const float* bias; int cout;
    float* y; int64_t ldy;
    double* col_sum; double* col_sumsq;
    int k_pad, n_pad, x_vec, debug, ns, na;
    // backward statistics in the epilogue (all NULL for the forward): the layer BELOW's pre-normalisation output and constants
    const float* py; int64_t ldpy; const float* p_scale; const float* p_shift; const float* p_mean; const float* p_invstd;
    int p_eval;      // the layer below normalises with FIXED statistics: store its dy = scale*g instead of dz (pn_train_gemm_bneval_bf16x3)
    const unsigned char* w_packed;   // bf16 hi/lo image of the weights in the kernel's shared-memory layout (train_pack_kernel)
};

// Weights fp32 -> bf16 hi/lo in the layout the GEMM keeps in shared memory: per 32-wide K chunk the hi image
// [n_pad x 32] then the lo image, K-major core matrices.  Done ONCE per GEMM into a scratch buffer; every CTA of the GEMM
// then fetches the image with bulk copies.  (Converting inside the GEMM cost ~18 us per CTA for a 128 x 128 layer: 296 CTAs
// gathering the same 64 KB with scattered 4-byte loads.)
__device__ __forceinline__ void pack_weights(const float* __restrict__ w, int w_transposed, int cin, int cout, int k_pad, int n_pad,
                                             unsigned char* __restrict__ out) {
    const int kblocks = k_pad / 8;
    const unsigned w_chunk_bytes = (unsigned)n_pad * KC * 4;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n_pad * kblocks; e += gridDim.x * blockDim.x) {
        // consecutive threads read consecutive memory: along k for a row-major [cout, cin] weight, along n for its transpose
        const int n = w_transposed ? e % n_pad : e / kblocks, kb = w_transposed ? e / n_pad : e % kblocks;
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = kb * 8 + j;
            float t = 0.0f;
            if (n < cout && k < cin) t = w_transposed ? __ldg(w + (int64_t)k * cout + n) : __ldg(w + (int64_t)n * cin + k);
            v[j] = t;
        }
        const int c = kb / (KC / 8), kbi = kb % (KC / 8);
        unsigned char* img = out + (size_t)c * w_chunk_bytes;
        const unsigned off = (unsigned)(n >> 3) * (KC / 8) * 128u + (unsigned)kbi * 128u + (unsigned)(n & 7) * 16u;
        tc::store_split8(img, img + (size_t)n_pad * KC * 2, off, v);
    }
}

__global__ void train_pack_kernel(const float* __restrict__ w, int w_transposed, int cin, int cout, int k_pad, int n_pad,
                                  unsigned char* __restrict__ out) {
    pack_weights(w, w_transposed, cin, cout, k_pad, n_pad, out);
}

// The same for MANY layers in one launch (blockIdx.y = item): all weights of a network, both orientations, packed once per
// training iteration instead of once per GEMM call.
__global__ void train_pack_many_kernel(const pn_train_pack_item* __restrict__ items) {
    const pn_train_pack_item it = items[blockIdx.y];
    pack_weights(it.w, it.transposed, it.cin, it.cout, (it.cin + KC - 1) / KC * KC, (it.cout + 31) / 32 * 32,
                 static_cast<unsigned char*>(it.out));
}

// The BatchNorm-backward terms of the layer BELOW for the 32 columns col0.. of one row: this GEMM's output v is dz of that
// layer (gradient w.r.t. its activated output); with its pre-normalisation output yp: g = dz * [yp*scale+shift > 0],
// xhat = (yp - mean) * invstd; f1 = g, f2 = g*xhat (the two sums its backward needs).  store_dy: v becomes scale*g.
__device__ __forceinline__ void bwd_terms(const Args& a, const float* pc, int64_t row, bool row_ok, int col0, float (&v)[32],
                                          float (&f1)[32], float (&f2)[32], bool store_dy) {
    const float* __restrict__ ypr = a.py + row * a.ldpy + col0;
    const bool vec = col0 + 32 <= a.cout && ((a.ldpy & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.py) & 15) == 0);
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
        float yp[4] = {0.f, 0.f, 0.f, 0.f};
        if (row_ok) {
            if (vec) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(ypr + j));
                yp[0] = t.x; yp[1] = t.y; yp[2] = t.z; yp[3] = t.w;
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (col0 + j + i < a.cout) yp[i] = __ldg(ypr + j + i);
            }
        }
        const float4 sc = *reinterpret_cast<const float4*>(pc + col0 + j);
        const float4 sh = *reinterpret_cast<const float4*>(pc + a.n_pad + col0 + j);
        const float4 mu = *reinterpret_cast<const float4*>(pc + 2 * a.n_pad + col0 + j);
        const float4 is = *reinterpret_cast<const float4*>(pc + 3 * a.n_pad + col0 + j);
        const float scv[4] = {sc.x, sc.y, sc.z, sc.w}, shv[4] = {sh.x, sh.y, sh.z, sh.w};
        const float muv[4] = {mu.x, mu.y, mu.z, mu.w}, isv[4] = {is.x, is.y, is.z, is.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float g = (row_ok && fmaf(yp[i], scv[i], shv[i]) > 0.0f) ? v[j + i] : 0.0f;
            f1[j + i] = g;
            f2[j + i] = g * ((yp[i] - muv[i]) * isv[i]);
            if (store_dy) v[j + i] = scv[i] * g;
        }
    }
}

// Column sums of f1 / f2 over a warp's 32 rows added to the CTA's shared-memory sums s1 / s2 (32 columns each): the
// butterfly's first three steps (16 + 8 + 4 columns exchanged: afterwards a lane holds 4 columns summed over 8 rows) in fp32,
// the last two and everything beyond in fp64.  Four warps meet per column; one global atomic per column and CTA at the end.
__device__ __forceinline__ void reduce_into(float (&f1)[32], float (&f2)[32], int lane, double* s1, double* s2) {
    const auto add = [](auto x, auto y) { return x + y; };
    tc::col_butterfly<16, 4>(f1, lane, add);
    tc::col_butterfly<16, 4>(f2, lane, add);
    double d1[32], d2[32];
#pragma unroll
    for (int j = 0; j < 4; ++j) { d1[j] = (double)f1[j]; d2[j] = (double)f2[j]; }
    tc::col_butterfly<2, 1>(d1, lane, add);
    tc::col_butterfly<2, 1>(d2, lane, add);
    atomicAdd(&s1[lane], d1[0]);
    atomicAdd(&s2[lane], d2[0]);
}

// dgamma += s2, dbeta += s1 (either may be NULL) after pn_train_gemm_bneval_bf16x3.
__global__ void bneval_finalize_kernel(const double* __restrict__ s1, const double* __restrict__ s2, int C, float* __restrict__ dgamma,
                                       float* __restrict__ dbeta) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    if (dgamma) dgamma[c] += (float)s2[c];
    if (dbeta) dbeta[c] += (float)s1[c];
}

// EVAL: the eval-mode epilogue (Args::p_eval), a separate instantiation so that the training GEMM's registers are not shared
template <bool EVAL>
__global__ void __launch_bounds__(THREADS, 2)
train_gemm_kernel(const Args a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int kch = a.k_pad / KC;                               // K chunks
    const int NS = a.ns, NA = a.na;
    const unsigned w_chunk_bytes = (unsigned)a.n_pad * KC * 4;  // hi + lo images of one K chunk of the weights
    unsigned char* w_smem = smem;                               // [kch][hi: n_pad x 32 | lo: n_pad x 32]
    unsigned char* a_smem = smem + (size_t)kch * w_chunk_bytes; // ring of NS stages
    // barriers: full[4] (128 producer arrivals), empty[4] (MMA commit), acc_full[4] (MMA commit), acc_empty[4] (128 epilogue arrivals), weights
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(a_smem + NS * A_STAGE);
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 4 * NS_MAX + 1);
    float* tf = reinterpret_cast<float*>(bars + 32);                                           // [2][k_pad]: in_scale | in_shift (16-byte aligned)
    double* cta_sum = reinterpret_cast<double*>(tf + 2 * a.k_pad);                             // [2][n_pad]: this CTA's column sums over all its tiles
    float* bias_s = reinterpret_cast<float*>(cta_sum + 2 * a.n_pad);                           // [n_pad], zero beyond cout
    float* pc = bias_s + a.n_pad;                                                               // [4][n_pad]: scale, shift, mean, invstd of the layer below (forward: [0] = statistics pivots)
    float* stg_all = pc + 4 * a.n_pad;                                                          // [4 epilogue warps][32 rows][20]: output staging
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const unsigned bar_full = tc::smem_u32(bars), bar_empty = tc::smem_u32(bars + NS_MAX), bar_accf = tc::smem_u32(bars + 2 * NS_MAX),
                   bar_acce = tc::smem_u32(bars + 3 * NS_MAX), bar_w = tc::smem_u32(bars + 4 * NS_MAX);

    unsigned tmem_cols = 32;
    while ((int)tmem_cols < NA * a.n_pad) tmem_cols <<= 1;      // NA accumulators: the MMAs of the next tiles overlap the epilogue of tile i
    if (tid == 0) {
        for (int s = 0; s < NS; ++s) {
            tc::mbar_init(bar_full + 8 * s, THREADS / 2);
            tc::mbar_init(bar_empty + 8 * s, 1);
        }
        for (int b = 0; b < NA; ++b) {
            tc::mbar_init(bar_accf + 8 * b, 1);
            tc::mbar_init(bar_acce + 8 * b, THREADS / 2);
        }
        tc::mbar_init(bar_w, 1);
        tc::mbar_init_fence();
        // the packed weights: bulk copies straight into their resident place, completion counted in bytes on bar_w
        tc::bulk_load_pieces(tc::smem_u32(w_smem), a.w_packed, (unsigned)kch * w_chunk_bytes, bar_w);
    }
    if (warp == 0) tc::tmem_alloc(tmem_slot, tmem_cols);
    const int64_t tiles = (a.rows + TM - 1) / TM;
    const int64_t my_tiles = blockIdx.x < tiles ? (tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    // the producers' first chunk is requested BEFORE the weight conversion, which then hides its latency
    float va[KC];
    auto load_chunk = [&](int64_t gc) {
        const int64_t it = gc / kch;
        const int c = (int)(gc - it * kch);
        const int64_t row = (blockIdx.x + it * gridDim.x) * TM + (tid & 127);
        const bool row_ok = row < a.rows;
        const float* __restrict__ xr = a.x + row * a.ldx + c * KC;
        if (a.x_vec && (c + 1) * KC <= a.cin) {
#pragma unroll
            for (int i = 0; i < KC / 4; ++i) {
                const float4 t = row_ok ? __ldg(reinterpret_cast<const float4*>(xr) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                va[4 * i] = t.x; va[4 * i + 1] = t.y; va[4 * i + 2] = t.z; va[4 * i + 3] = t.w;
            }
        } else {
#pragma unroll
            for (int j = 0; j < KC; ++j) va[j] = (row_ok && c * KC + j < a.cin) ? __ldg(xr + j) : 0.0f;
        }
    };
    if (warp < 4 && my_tiles > 0) {
        load_chunk(0);
        for (int g2 = 1; g2 < PF && g2 < my_tiles * kch; ++g2) {
            const int64_t it2 = g2 / kch;
            const int c2 = (int)(g2 - it2 * kch);
            const int64_t row2 = (blockIdx.x + it2 * gridDim.x) * TM + (tid & 127);
            if (row2 < a.rows && c2 * KC < a.cin) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.x + row2 * a.ldx + c2 * KC));
        }
    }
    if (a.col_sum) {
        for (int n = tid; n < 2 * a.n_pad; n += THREADS) cta_sum[n] = 0.0;
        if (!a.py)
            for (int n = tid; n < a.n_pad; n += THREADS) pc[n] = 0.0f;     // the pivots, set by the first tile's epilogue
    }
    for (int n = tid; n < a.n_pad; n += THREADS) bias_s[n] = (a.bias && n < a.cout) ? __ldg(a.bias + n) : 0.0f;
    if (a.py)
        for (int n = tid; n < a.n_pad; n += THREADS) {
            const bool ok = n < a.cout;
            pc[n] = ok ? __ldg(a.p_scale + n) : 0.0f;
            pc[a.n_pad + n] = ok ? __ldg(a.p_shift + n) : 0.0f;
            pc[2 * a.n_pad + n] = ok ? __ldg(a.p_mean + n) : 0.0f;
            pc[3 * a.n_pad + n] = ok ? __ldg(a.p_invstd + n) : 0.0f;
        }
    if (a.in_scale) {
        // the operand transform's per-channel constants: read through shared memory (a warp's lanes all want the same k)
        for (int k = tid; k < a.k_pad; k += THREADS) {
            tf[k] = k < a.cin ? __ldg(a.in_scale + k) : 0.0f;
            tf[a.k_pad + k] = k < a.cin ? __ldg(a.in_shift + k) : 0.0f;
        }
    }
    tc::fence_proxy_async();
    tc::fence_before();
    __syncthreads();
    tc::fence_after();
    const unsigned tbase = *tmem_slot;

    if (warp < 4) {
        // ================= producers (warps 0-3): thread = row of the tile; warp 0 also issues the MMAs =================
        const int64_t total_chunks = my_tiles * kch;
        const int m = tid;
        const unsigned row_off = (unsigned)(m >> 3) * (KC / 8) * 128u + (unsigned)(m & 7) * 16u;
        const unsigned idesc = tc::idesc_bf16_f32(TM, a.n_pad);
        const unsigned long long dbase = tc::sdesc_base((KC / 8) * 128u);
        for (int64_t gc = 0; gc < total_chunks; ++gc) {
            const int64_t it = gc / kch;
            const int c = (int)(gc - it * kch);
            const int s = (int)(gc % NS);
            const unsigned use = (unsigned)(gc / NS);
            float cur[KC];
#pragma unroll
            for (int j = 0; j < KC; ++j) cur[j] = va[j];
            if (gc + 1 < total_chunks) load_chunk(gc + 1);
            // The register buffer keeps only ONE chunk (16 KB per CTA) in flight, far too little to cover the HBM latency:
            // the line this thread will load PF chunks from now (its row's 128 bytes of that chunk) is requested into L2
            // ahead of time -- a prefetch holds no register.
            if (gc + PF < total_chunks) {
                const int64_t g2 = gc + PF, it2 = g2 / kch;
                const int c2 = (int)(g2 - it2 * kch);
                const int64_t row2 = (blockIdx.x + it2 * gridDim.x) * TM + m;
                if (row2 < a.rows && c2 * KC < a.cin)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(a.x + row2 * a.ldx + c2 * KC));
            }
            // f(): normalise + ReLU of the previous layer, applied to the operand on its way into shared memory
            if (a.in_scale) {
                const bool row_ok = (blockIdx.x + it * gridDim.x) * TM + m < a.rows;
                const float4* sc4 = reinterpret_cast<const float4*>(tf + c * KC);
                const float4* sh4 = reinterpret_cast<const float4*>(tf + a.k_pad + c * KC);
#pragma unroll
                for (int i = 0; i < KC / 4; ++i) {
                    const float4 sc = sc4[i], sh = sh4[i];       // padded channels: scale = shift = 0 -> 0
                    float t0 = fmaf(cur[4 * i], sc.x, sh.x), t1 = fmaf(cur[4 * i + 1], sc.y, sh.y);
                    float t2 = fmaf(cur[4 * i + 2], sc.z, sh.z), t3 = fmaf(cur[4 * i + 3], sc.w, sh.w);
                    if (a.in_relu) { t0 = fmaxf(t0, 0.0f); t1 = fmaxf(t1, 0.0f); t2 = fmaxf(t2, 0.0f); t3 = fmaxf(t3, 0.0f); }
                    cur[4 * i] = row_ok ? t0 : 0.0f; cur[4 * i + 1] = row_ok ? t1 : 0.0f;
                    cur[4 * i + 2] = row_ok ? t2 : 0.0f; cur[4 * i + 3] = row_ok ? t3 : 0.0f;
                }
            }
            if (gc >= NS) tc::mbar_wait(bar_empty + 8 * s, (use - 1) & 1);
            unsigned char* st = a_smem + s * A_STAGE;
#pragma unroll
            for (int kb = 0; kb < ((a.debug & 4) ? 0 : KC / 8); ++kb) {
                float v8[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) v8[j] = cur[kb * 8 + j];
                tc::store_split8(st, st + A_IMG, row_off + (unsigned)kb * 128u, v8);
            }
            tc::fence_proxy_async();
            tc::mbar_arrive(bar_full + 8 * s);
            if (warp == 0) {
                const int b = (int)(it % NA);
                tc::mbar_wait(bar_full + 8 * s, use & 1);
                if (gc == 0) tc::mbar_wait(bar_w, 0);                      // the weight image has landed
                if (c == 0 && it >= NA) tc::mbar_wait(bar_acce + 8 * b, (unsigned)(it / NA - 1) & 1);   // epilogue of tile it-NA has read it
                tc::fence_after();
                if (tc::elect()) {
                    const unsigned acc = tbase + (unsigned)(b * a.n_pad);
                    const unsigned a_hi = tc::smem_u32(st), a_lo = a_hi + A_IMG;
                    const unsigned b_hi = tc::smem_u32(w_smem) + (unsigned)c * w_chunk_bytes, b_lo = b_hi + (unsigned)a.n_pad * KC * 2;
#pragma unroll
                    for (int t = 0; t < ((a.debug & 1) ? 0 : KC / 16); ++t)
                        tc::mma_bf16x3(acc, tc::sdesc(dbase, a_hi + t * 256), tc::sdesc(dbase, a_lo + t * 256),
                                       tc::sdesc(dbase, b_hi + t * 256), tc::sdesc(dbase, b_lo + t * 256), idesc, (c > 0 || t > 0) ? 1u : 0u);
                    tc::commit(bar_empty + 8 * s);
                    if (c + 1 == kch) tc::commit(bar_accf + 8 * b);
                }
                __syncwarp();
            }
        }
    } else {
        // ================= epilogue (warps 4-7): thread = row (TMEM lane), all output channels =================
        const int q = warp - 4;                                  // a warp reads the TMEM lanes of its quarter
        const int nch = a.n_pad / 32;
        for (int64_t it = 0; it < my_tiles; ++it) {
            const int b = (int)(it % NA);
            tc::mbar_wait(bar_accf + 8 * b, (unsigned)(it / NA) & 1);
            tc::fence_after();
            const int64_t row = (blockIdx.x + it * gridDim.x) * TM + q * 32 + lane;
            const bool row_ok = row < a.rows;
            for (int ch = 0; ch < nch; ++ch) {
                const int col0 = ch * 32;
                unsigned r[32];
                if (!(a.debug & 16)) tc::ld32(tbase + ((unsigned)(q * 32) << 16) + (unsigned)(b * a.n_pad + col0), r);
                if (ch + 1 == nch) {                             // the accumulator has been read: the MMAs of tile it+2 may overwrite it
                    tc::fence_before();
                    tc::mbar_arrive(bar_acce + 8 * b);
                }
                float v[32];
                const float4* b4 = reinterpret_cast<const float4*>(bias_s + col0);       // (a warp's lanes all want the same n)
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 bb = b4[j >> 2];
                    v[j] = __uint_as_float(r[j]) + bb.x;
                    v[j + 1] = __uint_as_float(r[j + 1]) + bb.y;
                    v[j + 2] = __uint_as_float(r[j + 2]) + bb.z;
                    v[j + 3] = __uint_as_float(r[j + 3]) + bb.w;
                }
                if ((a.debug & 2) && v[0] != 12345.678f) continue;
                if (EVAL) {
                    // fixed statistics below: g and g*xhat as in the branch further down, their sums first, then the stored
                    // value is the layer below's dy = scale*g (no BatchNorm pass of its own)
                    float f1[32], f2[32];
                    bwd_terms(a, pc, row, row_ok, col0, v, f1, f2, true);
                    reduce_into(f1, f2, lane, cta_sum + col0, cta_sum + a.n_pad + col0);
                }
                if (!(a.debug & 64)) {
                    if (col0 + 32 <= a.cout && ((a.ldy & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.y) & 15) == 0)) {
                        // A thread owns a ROW of the accumulator, so storing straight from registers makes every store
                        // instruction touch 32 different lines with 16 bytes each (measured: 11 of 38 us for a 128 x 128
                        // layer).  The 32 x 32 block goes through a per-warp shared-memory tile in two halves of 16
                        // columns instead: 4 lanes then write the 64 contiguous bytes of a row, 8 rows per instruction.
                        float* stg = stg_all + q * (32 * 20);
                        const int64_t row0 = (blockIdx.x + it * gridDim.x) * TM + q * 32;
#pragma unroll
                        for (int hcol = 0; hcol < 2; ++hcol) {
#pragma unroll
                            for (int j = 0; j < 16; j += 4)
                                *reinterpret_cast<float4*>(stg + lane * 20 + j) =
                                    make_float4(v[hcol * 16 + j], v[hcol * 16 + j + 1], v[hcol * 16 + j + 2], v[hcol * 16 + j + 3]);
                            __syncwarp();
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const int r = (lane >> 2) + 8 * i;
                                const float4 t = *reinterpret_cast<const float4*>(stg + r * 20 + (lane & 3) * 4);
                                if (row0 + r < a.rows)
                                    *reinterpret_cast<float4*>(a.y + (row0 + r) * a.ldy + col0 + hcol * 16 + (lane & 3) * 4) = t;
                            }
                            __syncwarp();
                        }
                    } else if (row_ok) {
                        float* dst = a.y + row * a.ldy + col0;
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (col0 + j < a.cout) dst[j] = v[j];
                    }
                }
                if (!EVAL && a.col_sum && !(a.debug & 32)) {
                    // column sums over the warp's 32 rows: the butterfly's first three steps (16 + 8 + 4 columns exchanged:
                    // afterwards a lane holds 4 columns summed over 8 rows) in fp32, the last two and everything beyond in fp64
                    float f1[32], f2[32];
                    if (a.py) {
                        bwd_terms(a, pc, row, row_ok, col0, v, f1, f2, false);
                    } else {
                        // FORWARD statistics, shifted by a per-column pivot p (the CTA's first row): sum (y-p), sum (y-p)^2.
                        // Unshifted, the fp32 square would carry a rounding of |mean|^2 * 2^-24 that does not average out
                        // (a constant channel at 27.1 gets var = 7.5e-5 instead of 0), and var = E[y^2] - mean^2 keeps it.
                        float* piv = pc;                         // (pc holds the layer below's constants in the backward only)
                        if (it == 0) {
                            if (q == 0 && lane == 0)
#pragma unroll
                                for (int j = 0; j < 32; ++j) piv[col0 + j] = v[j];
                            asm volatile("bar.sync 1, 128;" ::: "memory");       // the four epilogue warps
                        }
                        const float4* p4 = reinterpret_cast<const float4*>(piv + col0);
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            const float4 pp = p4[j >> 2];
                            const float pv[4] = {pp.x, pp.y, pp.z, pp.w};
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const float d = row_ok ? v[j + i] - pv[i] : 0.0f;
                                f1[j + i] = d;
                                f2[j + i] = d * d;
                            }
                        }
                    }
                    reduce_into(f1, f2, lane, cta_sum + col0, cta_sum + a.n_pad + col0);
                }
            }
        }
    }
    tc::fence_before();
    __syncthreads();
    if (a.col_sum && my_tiles > 0) {
        // forward: the shifted sums of the CTA's rows back to plain sums, in fp64 (s2 + 2 p s1 + n p^2 loses nothing
        // that matters: var = E[y^2] - mean^2 in fp64 keeps a relative error of (mean/std)^2 * 2^-53)
        const int64_t short_rows = (blockIdx.x == (tiles - 1) % gridDim.x) ? tiles * TM - a.rows : 0;
        const double nc = (double)(my_tiles * TM - short_rows);
        for (int n = tid; n < a.cout; n += THREADS) {
            double s1 = cta_sum[n], s2 = cta_sum[a.n_pad + n];
            if (!a.py) {
                const double p = (double)pc[n];
                s2 += p * (2.0 * s1 + nc * p);
                s1 += nc * p;
            }
            atomicAdd(a.col_sum + n, s1);
            atomicAdd(a.col_sumsq + n, s2);
        }
    }
    if (warp == 0) tc::tmem_dealloc(tbase, tmem_cols);
}

static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

}  // namespace gemm
}  // namespace pn

PN_EXPORT int pn_train_gemm_supported(int cin, int cout) {
    using namespace pn::gemm;
    if (cin < 1 || cout < 1) return 0;
    const int k_pad = round_up(cin, KC), n_pad = round_up(cout, 32);
    return n_pad <= 256 && (size_t)k_pad * n_pad * 4 <= (size_t)W_MAX_BYTES;
}

PN_EXPORT int pn_train_pack_many(const pn_train_pack_item* items, int n_items, int max_cin, int max_cout, pn_stream_t stream) {
    using namespace pn;
    using namespace pn::gemm;
    PN_REQUIRE(items && n_items > 0 && n_items <= 65535 && max_cin > 0 && max_cout > 0, PN_ERR_BAD_ARG, "pn_train_pack_many: bad arguments");
    const int entries = round_up(max_cout, 32) * (round_up(max_cin, KC) / 8);
    int bx = (entries + 255) / 256;
    if (bx > 16) bx = 16;
    train_pack_many_kernel<<<dim3((unsigned)bx, (unsigned)n_items), 256, 0, (cudaStream_t)stream>>>(items);
    return finish_launch("pn_train_pack_many");
}

PN_EXPORT size_t pn_train_gemm_scratch_bytes(int cin, int cout) {
    using namespace pn::gemm;
    if (!pn_train_gemm_supported(cin, cout)) return 0;
    return (size_t)round_up(cin, KC) * round_up(cout, 32) * 4;
}

static int train_gemm_launch(const float* x, int64_t ldx, int64_t rows, int cin, const float* in_scale, const float* in_shift,
                             int in_relu, const float* w, int w_transposed, const float* bias, int cout, float* y, int64_t ldy,
                             double* col_sum, double* col_sumsq, const float* py, int64_t ldpy, const float* p_scale,
                             const float* p_shift, const float* p_mean, const float* p_invstd, void* w_scratch, pn_stream_t stream,
                             int p_eval = 0);

PN_EXPORT int pn_train_gemm_bf16x3(const float* x, int64_t ldx, int64_t rows, int cin, const float* in_scale,
                                   const float* in_shift, int in_relu, const float* w, int w_transposed, const float* bias,
                                   int cout, float* y, int64_t ldy, double* col_sum, double* col_sumsq, void* w_scratch,
                                   pn_stream_t stream) {
    return train_gemm_launch(x, ldx, rows, cin, in_scale, in_shift, in_relu, w, w_transposed, bias, cout, y, ldy, col_sum, col_sumsq,
                             nullptr, 0, nullptr, nullptr, nullptr, nullptr, w_scratch, stream);
}

PN_EXPORT int pn_train_gemm_bnbwd_bf16x3(const float* dy, int64_t lddy, int64_t rows, int cin, const float* w, int w_transposed,
                                         int cout, float* dz, int64_t lddz, const float* prev_y, int64_t ld_prev,
                                         const float* prev_scale, const float* prev_shift, const float* prev_mean,
                                         const float* prev_invstd, double* s1, double* s2, void* w_scratch, pn_stream_t stream) {
    PN_REQUIRE(prev_y && prev_scale && prev_shift && prev_mean && prev_invstd && s1 && s2, PN_ERR_BAD_ARG,
               "pn_train_gemm_bnbwd_bf16x3: null pointer");
    PN_REQUIRE(ld_prev >= cout, PN_ERR_BAD_ARG, "pn_train_gemm_bnbwd_bf16x3: ld_prev smaller than cout");
    return train_gemm_launch(dy, lddy, rows, cin, nullptr, nullptr, 0, w, w_transposed, nullptr, cout, dz, lddz, s1, s2, prev_y, ld_prev,
                             prev_scale, prev_shift, prev_mean, prev_invstd, w_scratch, stream);
}

PN_EXPORT int pn_train_gemm_bneval_bf16x3(const float* dy, int64_t lddy, int64_t rows, int cin, const float* w, int w_transposed,
                                          int cout, float* dy_prev, int64_t ld_dy_prev, const float* prev_y, int64_t ld_prev,
                                          const float* prev_scale, const float* prev_shift, const float* prev_mean,
                                          const float* prev_invstd, double* s1, double* s2, float* dgamma, float* dbeta,
                                          void* w_scratch, pn_stream_t stream) {
    PN_REQUIRE(dy_prev && prev_y && prev_scale && prev_shift && prev_mean && prev_invstd && s1 && s2, PN_ERR_BAD_ARG,
               "pn_train_gemm_bneval_bf16x3: null pointer");
    PN_REQUIRE(ld_prev >= cout, PN_ERR_BAD_ARG, "pn_train_gemm_bneval_bf16x3: ld_prev smaller than cout");
    const int rc = train_gemm_launch(dy, lddy, rows, cin, nullptr, nullptr, 0, w, w_transposed, nullptr, cout, dy_prev, ld_dy_prev, s1, s2,
                                     prev_y, ld_prev, prev_scale, prev_shift, prev_mean, prev_invstd, w_scratch, stream, 1);
    if (rc != 0 || !(dgamma || dbeta)) return rc;
    pn::gemm::bneval_finalize_kernel<<<(unsigned)pn::ceil_div(cout, 128), 128, 0, (cudaStream_t)stream>>>(s1, s2, cout, dgamma, dbeta);
    return pn::finish_launch("pn_train_gemm_bneval_bf16x3");
}

static int train_gemm_launch(const float* x, int64_t ldx, int64_t rows, int cin, const float* in_scale, const float* in_shift,
                             int in_relu, const float* w, int w_transposed, const float* bias, int cout, float* y, int64_t ldy,
                             double* col_sum, double* col_sumsq, const float* py, int64_t ldpy, const float* p_scale,
                             const float* p_shift, const float* p_mean, const float* p_invstd, void* w_scratch, pn_stream_t stream,
                             int p_eval) {
    using namespace pn;
    using namespace pn::gemm;
    PN_REQUIRE(x && y && w_scratch, PN_ERR_BAD_ARG, "pn_train_gemm_bf16x3: null pointer");
    PN_REQUIRE(((uintptr_t)w_scratch & 127) == 0, PN_ERR_ALIGNMENT, "pn_train_gemm_bf16x3: w_scratch must be 128-byte aligned");
    PN_REQUIRE(rows > 0 && cin > 0 && cout > 0 && ldx >= cin && ldy >= cout, PN_ERR_BAD_ARG, "pn_train_gemm_bf16x3: bad shape");
    PN_REQUIRE((in_scale == nullptr) == (in_shift == nullptr) && (col_sum == nullptr) == (col_sumsq == nullptr), PN_ERR_BAD_ARG,
               "pn_train_gemm_bf16x3: in_scale/in_shift and col_sum/col_sumsq come in pairs");
    PN_REQUIRE(pn_train_gemm_supported(cin, cout), PN_ERR_UNSUPPORTED,
               "pn_train_gemm_bf16x3: layer %d -> %d does not fit the resident-weight kernel (cout <= 256, padded cin*cout*4 <= 128 KB)", cin, cout);
    Args a;
    a.x = x; a.ldx = ldx; a.rows = rows; a.cin = cin;
    a.in_scale = in_scale; a.in_shift = in_shift; a.in_relu = in_relu;
    a.w = w; a.w_transposed = w_transposed; a.bias = bias; a.cout = cout;
    a.y = y; a.ldy = ldy; a.col_sum = col_sum; a.col_sumsq = col_sumsq;
    a.p_eval = p_eval;
    a.py = py; a.ldpy = ldpy; a.p_scale = p_scale; a.p_shift = p_shift; a.p_mean = p_mean; a.p_invstd = p_invstd;
    a.k_pad = round_up(cin, KC);
    a.n_pad = round_up(cout, 32);
    a.x_vec = ((uintptr_t)x % 16 == 0) && (ldx % 4 == 0);
    {
        static int dbg = -1;
        if (dbg < 0) {
            const char* e = getenv("PN12_GEMM_DEBUG");     // profiling only: 1 = no MMAs, 2 = no epilogue work, 4 = no operand stores, 8 = (unused), 16 = no TMEM loads, 32 = no statistics, 64 = no y stores
            dbg = e ? atoi(e) : 0;
        }
        a.debug = dbg;
    }
    // Ring depth and accumulator count: a row tile is handed producer -> tensor core -> epilogue through mbarriers, ~3 us per
    // tile of latency, so narrow layers (one or two K chunks per tile) need several tiles in flight.  Layers whose weights
    // leave room get 4 stages; two CTAs share the SM's 512 TMEM columns, so each may hold 256 / n_pad accumulators.
    const size_t w_bytes = (size_t)a.k_pad * a.n_pad * 4;
    const size_t fixed = 256 /* barriers + TMEM slot */ + (size_t)2 * a.n_pad * sizeof(double) + (size_t)2 * a.k_pad * sizeof(float) +
                         (size_t)5 * a.n_pad * sizeof(float) + (size_t)4 * 32 * 20 * sizeof(float) + 64;
    a.ns = (w_bytes + 4 * A_STAGE + fixed <= 112 * 1024) ? 4 : 2;
    const size_t smem = w_bytes + (size_t)a.ns * A_STAGE + fixed;
    const int per_sm = (smem <= 112 * 1024 && a.n_pad <= 128) ? 2 : 1;      // two CTAs share the SM's 512 TMEM columns
    a.na = (per_sm == 2 ? 256 : 512) / a.n_pad;
    if (a.na > NA_MAX) a.na = NA_MAX;
    static int sms = 0;
    static size_t smem_set = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    if (smem > smem_set) {
        cudaError_t e = cudaFuncSetAttribute(train_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(train_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_error("pn_train_gemm_bf16x3: cannot reserve %zu bytes of shared memory: %s", smem, cudaGetErrorString(e));
            return (int)e;
        }
        smem_set = smem;
    }
    a.w_packed = static_cast<const unsigned char*>(w_scratch);
    if (w) {      // w == NULL: w_scratch already holds the image (pn_train_pack_many at the start of the iteration)
        const int items = a.n_pad * (a.k_pad / 8);
        train_pack_kernel<<<(items + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, w_transposed, cin, cout, a.k_pad, a.n_pad,
                                                                                static_cast<unsigned char*>(w_scratch));
    }
    const int64_t tiles = ceil_div(rows, TM);
    const int64_t grid = tiles < (int64_t)sms * per_sm ? tiles : (int64_t)sms * per_sm;
    if (p_eval)
        train_gemm_kernel<true><<<(unsigned)grid, THREADS, smem, (cudaStream_t)stream>>>(a);
    else
        train_gemm_kernel<false><<<(unsigned)grid, THREADS, smem, (cudaStream_t)stream>>>(a);
    return finish_launch("pn_train_gemm_bf16x3");
}
