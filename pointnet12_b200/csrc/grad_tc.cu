// grad_tc.cu -- weight gradient of a 1x1 conv on the tensor cores (training step, SURVEY.md section 8 row f-1):
//     dW[co, ci] += sum_r dy[r, co] * x[r, ci]          db[co] += sum_r dy[r, co]
// Reference: the autograd backward of the Conv1d / Conv2d(kernel 1) layers of model/pointnet_util.py:195-197, :310-312
// and pointnet2.py:172-173, as driven by loss.backward() in pcdseg.py:184.
//
// This is a GEMM whose reduction dimension is the ROWS (64 k .. 262 k of them at config C5) and whose output is tiny
// (<= 512 x 768), so it is bound by reading dy and x once from HBM -- provided the arithmetic keeps up, which the CUDA
// cores do not (pn_grad_weight_f32: 65 us for a 128 x 128 layer over 64 k rows = 2.1 GFLOP, against 10 us of traffic).
// Here a CTA owns a 128 (co) x 128 (ci) tile of dW in TMEM (fp32, 128 columns) and a slab of rows:
//   * all 8 warps stream 32 rows at a time: every thread reads one channel of 16 rows (loads coalesced over the
//     channels), splits the fp32 values into bf16 hi + lo and writes them with 16-byte stores straight into the UMMA
//     K-major core-matrix layout (8 rows x 16 bytes, no swizzle) -- the transposition dy -> dy^T costs nothing, it is
//     just the address the thread writes to;
//   * an elected lane of warp 0 issues, per 16 rows, hi*hi + hi*lo + lo*hi (tcgen05.mma kind::f16, both operands from
//     shared memory, fp32 accumulation: fp32 parity like the forward chains) and commits the stage's mbarrier so the
//     producers can refill it (3-stage ring);
//   * at the end the accumulator is read back with tcgen05.ld and added to dW with fp32 atomics (the row slabs of one
//     tile meet there); the producers of the first ci tile also carry the column sums of dy for db.
#include "common.cuh"
#include "tcgen05.cuh"

namespace pn {
namespace gtc {

constexpr int TM = 128, TN = 128, KC = 32, NS = 3, THREADS = 256;
constexpr int IMG = TM * KC * 2;              // one bf16 image of a 128 x 32 operand tile: 8 KB
constexpr int STAGE = 4 * IMG;                // A hi, A lo, B hi, B lo
constexpr int SMEM = NS * STAGE + 1024;

__global__ void __launch_bounds__(THREADS)
grad_weight_tc_kernel(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ x, int64_t ldx, int64_t rows,
                      int64_t rows_per_split, int cout, int cin, float* __restrict__ dw, int64_t lddw,
                      float* __restrict__ db, int vec_red, const float* __restrict__ x_scale, const float* __restrict__ x_shift,
                      int x_relu) {
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + NS * STAGE);   // full[NS], empty[NS], done
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(bars + 2 * NS + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int co0 = blockIdx.x * TM, ci0 = blockIdx.y * TN;
    const int64_t r0 = (int64_t)blockIdx.z * rows_per_split;
    const int64_t r1 = min(rows, r0 + rows_per_split);
    const int chunks = (int)((r1 - r0 + KC - 1) / KC);
    const unsigned bar_full = tc::smem_u32(bars), bar_empty = tc::smem_u32(bars + NS), bar_done = tc::smem_u32(bars + 2 * NS);

    if (tid == 0) {
        for (int s = 0; s < NS; ++s) {
            tc::mbar_init(bar_full + 8 * s, THREADS);
            tc::mbar_init(bar_empty + 8 * s, 1);
        }
        tc::mbar_init(bar_done, 1);
        tc::mbar_init_fence();
    }
    if (warp == 0) tc::tmem_alloc(tmem_slot, 128);
    tc::fence_before();
    __syncthreads();
    tc::fence_after();
    const unsigned tbase = *tmem_slot;

    // producer role of this thread: channel m of both operand tiles, k-blocks {half, half + 2} of every 32-row chunk
    const int m = tid & 127, half = tid >> 7;
    const bool a_ok = co0 + m < cout, b_ok = ci0 + m < cin;
    const float* __restrict__ ap = dy + co0 + m;
    const float* __restrict__ bp = x + ci0 + m;
    const unsigned row_off = (unsigned)(m >> 3) * (KC / 8) * 128u + (unsigned)(m & 7) * 16u;
    const bool do_bias = db != nullptr && blockIdx.y == 0 && a_ok;
    // optional f(x) = relu(x * scale[ci] + shift[ci]) on the x operand: the normalise + ReLU of the layer that produced x,
    // when the forward kept only its pre-normalisation output (pn_train_gemm_bf16x3)
    const bool x_tf = x_scale != nullptr;
    const float xs = (x_tf && b_ok) ? x_scale[ci0 + m] : 1.0f, xh = (x_tf && b_ok) ? x_shift[ci0 + m] : 0.0f;
    float bsum = 0.0f;
    const unsigned idesc = tc::idesc_bf16_f32(TM, TN);
    const unsigned long long dbase = tc::sdesc_base((KC / 8) * 128u);      // 8-row groups (KC / 8) * 128 B apart

    // register double buffer: the loads of chunk c+1 are in flight while chunk c is converted, stored and multiplied
    float va[2][8], vb[2][8];
    auto load_chunk = [&](int c) {
        const int64_t k0 = r0 + (int64_t)c * KC;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int kb = half + 2 * q;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int64_t r = k0 + kb * 8 + j;
                const bool in = r < r1;
                va[q][j] = (in && a_ok) ? __ldg(ap + r * lddy) : 0.0f;
                vb[q][j] = (in && b_ok) ? __ldg(bp + r * ldx) : 0.0f;      // (kept branch-free: 32 loads in flight per thread)
            }
        }
    };
    if (chunks > 0) load_chunk(0);
    for (int c = 0; c < chunks; ++c) {
        const int s = c % NS;
        const unsigned use = (unsigned)(c / NS);
        float ca[2][8], cb[2][8];
#pragma unroll
        for (int q = 0; q < 2; ++q)
#pragma unroll
            for (int j = 0; j < 8; ++j) { ca[q][j] = va[q][j]; cb[q][j] = vb[q][j]; }
        if (c + 1 < chunks) load_chunk(c + 1);
        if (x_tf) {      // f(x) on the copy, after the next chunk's loads have been issued
            const int64_t k0 = r0 + (int64_t)c * KC;
#pragma unroll
            for (int q = 0; q < 2; ++q)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float t = fmaf(cb[q][j], xs, xh);
                    if (x_relu) t = fmaxf(t, 0.0f);
                    cb[q][j] = (b_ok && k0 + (half + 2 * q) * 8 + j < r1) ? t : 0.0f;
                }
        }
        if (c >= NS) tc::mbar_wait(bar_empty + 8 * s, (use - 1) & 1);      // the MMAs that read this stage have completed
        unsigned char* st = smem + s * STAGE;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int kb = half + 2 * q;
            if (do_bias) {
#pragma unroll
                for (int j = 0; j < 8; ++j) bsum += ca[q][j];
            }
            tc::store_split8(st, st + IMG, row_off + (unsigned)kb * 128u, ca[q]);
            tc::store_split8(st + 2 * IMG, st + 3 * IMG, row_off + (unsigned)kb * 128u, cb[q]);
        }
        tc::fence_proxy_async();
        tc::mbar_arrive(bar_full + 8 * s);
        if (warp == 0) {
            tc::mbar_wait(bar_full + 8 * s, use & 1);
            tc::fence_after();
            if (tc::elect()) {
                const unsigned a_hi = tc::smem_u32(st), a_lo = a_hi + IMG, b_hi = a_hi + 2 * IMG, b_lo = a_hi + 3 * IMG;
#pragma unroll
                for (int t = 0; t < KC / 16; ++t)
                    tc::mma_bf16x3(tbase, tc::sdesc(dbase, a_hi + t * 256), tc::sdesc(dbase, a_lo + t * 256),
                                   tc::sdesc(dbase, b_hi + t * 256), tc::sdesc(dbase, b_lo + t * 256), idesc, (c > 0 || t > 0) ? 1u : 0u);
                tc::commit(bar_empty + 8 * s);
                if (c + 1 == chunks) tc::commit(bar_done);
            }
            __syncwarp();
        }
    }
    // ---- epilogue: accumulator (lane = co row, column = ci) -> atomics into dW
    if (chunks > 0) {
        tc::mbar_wait(bar_done, 0);
        tc::fence_after();
        const int row = (warp & 3) * 32 + lane;                       // a warp reads the TMEM lanes of its quarter
        const int co = co0 + row;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int col0 = (warp >> 2) * 64 + h * 32;
            unsigned r[32];
            tc::ld32(tbase + ((unsigned)((warp & 3) * 32) << 16) + (unsigned)col0, r);
            if (co < cout) {
                float* dst = dw + (int64_t)co * lddw + ci0 + col0;
                if (vec_red && ci0 + col0 + 32 <= cin) {
                    // 16-byte vector reductions: a quarter of the atomic operations the row slabs send to the same tile
#pragma unroll
                    for (int j = 0; j < 32; j += 4)
                        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + j), "f"(__uint_as_float(r[j])),
                                     "f"(__uint_as_float(r[j + 1])), "f"(__uint_as_float(r[j + 2])), "f"(__uint_as_float(r[j + 3]))
                                     : "memory");
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (ci0 + col0 + j < cin) atomicAdd(dst + j, __uint_as_float(r[j]));
                }
            }
        }
        if (do_bias) atomicAdd(&db[co0 + m], bsum);
    }
    tc::fence_before();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tbase, 128);
}

}  // namespace gtc
}  // namespace pn

static int grad_weight_tc(const float* dy, int64_t lddy, const float* x, int64_t ldx, int64_t rows, int cout, int cin, float* dw,
                          int64_t lddw, float* db, const float* x_scale, const float* x_shift, int x_relu, pn_stream_t stream);
PN_EXPORT int pn_grad_weight_bf16x3(const float* dy, int64_t lddy, const float* x, int64_t ldx, int64_t rows, int cout,
                                    int cin, float* dw, int64_t lddw, float* db, pn_stream_t stream) {
    return grad_weight_tc(dy, lddy, x, ldx, rows, cout, cin, dw, lddw, db, nullptr, nullptr, 0, stream);
}

PN_EXPORT int pn_grad_weight_bn_bf16x3(const float* dy, int64_t lddy, const float* x, int64_t ldx, const float* x_scale,
                                       const float* x_shift, int x_relu, int64_t rows, int cout, int cin, float* dw,
                                       int64_t lddw, float* db, pn_stream_t stream) {
    PN_REQUIRE(x_scale && x_shift, PN_ERR_BAD_ARG, "pn_grad_weight_bn_bf16x3: null scale / shift");
    return grad_weight_tc(dy, lddy, x, ldx, rows, cout, cin, dw, lddw, db, x_scale, x_shift, x_relu, stream);
}

static int grad_weight_tc(const float* dy, int64_t lddy, const float* x, int64_t ldx, int64_t rows, int cout, int cin, float* dw,
                          int64_t lddw, float* db, const float* x_scale, const float* x_shift, int x_relu, pn_stream_t stream) {
    using namespace pn;
    using namespace pn::gtc;
    PN_REQUIRE(dy && x && dw, PN_ERR_BAD_ARG, "pn_grad_weight_bf16x3: null pointer");
    PN_REQUIRE(rows > 0 && cout > 0 && cin > 0 && lddy >= cout && ldx >= cin && lddw >= cin, PN_ERR_BAD_ARG,
               "pn_grad_weight_bf16x3: bad shape");
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaFuncSetAttribute(grad_weight_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
        if (sms <= 0) sms = 148;
    }
    const int64_t tiles = ceil_div(cout, TM) * ceil_div(cin, TN);
    // one CTA per SM: every extra row slab adds a whole tile of atomics on the same 128 x 128 addresses
    int64_t splits = ceil_div((int64_t)sms, tiles);
    int64_t rps = ceil_div(ceil_div(rows, splits), KC) * KC;
    if (rps < 4 * KC) rps = 4 * KC;
    splits = ceil_div(rows, rps);
    PN_REQUIRE(splits <= 65535, PN_ERR_UNSUPPORTED, "pn_grad_weight_bf16x3: too many row splits");
    dim3 grid((unsigned)ceil_div(cout, TM), (unsigned)ceil_div(cin, TN), (unsigned)splits);
    const int vec_red = ((uintptr_t)dw % 16 == 0) && (lddw % 4 == 0);
    grad_weight_tc_kernel<<<grid, THREADS, SMEM, (cudaStream_t)stream>>>(dy, lddy, x, ldx, rows, rps, cout, cin, dw, lddw, db,
                                                                        vec_red, x_scale, x_shift, x_relu);
    return finish_launch("pn_grad_weight_bf16x3");
}
