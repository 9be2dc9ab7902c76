// train.cu -- kernels of the TRAINING step of PointNet2SemSeg (SURVEY.md section 8, row f-1) and of the
// evaluation metrics (row f-2).  Reference: pcdseg.py:157-186 (forward in train mode, CrossEntropyLoss on the
// log-probabilities, backward, Adam) and pcdseg.py:58-97 (argmax, per-class I/U, accuracy).
//
// The training forward differs from inference in one way that matters for the kernels: BatchNorm normalises with the
// statistics of the CURRENT batch (over every row of the layer: B*S*K rows for a set-abstraction level, B*N for a
// feature-propagation level), so a layer is  GEMM -> column statistics -> normalise+ReLU  with a grid-wide reduction
// in the middle, and the activations of every layer are kept for the backward pass.  Everything here works on the
// point-major row matrices [rows, C] of the inference path.
//
//   forward   pn_linear_f32 (linear.cu)           y = x W^T + b
//             pn_bn_stats_f32                     column sums / sums of squares in fp64
//             pn_bn_finalize_f32                  mean, 1/sqrt(var+eps), scale/shift, running statistics (momentum)
//             pn_bn_act_f32 / pn_bn_act_max_f32   z = relu(y*scale+shift) / the same + max over nsample + arg-max
//             pn_dropout_f32                      Philox mask (or a given mask), scale 1/(1-p)
//             pn_log_softmax_f32 (group.cu), pn_cross_entropy_f32
//   backward  pn_log_softmax_bwd_f32, pn_dropout_f32 (mask reuse)
//             pn_bn_bwd_stats_f32                 sum(g), sum(g*xhat) with g = dz * [z > 0] (pooled: routed by arg-max)
//             pn_bn_bwd_apply_f32                 dy = gamma*invstd*(g - mean(g) - xhat*mean(g*xhat)); dgamma, dbeta
//             pn_bn_eval_bwd_f32                  eval-mode BatchNorm (running statistics): dy = scale*g, dgamma, dbeta
//                                                 in one pass (no batch coupling)
//             pn_grad_weight_f32                  dW += dy^T x, db += sum(dy)     (split over the rows, fp32 atomics)
//             pn_linear_f32 on W^T (pn_transpose_f32)   dx = dy W
//             pn_group_bwd_f32, pn_three_interpolate_bwd_f32    scatter-add through the gathers
//   step      pn_adam_f32                         torch.optim.Adam (L2 weight decay) on one flat parameter buffer
//   metrics   pn_seg_metrics_f32 + pn_seg_metrics_accumulate     pcdseg.py:72-83 without host round trips
//   function-level gradients (model/pointnet_util.py, model/chamfer.py)
//             pn_square_distance_bwd_f32          one read of dL/ddist: row and column sums, then 2 (sum g) x - 2 sum g y
//             pn_chamfer_argmin_f32, pn_chamfer_bwd_f32    nearest points kept by the forward, norm backward of each pair
//
// All of these are HBM-bound streaming / reduction kernels except pn_grad_weight_f32 (CUDA-core SGEMM with a long K).
#include <math_constants.h>

#include "common.cuh"

namespace pn {

static inline int sm_count() {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return sms;
}

// ------------------------------------------------------------------------------------------------
// Column statistics.  Block = 32 channels x 16 row lanes; a warp reads 128 contiguous bytes of a row.
// MODE 0: s1 = sum y, s2 = sum y^2.
// MODE 1: g = dz * [y*scale+shift > 0] (relu) ; xhat = (y-mean)*invstd ; s1 = sum g, s2 = sum g*xhat.
// MODE 2: as 1 with dz routed from the pooled gradient: g = dpool[row/K] if argmax[row/K] == row%K.
constexpr int ST_LANES = 16;

// DET: s1 / s2 are [gridDim.x, C] partial rows, one per block, written instead of added (col_partials_sum_kernel adds them in
// block order).
template <int MODE, bool DET = false>
__global__ void __launch_bounds__(32 * ST_LANES)
col_stats_kernel(const float* __restrict__ y, int64_t ldy, int64_t rows, int C, int64_t rows_per_block,
                 const float* __restrict__ dz, int64_t lddz, const int32_t* __restrict__ argmax, int K,
                 const float* __restrict__ scale, const float* __restrict__ shift, const float* __restrict__ mean,
                 const float* __restrict__ invstd, int relu, double* __restrict__ s1, double* __restrict__ s2) {
    __shared__ double r1[ST_LANES][33], r2[ST_LANES][33];
    const int lane = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int c = blockIdx.y * 32 + lane;
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
    const int64_t r1e = min(rows, r0 + rows_per_block);
    double a1 = 0.0, a2 = 0.0;
    if (c < C) {
        float sc = 0.f, sh = 0.f, mu = 0.f, is = 0.f;
        if (MODE != 0) { sc = scale[c]; sh = shift[c]; mu = mean[c]; is = invstd[c]; }
        for (int64_t r = r0 + ry; r < r1e; r += ST_LANES) {
            const float v = y[r * ldy + c];
            if (MODE == 0) {
                const double d = (double)v;
                a1 += d;
                a2 = fma(d, d, a2);
            } else {
                float g;
                if (MODE == 1) {
                    g = dz[r * lddz + c];
                } else {
                    const int64_t grp = r / K;
                    g = (argmax[grp * C + c] == (int)(r - grp * K)) ? dz[grp * lddz + c] : 0.0f;
                }
                if (relu && !(fmaf(v, sc, sh) > 0.0f)) g = 0.0f;
                const float xh = (v - mu) * is;
                a1 += (double)g;
                a2 = fma((double)g, (double)xh, a2);
            }
        }
    }
    r1[ry][lane] = a1;
    r2[ry][lane] = a2;
    __syncthreads();
    if (ry == 0 && c < C) {
#pragma unroll
        for (int i = 1; i < ST_LANES; ++i) { a1 += r1[i][lane]; a2 += r2[i][lane]; }
        if (DET) {
            s1[(int64_t)blockIdx.x * C + c] = a1;
            s2[(int64_t)blockIdx.x * C + c] = a2;
        } else {
            atomicAdd(&s1[c], a1);
            atomicAdd(&s2[c], a2);
        }
    }
}

// s1[c] += sum_b part[b, c], s2[c] += sum_b part[blocks + b, c], b ascending: the deterministic end of the column reductions.
__global__ void col_partials_sum_kernel(const double* __restrict__ part, int blocks, int C, double* __restrict__ s1,
                                        double* __restrict__ s2) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double a1 = 0.0, a2 = 0.0;
    for (int b = 0; b < blocks; ++b) {
        a1 += part[(int64_t)b * C + c];
        a2 += part[(int64_t)(blocks + b) * C + c];
    }
    s1[c] += a1;
    s2[c] += a2;
}

static inline void stats_grid(int64_t rows, int C, dim3* grid, int64_t* rows_per_block) {
    const int cy = (int)ceil_div(C, 32);
    int64_t bx = ceil_div((int64_t)sm_count() * 8, cy);
    int64_t rpb = ceil_div(rows, bx);
    rpb = ceil_div(rpb < 64 ? 64 : rpb, ST_LANES) * ST_LANES;
    *rows_per_block = rpb;
    *grid = dim3((unsigned)ceil_div(rows, rpb), (unsigned)cy, 1);
}

__global__ void bn_finalize_kernel(const double* __restrict__ s1, const double* __restrict__ s2, int64_t n, int C,
                                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                   float momentum, float* __restrict__ running_mean, float* __restrict__ running_var,
                                   int64_t* __restrict__ num_batches_tracked, float* __restrict__ scale,
                                   float* __restrict__ shift, float* __restrict__ mean, float* __restrict__ invstd) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c == 0 && num_batches_tracked) *num_batches_tracked += 1;
    if (c >= C) return;
    const double mu = s1[c] / (double)n;
    double var = s2[c] / (double)n - mu * mu;
    if (var < 0.0) var = 0.0;
    const float is = (float)(1.0 / sqrt(var + (double)eps));
    const float g = gamma ? gamma[c] : 1.0f, b = beta ? beta[c] : 0.0f;
    mean[c] = (float)mu;
    invstd[c] = is;
    scale[c] = g * is;
    shift[c] = b - (float)mu * (g * is);
    if (running_mean) running_mean[c] = (1.0f - momentum) * running_mean[c] + momentum * (float)mu;
    if (running_var) {
        const double unbiased = n > 1 ? var * ((double)n / (double)(n - 1)) : var;
        running_var[c] = (1.0f - momentum) * running_var[c] + momentum * (float)unbiased;
    }
}

// z = act(y*scale + shift), elementwise over [rows, C].
__global__ void bn_act_kernel(const float* __restrict__ y, int64_t ldy, int64_t rows, int C,
                              const float* __restrict__ scale, const float* __restrict__ shift, int relu,
                              float* __restrict__ z, int64_t ldz) {
    const int64_t total = rows * C;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(e % C);
        const int64_t r = e / C;
        float v = fmaf(y[r * ldy + c], scale[c], shift[c]);
        if (relu) v = fmaxf(v, 0.0f);
        z[r * ldz + c] = v;
    }
}

// pooled[g,c] = max_k act(y[g*K+k,c]*scale+shift), argmax = the first k attaining it (torch.max(dim) on CPU).
__global__ void bn_act_max_kernel(const float* __restrict__ y, int64_t ldy, int64_t groups, int K, int C,
                                  const float* __restrict__ scale, const float* __restrict__ shift, int relu,
                                  float* __restrict__ out, int64_t ldo, int32_t* __restrict__ argmax) {
    const int64_t total = groups * C;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(e % C);
        const int64_t g = e / C;
        const float sc = scale[c], sh = shift[c];
        const float* __restrict__ r = y + g * K * ldy + c;
        float m = -CUDART_INF_F;
        int am = 0;
        for (int k = 0; k < K; ++k) {
            float v = fmaf(r[(int64_t)k * ldy], sc, sh);
            if (relu) v = fmaxf(v, 0.0f);
            if (v > m) { m = v; am = k; }
        }
        out[g * ldo + c] = m;
        argmax[g * C + c] = am;
    }
}

// Tall variant (K >= 256: the global max over the N points of a cloud in the PointNet nets and group-all levels): one CTA per
// (group, 32-channel slab), 8 row lanes per channel, then a shared-memory reduction that keeps the FIRST maximum.
__global__ void __launch_bounds__(256)
bn_act_max_tall_kernel(const float* __restrict__ y, int64_t ldy, int K, int C, const float* __restrict__ scale,
                       const float* __restrict__ shift, int relu, float* __restrict__ out, int64_t ldo,
                       int32_t* __restrict__ argmax) {
    __shared__ float vmax[8][33];
    __shared__ int vidx[8][33];
    const int64_t g = blockIdx.y;
    const int lane = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + lane;
    float m = -CUDART_INF_F;
    int am = 0;
    if (c < C) {
        const float sc = scale[c], sh = shift[c];
        const float* __restrict__ r = y + g * K * ldy + c;
        for (int k = ry; k < K; k += 8) {
            float v = fmaf(r[(int64_t)k * ldy], sc, sh);
            if (relu) v = fmaxf(v, 0.0f);
            if (v > m) { m = v; am = k; }           // a lane sees its rows in ascending order: first maximum of the lane
        }
    }
    vmax[ry][lane] = m;
    vidx[ry][lane] = am;
    __syncthreads();
    if (ry == 0 && c < C) {
#pragma unroll
        for (int i = 1; i < 8; ++i) {
            const float v = vmax[i][lane];
            const int k = vidx[i][lane];
            if (v > m || (v == m && k < am)) { m = v; am = k; }      // ties across lanes: the lowest row index
        }
        out[g * ldo + c] = m;
        argmax[g * C + c] = am;
    }
}

// dy = gamma*invstd * (g - s1/n - xhat*s2/n); block 0 also adds s2 to dgamma and s1 to dbeta.
template <int MODE>
__global__ void bn_bwd_apply_kernel(const float* __restrict__ y, int64_t ldy, int64_t rows, int C,
                                    const float* __restrict__ dz, int64_t lddz, const int32_t* __restrict__ argmax, int K,
                                    const float* __restrict__ scale, const float* __restrict__ shift,
                                    const float* __restrict__ mean, const float* __restrict__ invstd, int relu,
                                    const double* __restrict__ s1, const double* __restrict__ s2,
                                    float* __restrict__ dy, int64_t lddy, float* __restrict__ dgamma,
                                    float* __restrict__ dbeta) {
    const int64_t total = rows * C;
    const double inv_n = 1.0 / (double)rows;
    if (blockIdx.x == 0) {
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            if (dgamma) dgamma[c] += (float)s2[c];      // accumulated, like dW / db (a single writer: no atomics)
            if (dbeta) dbeta[c] += (float)s1[c];
        }
    }
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(e % C);
        const int64_t r = e / C;
        const float v = y[r * ldy + c];
        const float sc = scale[c], sh = shift[c];
        float g;
        if (MODE == 1) {
            g = dz[r * lddz + c];
        } else {
            const int64_t grp = r / K;
            g = (argmax[grp * C + c] == (int)(r - grp * K)) ? dz[grp * lddz + c] : 0.0f;
        }
        if (relu && !(fmaf(v, sc, sh) > 0.0f)) g = 0.0f;
        const float xh = (v - mean[c]) * invstd[c];
        const float m1 = (float)(s1[c] * inv_n), m2 = (float)(s2[c] * inv_n);
        dy[r * lddy + c] = sc * (g - m1 - xh * m2);      // scale = gamma * invstd
    }
}

// Backward of act(bn(y)) with FIXED statistics (eval-mode BatchNorm: running mean / variance), one pass: the statistics
// do not depend on the batch, so dy = scale*g needs no column reduction first.  g = dz * [y*scale+shift > 0] (POOLED:
// routed from dz[row/K] by the arg-max of bn_act_max, either layout); dy = scale*g; s1 += sum g, s2 += sum g*xhat with
// xhat = (y-mean)*invstd (fp64 per block, one atomic per column per block).  Same block shape as col_stats_kernel.
template <bool POOLED, bool DET = false>
__global__ void __launch_bounds__(32 * ST_LANES)
bn_eval_bwd_kernel(const float* __restrict__ y, int64_t ldy, int64_t rows, int C, int64_t rows_per_block,
                   const float* __restrict__ dz, int64_t lddz, const int32_t* __restrict__ argmax, int K,
                   const float* __restrict__ scale, const float* __restrict__ shift, const float* __restrict__ mean,
                   const float* __restrict__ invstd, int relu, double* __restrict__ s1, double* __restrict__ s2,
                   float* __restrict__ dy, int64_t lddy) {
    __shared__ double r1[ST_LANES][33], r2[ST_LANES][33];
    const int lane = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int c = blockIdx.y * 32 + lane;
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
    const int64_t r1e = min(rows, r0 + rows_per_block);
    double a1 = 0.0, a2 = 0.0;
    if (c < C) {
        const float sc = scale[c], sh = shift[c], mu = mean[c], is = invstd[c];
        for (int64_t r = r0 + ry; r < r1e; r += ST_LANES) {
            const float v = y[r * ldy + c];
            float g;
            if (!POOLED) {
                g = dz[r * lddz + c];
            } else {
                const int64_t grp = r / K;
                g = (argmax[grp * C + c] == (int)(r - grp * K)) ? dz[grp * lddz + c] : 0.0f;
            }
            if (relu && !(fmaf(v, sc, sh) > 0.0f)) g = 0.0f;
            dy[r * lddy + c] = sc * g;
            a1 += (double)g;
            a2 = fma((double)g, (double)((v - mu) * is), a2);
        }
    }
    r1[ry][lane] = a1;
    r2[ry][lane] = a2;
    __syncthreads();
    if (ry == 0 && c < C) {
#pragma unroll
        for (int i = 1; i < ST_LANES; ++i) { a1 += r1[i][lane]; a2 += r2[i][lane]; }
        if (DET) {      // partial rows as in col_stats_kernel
            s1[(int64_t)blockIdx.x * C + c] = a1;
            s2[(int64_t)blockIdx.x * C + c] = a2;
        } else {
            atomicAdd(&s1[c], a1);
            atomicAdd(&s2[c], a2);
        }
    }
}

// dgamma += s2, dbeta += s1 (either may be NULL): the affine gradients of the fixed-statistics backward.
__global__ void bn_eval_bwd_finalize_kernel(const double* __restrict__ s1, const double* __restrict__ s2, int C,
                                            float* __restrict__ dgamma, float* __restrict__ dbeta) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    if (dgamma) dgamma[c] += (float)s2[c];
    if (dbeta) dbeta[c] += (float)s1[c];
}

// ------------------------------------------------------------------------------------------------
// dW[co,ci] += sum_r dy[r,co] * x[r,ci]; db[co] += sum_r dy[r,co].  Both operands are read along their rows
// (channels contiguous), so a K step is BK rows of each: straight 16-byte loads into shared memory, no transpose.
// grid = (co tiles, ci tiles, row splits); fp32 atomics into the pre-zeroed (or accumulating) dW.
// DET: dw / db point to a workspace of [gridDim.z] slabs of [cout, lddw] / [cout]; each row split stores its partial tile
// there (slab_sum_kernel adds the slabs in split order).
template <int BM, int BN, int BK, int TM, int TN, bool DET = false>
__global__ void __launch_bounds__((BM / TM) * (BN / TN))
grad_weight_kernel(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ x, int64_t ldx, int64_t rows,
                   int64_t rows_per_split, int cout, int cin, float* __restrict__ dw, int64_t lddw,
                   float* __restrict__ db, int vec_ok) {
    constexpr int THREADS = (BM / TM) * (BN / TN);
    __shared__ __align__(16) float As[BK][BM + 4];
    __shared__ __align__(16) float Bs[BK][BN + 4];
    const int co0 = blockIdx.x * BM, ci0 = blockIdx.y * BN;
    const int64_t r0 = (int64_t)blockIdx.z * rows_per_split;
    const int64_t r1 = min(rows, r0 + rows_per_split);
    const int tid = threadIdx.x;
    const int tx = tid % (BN / TN), ty = tid / (BN / TN);
    const bool do_bias = db != nullptr && blockIdx.y == 0 && tx == 0;
    float acc[TM][TN];
    float bsum[TM];
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        bsum[i] = 0.0f;
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.0f;
    }
    constexpr int AV = BM / 4, BV = BN / 4;
    for (int64_t k0 = r0; k0 < r1; k0 += BK) {
        for (int e = tid; e < BK * AV; e += THREADS) {
            const int k = e / AV, cq = (e % AV) * 4;
            const int64_t r = k0 + k;
            const int gc = co0 + cq;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < r1) {
                const float* src = dy + r * lddy + gc;
                if ((vec_ok & 1) && gc + 3 < cout) {
                    v = *reinterpret_cast<const float4*>(src);
                } else {
                    if (gc < cout) v.x = src[0];
                    if (gc + 1 < cout) v.y = src[1];
                    if (gc + 2 < cout) v.z = src[2];
                    if (gc + 3 < cout) v.w = src[3];
                }
            }
            *reinterpret_cast<float4*>(&As[k][cq]) = v;
        }
        for (int e = tid; e < BK * BV; e += THREADS) {
            const int k = e / BV, cq = (e % BV) * 4;
            const int64_t r = k0 + k;
            const int gc = ci0 + cq;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < r1) {
                const float* src = x + r * ldx + gc;
                if ((vec_ok & 2) && gc + 3 < cin) {
                    v = *reinterpret_cast<const float4*>(src);
                } else {
                    if (gc < cin) v.x = src[0];
                    if (gc + 1 < cin) v.y = src[1];
                    if (gc + 2 < cin) v.z = src[2];
                    if (gc + 3 < cin) v.w = src[3];
                }
            }
            *reinterpret_cast<float4*>(&Bs[k][cq]) = v;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float a[TM], b[TN];
#pragma unroll
            for (int i = 0; i < TM; i += 4) {
                const float4 t = *reinterpret_cast<const float4*>(&As[k][ty * TM + i]);
                a[i] = t.x; a[i + 1] = t.y; a[i + 2] = t.z; a[i + 3] = t.w;
            }
#pragma unroll
            for (int j = 0; j < TN; j += 4) {
                const float4 t = *reinterpret_cast<const float4*>(&Bs[k][tx * TN + j]);
                b[j] = t.x; b[j + 1] = t.y; b[j + 2] = t.z; b[j + 3] = t.w;
            }
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            if (do_bias) {
#pragma unroll
                for (int i = 0; i < TM; ++i) bsum[i] += a[i];
            }
        }
        __syncthreads();
    }
    if (DET) {
        dw += (int64_t)blockIdx.z * cout * lddw;
        if (db) db += (int64_t)blockIdx.z * cout;
    }
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        const int co = co0 + ty * TM + i;
        if (co >= cout) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int ci = ci0 + tx * TN + j;
            if (ci < cin) {
                if (DET) dw[(int64_t)co * lddw + ci] = acc[i][j];
                else atomicAdd(&dw[(int64_t)co * lddw + ci], acc[i][j]);
            }
        }
        if (do_bias) {
            if (DET) db[co] = bsum[i];
            else atomicAdd(&db[co], bsum[i]);
        }
    }
}

// dw[co, ci] += sum_s ws[s, co, ci] and db[co] += sum_p wsb[p, co] in ascending slab order: the deterministic end of the
// weight gradients (ws [splits, cout, cin], wsb [bias_parts, cout] right behind it).
__global__ void slab_sum_kernel(const float* __restrict__ ws, int splits, int bias_parts, int cout, int cin,
                                float* __restrict__ dw, int64_t lddw, float* __restrict__ db) {
    const int64_t tile = (int64_t)cout * cin, total = tile + (db ? cout : 0);
    const float* __restrict__ wsb = ws + (int64_t)splits * tile;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        float acc = 0.0f;
        if (e < tile) {
            for (int s = 0; s < splits; ++s) acc += ws[s * tile + e];
            dw[(e / cin) * lddw + e % cin] += acc;
        } else {
            const int64_t co = e - tile;
            for (int p = 0; p < bias_parts; ++p) acc += wsb[p * (int64_t)cout + co];
            db[co] += acc;
        }
    }
}

__global__ void transpose_kernel(const float* __restrict__ in, int rows, int cols, float* __restrict__ out) {
    __shared__ float tile[32][33];
    const int x = blockIdx.x * 32 + threadIdx.x;
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int yy = blockIdx.y * 32 + j;
        if (x < cols && yy < rows) tile[j][threadIdx.x] = in[(int64_t)yy * cols + x];
    }
    __syncthreads();
    const int ox = blockIdx.y * 32 + threadIdx.x;   // column of out = row of in
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int oy = blockIdx.x * 32 + j;
        if (ox < rows && oy < cols) out[(int64_t)oy * rows + ox] = tile[threadIdx.x][j];
    }
}

// ------------------------------------------------------------------------------------------------
// Scatter-add through the gathers.
// grouped rows (b,s,k) had channels [xyz_rel(3), feat(D)] (or [feat, xyz_rel] in MSG order); only feat carries grad.
__global__ void group_bwd_kernel(const float* __restrict__ dg, int64_t ldg, int col0, int D,
                                 const int64_t* __restrict__ idx, int N, int64_t SK, int64_t total,
                                 float* __restrict__ dfeat) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(e % D);
        const int64_t row = e / D;
        const int64_t b = row / SK;
        int64_t j = idx[row];
        j = j < 0 ? 0 : (j >= N ? N - 1 : j);
        atomicAdd(&dfeat[(b * N + j) * D + c], dg[row * ldg + col0 + c]);
    }
}

// rows (b,n) of dx = [d points1 (D1) | d interpolated (D2)]; DP2 = false: dp1 only (the deterministic path pulls dp2)
template <bool DP2 = true>
__global__ void three_interpolate_bwd_kernel(const float* __restrict__ dx, int64_t ldx, int D1, int D2,
                                             const int64_t* __restrict__ idx, const float* __restrict__ weight, int N,
                                             int S, int64_t total, float* __restrict__ dp1, float* __restrict__ dp2) {
    const int C = D1 + D2;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(e % C);
        const int64_t row = e / C;
        const float g = dx[row * ldx + c];
        if (c < D1) {
            dp1[row * D1 + c] = g;
        } else if (DP2) {
            const int64_t b = row / N;
            const int cc = c - D1;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                int64_t j = idx[row * 3 + k];
                j = j < 0 ? 0 : (j >= S ? S - 1 : j);
                atomicAdd(&dp2[(b * S + j) * D2 + cc], g * weight[row * 3 + k]);
            }
        }
    }
}

// Coordinate gradient of the grouping (pointnet_util.py:127-131, :243-247; group-all :151-156).  The three xyz_rel
// columns at col0 of row (b,s,k) go to dxyz[b, idx[b,s,k]] (a padded ball repeats its first hit: each repeat adds its own
// share); the recentring subtracted new_xyz[b,s] from every row of the group, so dnew[b,s] = -sum_k (dnew = NULL: group-all,
// not recentred).  One warp per group, lanes over k.  SCATTER = false: dnew only (the deterministic path pulls dxyz).
template <bool SCATTER = true>
__global__ void __launch_bounds__(256)
group_bwd_xyz_kernel(const float* __restrict__ dg, int64_t ldg, int col0, const int64_t* __restrict__ idx, int N, int S,
                     int K, int64_t groups, float* __restrict__ dxyz, float* __restrict__ dnew) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t grp = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); grp < groups; grp += warps) {
        const int64_t b = grp / S;
        float sx = 0.0f, sy = 0.0f, sz = 0.0f;
        for (int k = lane; k < K; k += 32) {
            const int64_t row = grp * K + k;
            const float* r = dg + row * ldg + col0;
            const float x = r[0], y = r[1], z = r[2];
            if (SCATTER) {
                int64_t j = idx[row];
                j = j < 0 ? 0 : (j >= N ? N - 1 : j);
                float* o = dxyz + (b * N + j) * 3;
                atomicAdd(o, x);
                atomicAdd(o + 1, y);
                atomicAdd(o + 2, z);
            }
            sx += x;
            sy += y;
            sz += z;
        }
        if (dnew) {
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                sx += __shfl_xor_sync(0xffffffffu, sx, o);
                sy += __shfl_xor_sync(0xffffffffu, sy, o);
                sz += __shfl_xor_sync(0xffffffffu, sz, o);
            }
            if (lane == 0) {
                dnew[grp * 3] = -sx;
                dnew[grp * 3 + 1] = -sy;
                dnew[grp * 3 + 2] = -sz;
            }
        }
    }
}

// three_interpolate_bwd_kernel plus the gradient of the 3-NN weights w.r.t. both clouds (pointnet_util.py:295-307).  One
// warp per fine row n of cloud b, lanes over the channels; the row of dx is read once.  With a = xyz1[n], b_k = xyz2[idx_k]:
//   d_k = the forward's fp32 expansion-formula distance (sqdist_expand: same clamp decision, same 1/d as the 3-NN kernels)
//   r_k = 1/max(d_k, 1e-10), R = sum r, w_k = r_k/R (the forward's weights), g_k = <dinterp, p2[idx_k]>
//   dL/dd_j = -(g_j - sum_k w_k g_k) / R * r_j^2, or 0 where d_j was clamped (the masked assignment stops the gradient)
//   dxyz1[n] = sum_j dL/dd_j * 2(a - b_j),   dxyz2[idx_j] += -dL/dd_j * 2(a - b_j)
// VEC: the dx row (from D1), the p2 rows and the dp2 rows are read / added as float4.
// DET: nothing is added to dp2 (pulled afterwards) and dxyz2 is a [rows, 3, 3] workspace of the per-slot terms, written.
template <bool VEC, bool DET = false>
__global__ void __launch_bounds__(256)
three_interpolate_bwd_xyz_kernel(const float* __restrict__ dx, int64_t ldx, int D1, int D2, const int64_t* __restrict__ idx,
                                 const float* __restrict__ weight, const float* __restrict__ p2, int64_t p2B, int64_t p2S,
                                 int64_t p2C, const float* __restrict__ xyz1, int64_t aB, int64_t aN, int64_t aC,
                                 const float* __restrict__ xyz2, int64_t bB, int64_t bS, int64_t bC, int N, int S, int64_t rows,
                                 float* __restrict__ dp1, float* __restrict__ dp2, float* __restrict__ dxyz1,
                                 float* __restrict__ dxyz2) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t row = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); row < rows; row += warps) {
        const int64_t b = row / N, n = row - b * N;
        const float* g = dx + row * ldx;
        int64_t j[3];
        float w[3], dot[3] = {0.0f, 0.0f, 0.0f};
        const float* q[3];
        float* o[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            int64_t jj = idx[row * 3 + k];
            j[k] = jj < 0 ? 0 : (jj >= S ? S - 1 : jj);
            w[k] = weight[row * 3 + k];
            q[k] = p2 + b * p2B + j[k] * p2S;
            o[k] = dp2 + (b * S + j[k]) * D2;
        }
        if (VEC) {
            for (int c = lane * 4; c < D1; c += 128)
                *reinterpret_cast<float4*>(dp1 + row * D1 + c) = *reinterpret_cast<const float4*>(g + c);
            for (int c = lane * 4; c < D2; c += 128) {
                const float4 gv = *reinterpret_cast<const float4*>(g + D1 + c);
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float4 pv = *reinterpret_cast<const float4*>(q[k] + c);
                    dot[k] = fmaf(gv.x, pv.x, fmaf(gv.y, pv.y, fmaf(gv.z, pv.z, fmaf(gv.w, pv.w, dot[k]))));
                    if (!DET) atomicAdd(reinterpret_cast<float4*>(o[k] + c), make_float4(gv.x * w[k], gv.y * w[k], gv.z * w[k], gv.w * w[k]));
                }
            }
        } else {
            for (int c = lane; c < D1; c += 32) dp1[row * D1 + c] = g[c];
            for (int c = lane; c < D2; c += 32) {
                const float gv = g[D1 + c];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    dot[k] = fmaf(gv, q[k][c * p2C], dot[k]);
                    if (!DET) atomicAdd(o[k] + c, gv * w[k]);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int s = 16; s; s >>= 1) dot[k] += __shfl_xor_sync(0xffffffffu, dot[k], s);
        if (lane != 0) continue;
        const float* pa = xyz1 + b * aB + n * aN;
        const float ax = pa[0], ay = pa[aC], az = pa[2 * aC];
        const float sa = sqnorm3(ax, ay, az);
        float r[3], ex[3], ey[3], ez[3];
        bool live[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float* pb = xyz2 + b * bB + j[k] * bS;
            const float bx = pb[0], by = pb[bC], bz = pb[2 * bC];
            const float d = sqdist_expand(ax, ay, az, sa, bx, by, bz, sqnorm3(bx, by, bz));
            live[k] = !(d < 1e-10f);
            r[k] = __fdiv_rn(1.0f, live[k] ? d : 1e-10f);
            ex[k] = ax - bx;
            ey[k] = ay - by;
            ez[k] = az - bz;
        }
        const float R = r[0] + r[1] + r[2];
        const float mean = w[0] * dot[0] + w[1] * dot[1] + w[2] * dot[2];
        float gx = 0.0f, gy = 0.0f, gz = 0.0f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            // 2 dL/dd_k; the product is grouped so that r^2 (up to 1e20) never stands alone
            const float t = live[k] ? -2.0f * ((dot[k] - mean) / R * r[k]) * r[k] : 0.0f;
            const float tx = t * ex[k], ty = t * ey[k], tz = t * ez[k];
            gx += tx;
            gy += ty;
            gz += tz;
            if (DET) {
                float* o2 = dxyz2 + (row * 3 + k) * 3;
                o2[0] = -tx;
                o2[1] = -ty;
                o2[2] = -tz;
            } else {
                float* o2 = dxyz2 + (b * S + j[k]) * 3;
                atomicAdd(o2, -tx);
                atomicAdd(o2 + 1, -ty);
                atomicAdd(o2 + 2, -tz);
            }
        }
        dxyz1[row * 3] = gx;
        dxyz1[row * 3 + 1] = gy;
        dxyz1[row * 3 + 2] = gz;
    }
}

// ------------------------------------------------------------------------------------------------
// Dropout.  Philox4x32-10 keyed by (seed), counter = (element / 4, offset): four uniform words per call.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += 0x9E3779B9u;
        key.y += 0xBB67AE85u;
    }
    return ctr;
}

// y = x * keep / (1-p).  mask_in != NULL: keep = mask_in (bytes); else keep is drawn (P(keep) = 1-p) from the Philox
// stream named by *seed_offset = {seed, offset} (device memory: a CUDA graph replays with fresh values) and written
// to mask_out.  Dense [rows*C] element indexing for the random stream, leading dimensions for the data.
__global__ void dropout_kernel(const float* __restrict__ x, int64_t ldx, int64_t rows, int C, float p,
                               const uint64_t* __restrict__ seed_offset, const uint8_t* __restrict__ mask_in,
                               uint8_t* __restrict__ mask_out, float* __restrict__ y, int64_t ldy) {
    const int64_t total = rows * C;
    const float inv_keep = 1.0f / (1.0f - p);
    const int64_t quads = (total + 3) / 4;
    uint2 key = make_uint2(0, 0);
    uint32_t off_lo = 0, off_hi = 0;
    if (!mask_in) {
        const uint64_t seed = seed_offset[0], off = seed_offset[1];
        key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
        off_lo = (uint32_t)off;
        off_hi = (uint32_t)(off >> 32);
    }
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < quads; q += (int64_t)gridDim.x * blockDim.x) {
        uint32_t rnd[4] = {0, 0, 0, 0};
        if (!mask_in) {
            const uint4 r = philox4x32_10(make_uint4((uint32_t)q, (uint32_t)((uint64_t)q >> 32), off_lo, off_hi), key);
            rnd[0] = r.x; rnd[1] = r.y; rnd[2] = r.z; rnd[3] = r.w;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t e = q * 4 + i;
            if (e >= total) break;
            const int c = (int)(e % C);
            const int64_t r = e / C;
            uint8_t keep;
            if (mask_in) {
                keep = mask_in[e];
            } else {
                // uniform in [0,1) from the top 24 bits; keep when u >= p
                keep = ((float)(rnd[i] >> 8) * (1.0f / 16777216.0f)) >= p ? 1 : 0;
                if (mask_out) mask_out[e] = keep;
            }
            y[r * ldy + c] = keep ? x[r * ldx + c] * inv_keep : 0.0f;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// nn.CrossEntropyLoss()(x.transpose(2,1), target) of pcdseg.py:177-178 on rows x [rows, C] (the reference feeds the
// network's log-probabilities, so CrossEntropyLoss normalises them once more): loss = mean_i (lse(x_i) - x_i[t_i]);
// dx[i,c] = (softmax(x_i)[c] - [c == t_i]) * grad_scale / n.  Rows labelled IGNORE_INDEX (CrossEntropyLoss's default
// ignore_index) add nothing to the loss, get a zero gradient and are not counted in n, the number of the other rows;
// n is counted on the device by label_count_kernel first (so the call needs no host synchronisation), and with every
// row ignored the loss is 0/0 = NaN, as in torch.  One row per thread; loss summed in fp64.
constexpr int64_t IGNORE_INDEX = -100;

__global__ void __launch_bounds__(256)
label_count_kernel(const int64_t* __restrict__ target, int64_t rows, double* __restrict__ count) {
    int local = 0;
    for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x)
        local += target[r] != IGNORE_INDEX;
    local = __reduce_add_sync(0xffffffffu, local);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(count, (double)local);
}

// DET: loss_sum is a [gridDim.x] array of block partials, written (ordered_sum_kernel adds them in block order).
template <bool DET = false>
__global__ void __launch_bounds__(256)
cross_entropy_kernel(const float* __restrict__ x, int64_t ldx, const int64_t* __restrict__ target, int64_t rows, int C,
                     double* __restrict__ loss_sum, const double* __restrict__ count, float* __restrict__ dx, int64_t lddx,
                     float grad_scale) {
    __shared__ double red[8];
    double local = 0.0;
    const float k = grad_scale / (float)*count;
    for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
        if (target[r] == IGNORE_INDEX) {
            if (dx)
                for (int c = 0; c < C; ++c) dx[r * lddx + c] = 0.0f;
            continue;
        }
        const float* __restrict__ xr = x + r * ldx;
        float m = -CUDART_INF_F;
        for (int c = 0; c < C; ++c) m = fmaxf(m, xr[c]);
        float s = 0.0f;
        for (int c = 0; c < C; ++c) s += expf(xr[c] - m);
        const float ls = logf(s);
        const int64_t t = target[r];
        if (t < 0 || t >= C) {
            // nn.CrossEntropyLoss raises on any other label outside [0, C); an asynchronous kernel cannot, so the loss and this
            // row's gradient are poisoned with NaN instead of being computed against a clamped label
            local += (double)CUDART_NAN_F;
            if (dx)
                for (int c = 0; c < C; ++c) dx[r * lddx + c] = CUDART_NAN_F;
            continue;
        }
        // lse(x) = m + log(s) is not formed: at |m| ~ 1e4 its float32 rounding (1e-3) would be the error of every softmax
        // entry.  The loss is (m - x[t]) + log(s), the softmax exp(x - m) / s.
        local += (double)((m - xr[t]) + ls);
        if (dx) {
            const float inv_s = 1.0f / s;
            for (int c = 0; c < C; ++c) dx[r * lddx + c] = (expf(xr[c] - m) * inv_s - (c == (int)t ? 1.0f : 0.0f)) * k;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
        if (DET) loss_sum[blockIdx.x] = t;
        else atomicAdd(loss_sum, t);
    }
}

// *out = sum of part[0, n): one warp, lane l adds the partials l, l + 32, ... in order, then a fixed butterfly.
__global__ void ordered_sum_kernel(const double* __restrict__ part, int64_t n, double* __restrict__ out) {
    double t = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 32) t += part[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) *out = t;
}

__global__ void loss_finalize_kernel(const double* __restrict__ loss_sum, const double* __restrict__ count,
                                     float* __restrict__ loss) {
    *loss = (float)(*loss_sum / *count);
}

// log_softmax backward: dx = dy - exp(y) * sum_c dy   (y = the log-probabilities)
__global__ void log_softmax_bwd_kernel(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ y,
                                       int64_t ldy, int64_t rows, int C, float* __restrict__ dx, int64_t lddx) {
    for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
        float s = 0.0f;
        for (int c = 0; c < C; ++c) s += dy[r * lddy + c];
        for (int c = 0; c < C; ++c) dx[r * lddx + c] = dy[r * lddy + c] - expf(y[r * ldy + c]) * s;
    }
}

// ------------------------------------------------------------------------------------------------
// torch.optim.Adam (amsgrad off, L2 weight decay added to the gradient) on a flat buffer.
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, int64_t n, float lr_over_bc1, float beta1, float beta2, float eps,
                            float weight_decay, float inv_sqrt_bc2, float grad_scale) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float pi = p[i];
        const float gi = fmaf(weight_decay, pi, g[i] * grad_scale);
        const float mi = m[i] + (gi - m[i]) * (1.0f - beta1);                // exp_avg.lerp_(grad, 1 - beta1)
        const float vi = fmaf(1.0f - beta2, gi * gi, v[i] * beta2);          // exp_avg_sq.mul_(b2).addcmul_(g, g, 1-b2)
        const float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;
        m[i] = mi;
        v[i] = vi;
        p[i] = pi - lr_over_bc1 * (mi / denom);
    }
}

// The same update with the learning rate and the step count in DEVICE memory, so that a captured CUDA graph replays
// with the current values: *step is incremented by a one-thread kernel first, then every thread derives the bias
// corrections from it (double precision, like the host variant).
__global__ void adam_step_increment_kernel(int64_t* step) { *step += 1; }

__global__ void adam_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                float* __restrict__ v, int64_t n, const float* __restrict__ lr_ptr,
                                const int64_t* __restrict__ step_ptr, float beta1, float beta2, float eps,
                                float weight_decay, float grad_scale) {
    const double step = (double)*step_ptr;
    const double bc1 = 1.0 - pow((double)beta1, step), bc2 = 1.0 - pow((double)beta2, step);
    const float lr_over_bc1 = (float)((double)*lr_ptr / bc1), inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float pi = p[i];
        const float gi = fmaf(weight_decay, pi, g[i] * grad_scale);
        const float mi = m[i] + (gi - m[i]) * (1.0f - beta1);
        const float vi = fmaf(1.0f - beta2, gi * gi, v[i] * beta2);
        const float denom = sqrtf(vi) * inv_sqrt_bc2 + eps;
        m[i] = mi;
        v[i] = vi;
        p[i] = pi - lr_over_bc1 * (mi / denom);
    }
}

// ------------------------------------------------------------------------------------------------
// Evaluation metrics of pcdseg.py:72-83: arg-max label per point, per-class intersection / prediction / target
// counts and the number of correct points -- one pass over the log-probabilities, block-local histograms.
// counts layout (int64): [0,C) intersection, [C,2C) predicted, [2C,3C) target, [3C] correct.
constexpr int METRIC_MAX_CLASSES = 64;
__global__ void __launch_bounds__(256)
seg_metrics_kernel(const float* __restrict__ x, int64_t ldx, const int64_t* __restrict__ target, int64_t rows, int C,
                   int64_t* __restrict__ pred_out, unsigned long long* __restrict__ counts) {
    __shared__ unsigned int h[3 * METRIC_MAX_CLASSES + 1];
    for (int i = threadIdx.x; i < 3 * C + 1; i += blockDim.x) h[i] = 0;
    __syncthreads();
    for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
        const float* __restrict__ xr = x + r * ldx;
        float m = xr[0];
        int am = 0;
        for (int c = 1; c < C; ++c) {
            const float v = xr[c];
            if (v > m) { m = v; am = c; }        // first maximum, like torch.argmax on CPU
        }
        if (pred_out) pred_out[r] = am;
        const int64_t t = target[r];
        atomicAdd(&h[C + am], 1u);
        if (t >= 0 && t < C) atomicAdd(&h[2 * C + (int)t], 1u);
        if (t == am) {
            atomicAdd(&h[am], 1u);
            atomicAdd(&h[3 * C], 1u);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 3 * C + 1; i += blockDim.x)
        if (h[i]) atomicAdd(&counts[i], (unsigned long long)h[i]);
}

// One batch folded into the running totals exactly as the reference's Python loop does it (pcdseg.py:75-83):
// iou = 1 if U == 0 else I/U (double division, rounded to fp32 when added to the fp32 array), count += 1,
// accuracy list entry = correct / points (double).  state: ious fp32[C], count u32[C], acc_sum f64, batches i64.
__global__ void seg_metrics_accumulate_kernel(const unsigned long long* __restrict__ counts, int C, int64_t points,
                                              float* __restrict__ ious, unsigned int* __restrict__ count,
                                              double* __restrict__ acc_sum, int64_t* __restrict__ batches) {
    const int c = threadIdx.x;
    if (c < C) {
        const unsigned long long I = counts[c], U = counts[C + c] + counts[2 * C + c] - I;
        const double iou = U == 0 ? 1.0 : (double)I / (double)U;
        ious[c] = ious[c] + (float)iou;
        count[c] += 1;
    }
    if (c == 0) {
        *acc_sum += (double)counts[3 * C] / (double)points;
        *batches += 1;
    }
}

static inline unsigned ew_blocks(int64_t total, int threads) {
    const int64_t want = ceil_div(total, threads);
    const int64_t cap = (int64_t)sm_count() * 16;
    return (unsigned)(want < 1 ? 1 : (want > cap ? cap : want));
}

}  // namespace pn

using namespace pn;

PN_EXPORT int pn_bn_stats_f32(const float* y, int64_t ldy, int64_t rows, int C, double* sum, double* sumsq,
                              pn_stream_t stream) {
    PN_REQUIRE(y && sum && sumsq, PN_ERR_BAD_ARG, "pn_bn_stats_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && ldy >= C, PN_ERR_BAD_ARG, "pn_bn_stats_f32: bad shape");
    dim3 grid;
    int64_t rpb;
    stats_grid(rows, C, &grid, &rpb);
    col_stats_kernel<0><<<grid, 32 * ST_LANES, 0, (cudaStream_t)stream>>>(y, ldy, rows, C, rpb, nullptr, 0, nullptr, 1, nullptr,
                                                                          nullptr, nullptr, nullptr, 0, sum, sumsq);
    return finish_launch("pn_bn_stats_f32");
}

PN_EXPORT int pn_bn_finalize_f32(const double* sum, const double* sumsq, int64_t n, int C, const float* gamma,
                                 const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                                 int64_t* num_batches_tracked, float* scale, float* shift, float* mean, float* invstd,
                                 pn_stream_t stream) {
    PN_REQUIRE(sum && sumsq && scale && shift && mean && invstd, PN_ERR_BAD_ARG, "pn_bn_finalize_f32: null pointer");
    PN_REQUIRE(n > 0 && C > 0, PN_ERR_BAD_ARG, "pn_bn_finalize_f32: bad shape");
    bn_finalize_kernel<<<(unsigned)ceil_div(C, 128), 128, 0, (cudaStream_t)stream>>>(
        sum, sumsq, n, C, gamma, beta, eps, momentum, running_mean, running_var, num_batches_tracked, scale, shift, mean, invstd);
    return finish_launch("pn_bn_finalize_f32");
}

PN_EXPORT int pn_bn_act_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* scale, const float* shift,
                            int relu, float* z, int64_t ldz, pn_stream_t stream) {
    PN_REQUIRE(y && scale && shift && z, PN_ERR_BAD_ARG, "pn_bn_act_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && ldy >= C && ldz >= C, PN_ERR_BAD_ARG, "pn_bn_act_f32: bad shape");
    bn_act_kernel<<<ew_blocks(rows * C, 256), 256, 0, (cudaStream_t)stream>>>(y, ldy, rows, C, scale, shift, relu, z, ldz);
    return finish_launch("pn_bn_act_f32");
}

PN_EXPORT int pn_bn_act_max_f32(const float* y, int64_t ldy, int64_t groups, int K, int C, const float* scale,
                                const float* shift, int relu, float* out, int64_t ldo, int32_t* argmax,
                                pn_stream_t stream) {
    PN_REQUIRE(y && scale && shift && out && argmax, PN_ERR_BAD_ARG, "pn_bn_act_max_f32: null pointer");
    PN_REQUIRE(groups > 0 && K > 0 && C > 0 && ldy >= C && ldo >= C, PN_ERR_BAD_ARG, "pn_bn_act_max_f32: bad shape");
    if (K >= 256 && groups <= 65535) {
        bn_act_max_tall_kernel<<<dim3((unsigned)ceil_div(C, 32), (unsigned)groups), 256, 0, (cudaStream_t)stream>>>(y, ldy, K, C, scale, shift,
                                                                                                              relu, out, ldo, argmax);
    } else {
        bn_act_max_kernel<<<ew_blocks(groups * C, 128), 128, 0, (cudaStream_t)stream>>>(y, ldy, groups, K, C, scale, shift, relu, out,
                                                                                       ldo, argmax);
    }
    return finish_launch("pn_bn_act_max_f32");
}

PN_EXPORT int pn_bn_bwd_stats_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* dz, int64_t lddz,
                                  const int32_t* argmax, int K, const float* scale, const float* shift,
                                  const float* mean, const float* invstd, int relu, double* s1, double* s2,
                                  pn_stream_t stream) {
    PN_REQUIRE(y && dz && scale && shift && mean && invstd && s1 && s2, PN_ERR_BAD_ARG, "pn_bn_bwd_stats_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && ldy >= C && lddz >= C, PN_ERR_BAD_ARG, "pn_bn_bwd_stats_f32: bad shape");
    PN_REQUIRE(!argmax || (K > 0 && rows % K == 0), PN_ERR_BAD_ARG, "pn_bn_bwd_stats_f32: rows must be a multiple of K");
    dim3 grid;
    int64_t rpb;
    stats_grid(rows, C, &grid, &rpb);
    cudaStream_t st = (cudaStream_t)stream;
    if (argmax)
        col_stats_kernel<2><<<grid, 32 * ST_LANES, 0, st>>>(y, ldy, rows, C, rpb, dz, lddz, argmax, K, scale, shift, mean, invstd,
                                                            relu, s1, s2);
    else
        col_stats_kernel<1><<<grid, 32 * ST_LANES, 0, st>>>(y, ldy, rows, C, rpb, dz, lddz, nullptr, 1, scale, shift, mean, invstd,
                                                            relu, s1, s2);
    return finish_launch("pn_bn_bwd_stats_f32");
}

PN_EXPORT int pn_bn_bwd_apply_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* dz, int64_t lddz,
                                  const int32_t* argmax, int K, const float* scale, const float* shift,
                                  const float* mean, const float* invstd, int relu, const double* s1, const double* s2,
                                  float* dy, int64_t lddy, float* dgamma, float* dbeta, pn_stream_t stream) {
    PN_REQUIRE(y && dz && scale && shift && mean && invstd && s1 && s2 && dy, PN_ERR_BAD_ARG, "pn_bn_bwd_apply_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && ldy >= C && lddz >= C && lddy >= C, PN_ERR_BAD_ARG, "pn_bn_bwd_apply_f32: bad shape");
    PN_REQUIRE(!argmax || (K > 0 && rows % K == 0), PN_ERR_BAD_ARG, "pn_bn_bwd_apply_f32: rows must be a multiple of K");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned blocks = ew_blocks(rows * C, 256);
    if (argmax)
        bn_bwd_apply_kernel<2><<<blocks, 256, 0, st>>>(y, ldy, rows, C, dz, lddz, argmax, K, scale, shift, mean, invstd, relu, s1, s2,
                                                       dy, lddy, dgamma, dbeta);
    else
        bn_bwd_apply_kernel<1><<<blocks, 256, 0, st>>>(y, ldy, rows, C, dz, lddz, nullptr, 1, scale, shift, mean, invstd, relu, s1,
                                                       s2, dy, lddy, dgamma, dbeta);
    return finish_launch("pn_bn_bwd_apply_f32");
}

PN_EXPORT int pn_bn_eval_bwd_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* dz, int64_t lddz,
                                 const int32_t* argmax, int K, const float* scale, const float* shift, const float* mean,
                                 const float* invstd, int relu, double* s1, double* s2, float* dy, int64_t lddy,
                                 float* dgamma, float* dbeta, pn_stream_t stream) {
    PN_REQUIRE(y && dz && scale && shift && mean && invstd && s1 && s2 && dy, PN_ERR_BAD_ARG, "pn_bn_eval_bwd_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && ldy >= C && lddz >= C && lddy >= C, PN_ERR_BAD_ARG, "pn_bn_eval_bwd_f32: bad shape");
    PN_REQUIRE(!argmax || (K > 0 && rows % K == 0), PN_ERR_BAD_ARG, "pn_bn_eval_bwd_f32: rows must be a multiple of K");
    dim3 grid;
    int64_t rpb;
    stats_grid(rows, C, &grid, &rpb);
    cudaStream_t st = (cudaStream_t)stream;
    if (argmax)
        bn_eval_bwd_kernel<true><<<grid, 32 * ST_LANES, 0, st>>>(y, ldy, rows, C, rpb, dz, lddz, argmax, K, scale, shift, mean,
                                                                invstd, relu, s1, s2, dy, lddy);
    else
        bn_eval_bwd_kernel<false><<<grid, 32 * ST_LANES, 0, st>>>(y, ldy, rows, C, rpb, dz, lddz, nullptr, 1, scale, shift, mean,
                                                                 invstd, relu, s1, s2, dy, lddy);
    if (dgamma || dbeta) bn_eval_bwd_finalize_kernel<<<(unsigned)ceil_div(C, 128), 128, 0, st>>>(s1, s2, C, dgamma, dbeta);
    return finish_launch("pn_bn_eval_bwd_f32");
}

PN_EXPORT int pn_grad_weight_f32(const float* dy, int64_t lddy, const float* x, int64_t ldx, int64_t rows, int cout,
                                 int cin, float* dw, int64_t lddw, float* db, pn_stream_t stream) {
    PN_REQUIRE(dy && x && dw, PN_ERR_BAD_ARG, "pn_grad_weight_f32: null pointer");
    PN_REQUIRE(rows > 0 && cout > 0 && cin > 0 && lddy >= cout && ldx >= cin && lddw >= cin, PN_ERR_BAD_ARG,
               "pn_grad_weight_f32: bad shape");
    int vec_ok = 0;
    if (((uintptr_t)dy % 16 == 0) && (lddy % 4 == 0)) vec_ok |= 1;
    if (((uintptr_t)x % 16 == 0) && (ldx % 4 == 0)) vec_ok |= 2;
    // (A 128 x 128 tile with 8 x 8 register tiles measured SLOWER on B200 -- 73 vs 49 us for 128 x 128 over 64 k rows: two
    // resident CTAs cannot hide the global-load latency of a BK = 8 step -- so the 64 x 64 tile is used throughout; the
    // fast path for wide layers is the tensor-core kernel pn_grad_weight_bf16x3.)
    const bool wide = false;
    const int BM = wide ? 128 : 64, BN = BM, BK = wide ? 8 : 16;
    const int64_t tiles = ceil_div(cout, BM) * ceil_div(cin, BN);
    int64_t splits = ceil_div((int64_t)sm_count() * (wide ? 2 : 4), tiles);
    int64_t rps = ceil_div(ceil_div(rows, splits), BK) * BK;
    if (rps < 64) rps = 64;
    splits = ceil_div(rows, rps);
    PN_REQUIRE(splits <= 65535, PN_ERR_UNSUPPORTED, "pn_grad_weight_f32: too many row splits");
    dim3 grid((unsigned)ceil_div(cout, BM), (unsigned)ceil_div(cin, BN), (unsigned)splits);
    if (wide)
        grad_weight_kernel<128, 128, 8, 8, 8><<<grid, 256, 0, (cudaStream_t)stream>>>(dy, lddy, x, ldx, rows, rps, cout, cin, dw, lddw,
                                                                                     db, vec_ok);
    else
        grad_weight_kernel<64, 64, 16, 4, 4><<<grid, 256, 0, (cudaStream_t)stream>>>(dy, lddy, x, ldx, rows, rps, cout, cin, dw, lddw,
                                                                                    db, vec_ok);
    return finish_launch("pn_grad_weight_f32");
}

PN_EXPORT int pn_transpose_f32(const float* in, int rows, int cols, float* out, pn_stream_t stream) {
    PN_REQUIRE(in && out && rows > 0 && cols > 0, PN_ERR_BAD_ARG, "pn_transpose_f32: bad arguments");
    dim3 grid((unsigned)ceil_div(cols, 32), (unsigned)ceil_div(rows, 32));
    transpose_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(in, rows, cols, out);
    return finish_launch("pn_transpose_f32");
}

PN_EXPORT int pn_group_bwd_f32(const float* dgrouped, int64_t ldg, int col0, int D, const int64_t* idx, int B, int N,
                               int S, int K, float* dfeat, pn_stream_t stream) {
    PN_REQUIRE(dgrouped && idx && dfeat, PN_ERR_BAD_ARG, "pn_group_bwd_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && S > 0 && K > 0 && D > 0 && col0 >= 0 && ldg >= col0 + D, PN_ERR_BAD_ARG,
               "pn_group_bwd_f32: bad shape");
    const int64_t total = (int64_t)B * S * K * D;
    group_bwd_kernel<<<ew_blocks(total, 256), 256, 0, (cudaStream_t)stream>>>(dgrouped, ldg, col0, D, idx, N, (int64_t)S * K, total,
                                                                             dfeat);
    return finish_launch("pn_group_bwd_f32");
}

PN_EXPORT int pn_three_interpolate_bwd_f32(const float* dx, int64_t ldx, int D1, int D2, const int64_t* idx,
                                           const float* weight, int B, int N, int S, float* dpoints1, float* dpoints2,
                                           pn_stream_t stream) {
    PN_REQUIRE(dx && idx && weight && dpoints2 && (D1 == 0 || dpoints1), PN_ERR_BAD_ARG, "pn_three_interpolate_bwd_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && S > 0 && D1 >= 0 && D2 > 0 && ldx >= D1 + D2, PN_ERR_BAD_ARG,
               "pn_three_interpolate_bwd_f32: bad shape");
    const int64_t total = (int64_t)B * N * (D1 + D2);
    three_interpolate_bwd_kernel<<<ew_blocks(total, 256), 256, 0, (cudaStream_t)stream>>>(dx, ldx, D1, D2, idx, weight, N, S, total,
                                                                                         dpoints1, dpoints2);
    return finish_launch("pn_three_interpolate_bwd_f32");
}

PN_EXPORT int pn_group_bwd_xyz_f32(const float* dgrouped, int64_t ldg, int col0, const int64_t* idx, int B, int N, int S, int K,
                                   float* dxyz, float* dnew_xyz, pn_stream_t stream) {
    PN_REQUIRE(dgrouped && idx && dxyz, PN_ERR_BAD_ARG, "pn_group_bwd_xyz_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && S > 0 && K > 0 && col0 >= 0 && ldg >= col0 + 3, PN_ERR_BAD_ARG, "pn_group_bwd_xyz_f32: bad shape");
    const int64_t groups = (int64_t)B * S;
    group_bwd_xyz_kernel<<<ew_blocks(groups * 32, 256), 256, 0, (cudaStream_t)stream>>>(dgrouped, ldg, col0, idx, N, S, K, groups,
                                                                                       dxyz, dnew_xyz);
    return finish_launch("pn_group_bwd_xyz_f32");
}

PN_EXPORT int pn_three_interpolate_bwd_xyz_f32(const float* dx, int64_t ldx, int D1, int D2, const int64_t* idx,
                                               const float* weight, const float* points2, int64_t p2B, int64_t p2S, int64_t p2C,
                                               const float* xyz1, int64_t aB, int64_t aN, int64_t aC, const float* xyz2,
                                               int64_t bB, int64_t bS, int64_t bC, int B, int N, int S, float* dpoints1,
                                               float* dpoints2, float* dxyz1, float* dxyz2, pn_stream_t stream) {
    PN_REQUIRE(dx && idx && weight && points2 && xyz1 && xyz2 && dpoints2 && dxyz1 && dxyz2 && (D1 == 0 || dpoints1),
               PN_ERR_BAD_ARG, "pn_three_interpolate_bwd_xyz_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && D1 >= 0 && D2 > 0 && ldx >= D1 + D2, PN_ERR_BAD_ARG, "pn_three_interpolate_bwd_xyz_f32: bad shape");
    // S == 1 is the broadcast of pointnet_util.py:292-293, whose weights (1, 0, 0) do not come from distances; S == 2 has no
    // 3-NN forward (pn_three_nn_f32 needs S >= 3)
    PN_REQUIRE(S >= 3, PN_ERR_BAD_ARG, "pn_three_interpolate_bwd_xyz_f32: need S >= 3 (got %d)", S);
    const int64_t rows = (int64_t)B * N;
    const bool vec = D1 % 4 == 0 && D2 % 4 == 0 && ldx % 4 == 0 && p2C == 1 && p2S % 4 == 0 && p2B % 4 == 0 &&
                     ((uintptr_t)dx & 15) == 0 && ((uintptr_t)points2 & 15) == 0 && ((uintptr_t)dpoints2 & 15) == 0 &&
                     ((uintptr_t)dpoints1 & 15) == 0;
    const unsigned grid = (unsigned)ew_blocks(rows * 32, 256);
    if (vec)
        three_interpolate_bwd_xyz_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(
            dx, ldx, D1, D2, idx, weight, points2, p2B, p2S, p2C, xyz1, aB, aN, aC, xyz2, bB, bS, bC, N, S, rows, dpoints1, dpoints2,
            dxyz1, dxyz2);
    else
        three_interpolate_bwd_xyz_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(
            dx, ldx, D1, D2, idx, weight, points2, p2B, p2S, p2C, xyz1, aB, aN, aC, xyz2, bB, bS, bC, N, S, rows, dpoints1, dpoints2,
            dxyz1, dxyz2);
    return finish_launch("pn_three_interpolate_bwd_xyz_f32");
}

PN_EXPORT int pn_dropout_f32(const float* x, int64_t ldx, int64_t rows, int C, float p, const uint64_t* seed_offset,
                             const uint8_t* mask_in, uint8_t* mask_out, float* y, int64_t ldy, pn_stream_t stream) {
    PN_REQUIRE(x && y && (mask_in || seed_offset), PN_ERR_BAD_ARG, "pn_dropout_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && ldx >= C && ldy >= C && p >= 0.0f && p < 1.0f, PN_ERR_BAD_ARG, "pn_dropout_f32: bad arguments");
    dropout_kernel<<<ew_blocks((rows * C + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, rows, C, p, seed_offset, mask_in,
                                                                                        mask_out, y, ldy);
    return finish_launch("pn_dropout_f32");
}

PN_EXPORT int pn_cross_entropy_f32(const float* x, int64_t ldx, const int64_t* target, int64_t rows, int C,
                                   double* loss_sum, float* loss, float* dx, int64_t lddx, float grad_scale,
                                   pn_stream_t stream) {
    PN_REQUIRE(x && target && loss_sum && loss, PN_ERR_BAD_ARG, "pn_cross_entropy_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && ldx >= C && (!dx || lddx >= C), PN_ERR_BAD_ARG, "pn_cross_entropy_f32: bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(loss_sum, 0, 2 * sizeof(double), st);
    if (e != cudaSuccess) {
        set_error("pn_cross_entropy_f32: %s", cudaGetErrorString(e));
        return (int)e;
    }
    label_count_kernel<<<ew_blocks(rows, 256), 256, 0, st>>>(target, rows, loss_sum + 1);
    cross_entropy_kernel<<<ew_blocks(rows, 256), 256, 0, st>>>(x, ldx, target, rows, C, loss_sum, loss_sum + 1, dx, lddx, grad_scale);
    loss_finalize_kernel<<<1, 1, 0, st>>>(loss_sum, loss_sum + 1, loss);
    return finish_launch("pn_cross_entropy_f32");
}

PN_EXPORT int pn_log_softmax_bwd_f32(const float* dy, int64_t lddy, const float* y, int64_t ldy, int64_t rows, int C,
                                     float* dx, int64_t lddx, pn_stream_t stream) {
    PN_REQUIRE(dy && y && dx, PN_ERR_BAD_ARG, "pn_log_softmax_bwd_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && lddy >= C && ldy >= C && lddx >= C, PN_ERR_BAD_ARG, "pn_log_softmax_bwd_f32: bad shape");
    log_softmax_bwd_kernel<<<ew_blocks(rows, 256), 256, 0, (cudaStream_t)stream>>>(dy, lddy, y, ldy, rows, C, dx, lddx);
    return finish_launch("pn_log_softmax_bwd_f32");
}

PN_EXPORT int pn_adam_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                          float beta1, float beta2, float eps, float weight_decay, int64_t step, float grad_scale,
                          pn_stream_t stream) {
    PN_REQUIRE(param && grad && exp_avg && exp_avg_sq, PN_ERR_BAD_ARG, "pn_adam_f32: null pointer");
    PN_REQUIRE(n > 0 && step > 0, PN_ERR_BAD_ARG, "pn_adam_f32: n and step must be positive");
    // bias corrections in double like torch (python floats), then the per-element arithmetic in fp32
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    adam_kernel<<<ew_blocks(n, 256), 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, n, (float)((double)lr / bc1),
                                                                    beta1, beta2, eps, weight_decay, (float)(1.0 / sqrt(bc2)),
                                                                    grad_scale);
    return finish_launch("pn_adam_f32");
}

PN_EXPORT int pn_adam_dev_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                              const float* lr, int64_t* step, float beta1, float beta2, float eps, float weight_decay,
                              float grad_scale, pn_stream_t stream) {
    PN_REQUIRE(param && grad && exp_avg && exp_avg_sq && lr && step, PN_ERR_BAD_ARG, "pn_adam_dev_f32: null pointer");
    PN_REQUIRE(n > 0, PN_ERR_BAD_ARG, "pn_adam_dev_f32: n must be positive");
    cudaStream_t st = (cudaStream_t)stream;
    adam_step_increment_kernel<<<1, 1, 0, st>>>(step);
    adam_dev_kernel<<<ew_blocks(n, 256), 256, 0, st>>>(param, grad, exp_avg, exp_avg_sq, n, lr, step, beta1, beta2, eps, weight_decay,
                                                      grad_scale);
    return finish_launch("pn_adam_dev_f32");
}

PN_EXPORT int pn_seg_metrics_f32(const float* logp, int64_t ldx, const int64_t* target, int64_t rows, int C,
                                 int64_t* pred, int64_t* counts, pn_stream_t stream) {
    PN_REQUIRE(logp && target && counts, PN_ERR_BAD_ARG, "pn_seg_metrics_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && C <= METRIC_MAX_CLASSES && ldx >= C, PN_ERR_BAD_ARG, "pn_seg_metrics_f32: bad shape (C <= 64)");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(counts, 0, sizeof(int64_t) * (3 * C + 1), st);
    if (e != cudaSuccess) {
        set_error("pn_seg_metrics_f32: %s", cudaGetErrorString(e));
        return (int)e;
    }
    seg_metrics_kernel<<<ew_blocks(rows, 256), 256, 0, st>>>(logp, ldx, target, rows, C, pred, (unsigned long long*)counts);
    return finish_launch("pn_seg_metrics_f32");
}

PN_EXPORT int pn_seg_metrics_accumulate(const int64_t* counts, int C, int64_t points, float* ious, uint32_t* count,
                                        double* acc_sum, int64_t* batches, pn_stream_t stream) {
    PN_REQUIRE(counts && ious && count && acc_sum && batches, PN_ERR_BAD_ARG, "pn_seg_metrics_accumulate: null pointer");
    PN_REQUIRE(C > 0 && C <= METRIC_MAX_CLASSES && points > 0, PN_ERR_BAD_ARG, "pn_seg_metrics_accumulate: bad shape");
    seg_metrics_accumulate_kernel<<<1, METRIC_MAX_CLASSES, 0, (cudaStream_t)stream>>>((const unsigned long long*)counts, C, points, ious,
                                                                                     count, acc_sum, batches);
    return finish_launch("pn_seg_metrics_accumulate");
}

// ------------------------------------------------------------------------------------------------
// Row f-4 helpers.
// chamfer_batch / chamfer_non_batch (model/chamfer.py:7-53): sum over b, n of min_m ||p1[b,n] - p2[b,m]||_2, divided by B.
// One thread per p1 point, p2 staged through shared memory in tiles; the minimum is taken over squared distances
// (sqrt is monotonic) and the root drawn once per point; block sums in fp64.  ARGMIN: also the index of the nearest p2
// point (the first of equal minima, like torch's min(dim) on the CPU) for the backward pass.
namespace pn {
constexpr int CH_TILE = 256, CH_MAXD = 8;
// DET: total is a [gridDim.y * gridDim.x] array of block partials, written.
template <bool ARGMIN, bool DET = false>
__global__ void __launch_bounds__(CH_TILE)
chamfer_kernel(const float* __restrict__ p1, int64_t aB, int64_t aN, int64_t aC, const float* __restrict__ p2, int64_t bB,
               int64_t bN, int64_t bC, int N, int M, int D, float* __restrict__ per_point, double* __restrict__ total,
               int32_t* __restrict__ argmin) {
    __shared__ float tile[CH_TILE][CH_MAXD];
    __shared__ double red[CH_TILE / 32];
    const int b = blockIdx.y;
    const int n = blockIdx.x * CH_TILE + threadIdx.x;
    float q[CH_MAXD];
#pragma unroll
    for (int c = 0; c < CH_MAXD; ++c) q[c] = (n < N && c < D) ? p1[b * aB + (int64_t)n * aN + c * aC] : 0.0f;
    float best = CUDART_INF_F;
    int best_m = 0;
    for (int m0 = 0; m0 < M; m0 += CH_TILE) {
        const int m = m0 + threadIdx.x;
#pragma unroll
        for (int c = 0; c < CH_MAXD; ++c) tile[threadIdx.x][c] = (m < M && c < D) ? p2[b * bB + (int64_t)m * bN + c * bC] : 0.0f;
        __syncthreads();
        const int lim = min(CH_TILE, M - m0);
        for (int j = 0; j < lim; ++j) {
            float d = 0.0f;
#pragma unroll
            for (int c = 0; c < CH_MAXD; ++c) {
                const float t = q[c] - tile[j][c];
                d = fmaf(t, t, d);
            }
            if constexpr (ARGMIN) {
                if (d < best) {          // strict: the first minimum stays
                    best = d;
                    best_m = m0 + j;
                }
            } else {
                best = fminf(best, d);
            }
        }
        __syncthreads();
    }
    const float dist = n < N ? sqrtf(best) : 0.0f;
    if (n < N && per_point) per_point[(int64_t)b * N + n] = dist;
    if constexpr (ARGMIN) {
        if (n < N) argmin[(int64_t)b * N + n] = best_m;
    }
    double s = (double)dist;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < CH_TILE / 32; ++i) t += red[i];
        if (DET) total[blockIdx.y * gridDim.x + blockIdx.x] = t;
        else atomicAdd(total, t);
    }
}

// SemKITTI_2_Common.__call__ (data_utils/kitti_utils.py:97-110): common[..., j] = max(logits[..., src0[j]], logits[..., src1[j]])
__global__ void class_merge_kernel(const float* __restrict__ x, int64_t ldx, int64_t rows, int n_out, const int* __restrict__ src0,
                                   const int* __restrict__ src1, float* __restrict__ y) {
    const int64_t total = rows * n_out;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int j = (int)(e % n_out);
        const int64_t r = e / n_out;
        y[e] = fmaxf(x[r * ldx + src0[j]], x[r * ldx + src1[j]]);
    }
}

// Backward of chamfer_batch / chamfer_non_batch: per p1 point, r = p1[n] - p2[a(n)] with the nearest p2 point a(n) of the
// forward, d = ||r|| in the forward's rounding sequence, c = g*scale / d (0 where d == 0, as torch's norm backward);
// dp1[n] = c*r (written), dp2[a(n)] -= c*r (fp32 atomics; DET: dp2 is a [B*N, D] workspace of the terms -c*r, written).
template <bool DET = false>
__global__ void chamfer_bwd_kernel(const float* __restrict__ p1, int64_t aB, int64_t aN, int64_t aC, const float* __restrict__ p2,
                                   int64_t bB, int64_t bN, int64_t bC, int N, int M, int D, int64_t total,
                                   const int32_t* __restrict__ argmin, const float* __restrict__ g, float scale,
                                   float* __restrict__ dp1, float* __restrict__ dp2) {
    const float gs = *g * scale;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = i / N, n = i % N;
        const int a = argmin[i];
        float t[CH_MAXD];
        float d = 0.0f;
#pragma unroll
        for (int c = 0; c < CH_MAXD; ++c) {
            t[c] = c < D ? p1[b * aB + n * aN + c * aC] - p2[b * bB + (int64_t)a * bN + c * bC] : 0.0f;
            d = fmaf(t[c], t[c], d);
        }
        const float dist = sqrtf(d);
        const float coef = dist > 0.0f ? gs / dist : 0.0f;
#pragma unroll
        for (int c = 0; c < CH_MAXD; ++c) {
            if (c >= D) break;
            if (dp1) dp1[i * D + c] = coef * t[c];
            if (DET) dp2[i * D + c] = -(coef * t[c]);
            else if (dp2) atomicAdd(dp2 + (b * M + a) * D + c, -(coef * t[c]));
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Backward of square_distance (model/pointnet_util.py:19-40), dist = -2 src dst^T + |src|^2 + |dst|^2, g = dL/ddist [B,N,M]:
//   dsrc[n] = 2 (sum_m g[n,m]) src[n] - 2 sum_m g[n,m] dst[m],   ddst[m] = 2 (sum_n g[n,m]) dst[m] - 2 sum_n g[n,m] src[n].
// HBM-bound: g is read exactly once.  A CTA owns SDB_ROWS rows (SDB_RT per warp) and a chunk of columns, which its warps
// stream in steps of 128 columns (a float4 per lane and row).  Row sums (sum g, sum g*dst) stay in registers for the whole
// chunk; column sums (sum g, sum g*src) of a step are summed over the warp's rows in registers, then over the CTA's warps
// in shared memory (double-buffered: one barrier per step), and leave as ONE vector red.global.add per column and CTA.
// Both land in a small fp32 workspace, rows [B,N,4] and columns [B,M,4]; sqdist_bwd_finish_kernel forms the gradients
// from it, with the reference's two terms kept apart and subtracted last (as torch's matmul + sum backward add them).
constexpr int SDB_WARPS = 8, SDB_RT = 8, SDB_ROWS = SDB_WARPS * SDB_RT, SDB_STEP = 128;

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// DET: rws / cws are [gridDim.x, B, N, 4] / [gridDim.y, B, M, 4]: each CTA stores its sums in the slot of its column chunk /
// row tile instead of adding them (sqdist_partials_sum_kernel adds the slots in order).
template <bool VEC, bool ROWS, bool COLS, bool DET = false>
__global__ void __launch_bounds__(SDB_WARPS * 32, 2)
sqdist_bwd_kernel(const float* __restrict__ g, int64_t gB, int64_t gN, const float* __restrict__ src, int64_t aB, int64_t aN,
                  int64_t aC, const float* __restrict__ dst, int64_t bB, int64_t bN, int64_t bC, int N, int M, int chunk,
                  float* __restrict__ rws, float* __restrict__ cws) {
    __shared__ float4 part[COLS ? 2 : 1][SDB_WARPS][SDB_STEP];
    const int b = blockIdx.z, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r0 = blockIdx.y * SDB_ROWS + warp * SDB_RT;
    const int m_begin = blockIdx.x * chunk, m_end = min(M, m_begin + chunk);
    const float* __restrict__ gb = g + (int64_t)b * gB;
    float sx[SDB_RT], sy[SDB_RT], sz[SDB_RT];                 // the warp's src rows (column sums only)
    float rs[SDB_RT], rx[SDB_RT], ry[SDB_RT], rz[SDB_RT];     // row sums: sum g, sum g*dst
#pragma unroll
    for (int r = 0; r < SDB_RT; ++r) {
        const int n = r0 + r;
        const float* s = src + (int64_t)b * aB + (int64_t)n * aN;
        sx[r] = COLS && n < N ? s[0] : 0.0f;
        sy[r] = COLS && n < N ? s[aC] : 0.0f;
        sz[r] = COLS && n < N ? s[2 * aC] : 0.0f;
        rs[r] = rx[r] = ry[r] = rz[r] = 0.0f;
    }
    int buf = 0;
    for (int c0 = m_begin; c0 < m_end; c0 += SDB_STEP) {
        const int m = c0 + lane * 4;
        float dx[4], dy[4], dz[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float* q = dst + (int64_t)b * bB + (int64_t)(m + j) * bN;
            const bool ok = ROWS && m + j < m_end;
            dx[j] = ok ? q[0] : 0.0f;
            dy[j] = ok ? q[bC] : 0.0f;
            dz[j] = ok ? q[2 * bC] : 0.0f;
        }
        float v[SDB_RT][4];
#pragma unroll
        for (int r = 0; r < SDB_RT; ++r) {
            const int n = r0 + r;
            const float* row = gb + (int64_t)n * gN + m;
            if (VEC && n < N && m + 3 < m_end) {
                const float4 t = __ldcs(reinterpret_cast<const float4*>(row));
                v[r][0] = t.x, v[r][1] = t.y, v[r][2] = t.z, v[r][3] = t.w;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) v[r][j] = n < N && m + j < m_end ? __ldcs(row + j) : 0.0f;
            }
        }
        float cs[4], cx[4], cy[4], cz[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) cs[j] = cx[j] = cy[j] = cz[j] = 0.0f;
#pragma unroll
        for (int r = 0; r < SDB_RT; ++r) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float e = v[r][j];
                if (ROWS) {
                    rs[r] += e;
                    rx[r] = fmaf(e, dx[j], rx[r]);
                    ry[r] = fmaf(e, dy[j], ry[r]);
                    rz[r] = fmaf(e, dz[j], rz[r]);
                }
                if (COLS) {
                    cs[j] += e;
                    cx[j] = fmaf(e, sx[r], cx[j]);
                    cy[j] = fmaf(e, sy[r], cy[j]);
                    cz[j] = fmaf(e, sz[r], cz[j]);
                }
            }
        }
        if (COLS) {
            // slot j*32 + lane holds column m + j: conflict-free stores here and loads below
#pragma unroll
            for (int j = 0; j < 4; ++j) part[buf][warp][j * 32 + lane] = make_float4(cs[j], cx[j], cy[j], cz[j]);
            __syncthreads();
            if (threadIdx.x < SDB_STEP) {
                const int col = c0 + (threadIdx.x & 31) * 4 + (threadIdx.x >> 5);
                float4 t = part[buf][0][threadIdx.x];
#pragma unroll
                for (int w = 1; w < SDB_WARPS; ++w) {
                    const float4 u = part[buf][w][threadIdx.x];
                    t.x += u.x, t.y += u.y, t.z += u.z, t.w += u.w;
                }
                if (col < m_end) {
                    if (DET) *reinterpret_cast<float4*>(cws + (((int64_t)blockIdx.y * gridDim.z + b) * M + col) * 4) = t;
                    else red_add_v4(cws + ((int64_t)b * M + col) * 4, t.x, t.y, t.z, t.w);
                }
            }
            buf ^= 1;   // the other buffer was last read before this step's barrier
        }
    }
    if (ROWS) {
#pragma unroll
        for (int r = 0; r < SDB_RT; ++r) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                rs[r] += __shfl_xor_sync(0xffffffffu, rs[r], o);
                rx[r] += __shfl_xor_sync(0xffffffffu, rx[r], o);
                ry[r] += __shfl_xor_sync(0xffffffffu, ry[r], o);
                rz[r] += __shfl_xor_sync(0xffffffffu, rz[r], o);
            }
            if (lane == r && r0 + r < N) {
                if (DET)
                    *reinterpret_cast<float4*>(rws + (((int64_t)blockIdx.x * gridDim.z + b) * N + r0 + r) * 4) =
                        make_float4(rs[r], rx[r], ry[r], rz[r]);
                else
                    red_add_v4(rws + ((int64_t)b * N + r0 + r) * 4, rs[r], rx[r], ry[r], rz[r]);
            }
        }
    }
}

// out[i] = sum_s part[s * n + i] (s ascending), over the n records of [slots, n] float4 partials.
__global__ void sqdist_partials_sum_kernel(const float4* __restrict__ part, int slots, int64_t n, float4* __restrict__ out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float4 t = part[i];
        for (int s = 1; s < slots; ++s) {
            const float4 u = part[s * n + i];
            t.x += u.x, t.y += u.y, t.z += u.z, t.w += u.w;
        }
        out[i] = t;
    }
}

// out[p] = 2 (sum e) x[p] - 2 (sum e*y) from the workspace records {sum e, sum e*y_x, sum e*y_y, sum e*y_z}, for the
// B*N src points (rws -> dsrc) then the B*M dst points (cws -> ddst); a NULL output is skipped.
__global__ void sqdist_bwd_finish_kernel(const float* __restrict__ src, int64_t aB, int64_t aN, int64_t aC,
                                         const float* __restrict__ dst, int64_t bB, int64_t bN, int64_t bC, int B, int N, int M,
                                         const float4* __restrict__ rws, const float4* __restrict__ cws, float* __restrict__ dsrc,
                                         float* __restrict__ ddst) {
    const int64_t nsrc = (int64_t)B * N, total = nsrc + (int64_t)B * M;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const bool is_src = i < nsrc;
        float* out = is_src ? dsrc : ddst;
        if (!out) continue;
        const int64_t j = is_src ? i : i - nsrc;
        const int P = is_src ? N : M;
        const int64_t b = j / P, p = j % P;
        const float* x = is_src ? src + b * aB + p * aN : dst + b * bB + p * bN;
        const int64_t xc = is_src ? aC : bC;
        const float4 w = is_src ? rws[j] : cws[j];
        const float s2 = 2.0f * w.x;
        out[j * 3 + 0] = __fsub_rn(__fmul_rn(s2, x[0]), 2.0f * w.y);
        out[j * 3 + 1] = __fsub_rn(__fmul_rn(s2, x[xc]), 2.0f * w.z);
        out[j * 3 + 2] = __fsub_rn(__fmul_rn(s2, x[2 * xc]), 2.0f * w.w);
    }
}
}  // namespace pn

PN_EXPORT int pn_chamfer_f32(const float* p1, int64_t aB, int64_t aN, int64_t aC, const float* p2, int64_t bB, int64_t bN,
                             int64_t bC, int B, int N, int M, int D, float* per_point, double* total, pn_stream_t stream) {
    PN_REQUIRE(p1 && p2 && total, PN_ERR_BAD_ARG, "pn_chamfer_f32: null pointer");
    PN_REQUIRE(B > 0 && B <= 65535 && N > 0 && M > 0 && D > 0 && D <= CH_MAXD, PN_ERR_BAD_ARG, "pn_chamfer_f32: bad sizes (D <= 8)");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(total, 0, sizeof(double), st);
    if (e != cudaSuccess) {
        set_error("pn_chamfer_f32: %s", cudaGetErrorString(e));
        return (int)e;
    }
    dim3 grid((unsigned)ceil_div(N, CH_TILE), (unsigned)B);
    chamfer_kernel<false><<<grid, CH_TILE, 0, st>>>(p1, aB, aN, aC, p2, bB, bN, bC, N, M, D, per_point, total, nullptr);
    return finish_launch("pn_chamfer_f32");
}

PN_EXPORT int pn_class_merge_f32(const float* x, int64_t ldx, int64_t rows, int n_in, int n_out, const int* src0,
                                 const int* src1, float* y, pn_stream_t stream) {
    PN_REQUIRE(x && src0 && src1 && y, PN_ERR_BAD_ARG, "pn_class_merge_f32: null pointer");
    PN_REQUIRE(rows > 0 && n_in > 0 && n_out > 0 && ldx >= n_in, PN_ERR_BAD_ARG, "pn_class_merge_f32: bad shape");
    class_merge_kernel<<<ew_blocks(rows * n_out, 256), 256, 0, (cudaStream_t)stream>>>(x, ldx, rows, n_out, src0, src1, y);
    return finish_launch("pn_class_merge_f32");
}

PN_EXPORT int pn_chamfer_argmin_f32(const float* p1, int64_t aB, int64_t aN, int64_t aC, const float* p2, int64_t bB, int64_t bN,
                                    int64_t bC, int B, int N, int M, int D, float* per_point, double* total, int32_t* argmin,
                                    pn_stream_t stream) {
    PN_REQUIRE(p1 && p2 && total && argmin, PN_ERR_BAD_ARG, "pn_chamfer_argmin_f32: null pointer");
    PN_REQUIRE(B > 0 && B <= 65535 && N > 0 && M > 0 && D > 0 && D <= CH_MAXD, PN_ERR_BAD_ARG,
               "pn_chamfer_argmin_f32: bad sizes (D <= 8)");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(total, 0, sizeof(double), st);
    if (e != cudaSuccess) {
        set_error("pn_chamfer_argmin_f32: %s", cudaGetErrorString(e));
        return (int)e;
    }
    dim3 grid((unsigned)ceil_div(N, CH_TILE), (unsigned)B);
    chamfer_kernel<true><<<grid, CH_TILE, 0, st>>>(p1, aB, aN, aC, p2, bB, bN, bC, N, M, D, per_point, total, argmin);
    return finish_launch("pn_chamfer_argmin_f32");
}

PN_EXPORT int pn_chamfer_bwd_f32(const float* p1, int64_t aB, int64_t aN, int64_t aC, const float* p2, int64_t bB, int64_t bN,
                                 int64_t bC, int B, int N, int M, int D, const int32_t* argmin, const float* g_total, float scale,
                                 float* dp1, float* dp2, pn_stream_t stream) {
    PN_REQUIRE(p1 && p2 && argmin && g_total && (dp1 || dp2), PN_ERR_BAD_ARG, "pn_chamfer_bwd_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && M > 0 && D > 0 && D <= CH_MAXD, PN_ERR_BAD_ARG, "pn_chamfer_bwd_f32: bad sizes (D <= 8)");
    const int64_t total = (int64_t)B * N;
    chamfer_bwd_kernel<<<ew_blocks(total, 256), 256, 0, (cudaStream_t)stream>>>(p1, aB, aN, aC, p2, bB, bN, bC, N, M, D, total,
                                                                               argmin, g_total, scale, dp1, dp2);
    return finish_launch("pn_chamfer_bwd_f32");
}

PN_EXPORT int pn_square_distance_bwd_f32(const float* g, int64_t gB, int64_t gN, const float* src, int64_t aB, int64_t aN,
                                         int64_t aC, const float* dst, int64_t bB, int64_t bN, int64_t bC, int B, int N, int M,
                                         float* workspace, float* dsrc, float* ddst, pn_stream_t stream) {
    PN_REQUIRE(g && src && dst && workspace && (dsrc || ddst), PN_ERR_BAD_ARG, "pn_square_distance_bwd_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && M > 0, PN_ERR_BAD_ARG, "pn_square_distance_bwd_f32: B, N, M must be positive");
    PN_REQUIRE(B <= 65535 && ceil_div(N, SDB_ROWS) <= 65535, PN_ERR_UNSUPPORTED,
               "pn_square_distance_bwd_f32: B <= 65535 and N <= %d", 65535 * SDB_ROWS);
    PN_REQUIRE(gB >= 0 && gN >= 0, PN_ERR_BAD_ARG, "pn_square_distance_bwd_f32: negative stride of g");
    PN_REQUIRE(((uintptr_t)workspace & 15) == 0, PN_ERR_BAD_ARG, "pn_square_distance_bwd_f32: workspace must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    float* rws = workspace;                       // [B,N,4]
    float* cws = workspace + (int64_t)B * N * 4;  // [B,M,4]
    cudaError_t e = cudaMemsetAsync(workspace, 0, sizeof(float) * 4 * ((size_t)B * N + (size_t)B * M), st);
    if (e != cudaSuccess) {
        set_error("pn_square_distance_bwd_f32: %s", cudaGetErrorString(e));
        return (int)e;
    }
    // columns per CTA: enough CTAs for four per SM where the shape allows, whole 128-column steps
    const int64_t row_tiles = ceil_div(N, SDB_ROWS) * B;
    const int64_t steps = ceil_div(M, SDB_STEP);
    int64_t chunks = ceil_div((int64_t)sm_count() * 4, row_tiles);
    if (chunks > steps) chunks = steps;
    if (chunks > 65535) chunks = 65535;
    const int chunk = (int)(ceil_div(steps, chunks) * SDB_STEP);
    dim3 grid((unsigned)ceil_div(M, chunk), (unsigned)ceil_div(N, SDB_ROWS), (unsigned)B);
    const bool vec = ((uintptr_t)g & 15) == 0 && gN % 4 == 0 && (B == 1 || gB % 4 == 0);
    const bool rows = dsrc != nullptr, cols = ddst != nullptr;
    auto kern = vec ? (rows ? (cols ? sqdist_bwd_kernel<true, true, true> : sqdist_bwd_kernel<true, true, false>)
                            : sqdist_bwd_kernel<true, false, true>)
                    : (rows ? (cols ? sqdist_bwd_kernel<false, true, true> : sqdist_bwd_kernel<false, true, false>)
                            : sqdist_bwd_kernel<false, false, true>);
    kern<<<grid, SDB_WARPS * 32, 0, st>>>(g, gB, gN, src, aB, aN, aC, dst, bB, bN, bC, N, M, chunk, rws, cws);
    sqdist_bwd_finish_kernel<<<ew_blocks((int64_t)B * (N + (int64_t)M), 256), 256, 0, st>>>(
        src, aB, aN, aC, dst, bB, bN, bC, B, N, M, reinterpret_cast<const float4*>(rws), reinterpret_cast<const float4*>(cws),
        dsrc, ddst);
    return finish_launch("pn_square_distance_bwd_f32");
}

// ------------------------------------------------------------------------------------------------
// Deterministic variants (torch.use_deterministic_algorithms): the same arithmetic as the entry points above, with every
// floating-point sum taken in an order fixed by the shapes and the SM count -- per-block / per-slab partials in a
// caller-provided workspace, added in block order, and scatter-adds pulled through the CSR of pn_csr_build (scatter.cu).
namespace pn {
static inline size_t bn_det_bytes(int64_t rows, int C) {
    dim3 grid;
    int64_t rpb;
    stats_grid(rows, C, &grid, &rpb);
    return sizeof(double) * 2 * (size_t)grid.x * (size_t)C;
}

static inline void grad_weight_f32_shape(int64_t rows, int cout, int cin, int64_t* splits, int64_t* rps) {
    const int64_t tiles = ceil_div(cout, 64) * ceil_div(cin, 64);
    int64_t sp = ceil_div((int64_t)sm_count() * 4, tiles);
    int64_t r = ceil_div(ceil_div(rows, sp), 16) * 16;
    if (r < 64) r = 64;
    *rps = r;
    *splits = ceil_div(rows, r);
}

int grad_weight_slab_sum(const float* ws, int64_t splits, int64_t bias_parts, int cout, int cin, float* dw, int64_t lddw, float* db,
                         cudaStream_t st);

static inline void sqdist_bwd_shape(int B, int N, int M, int* chunk, dim3* grid) {
    const int64_t row_tiles = ceil_div(N, SDB_ROWS) * B;
    const int64_t steps = ceil_div(M, SDB_STEP);
    int64_t chunks = ceil_div((int64_t)sm_count() * 4, row_tiles);
    if (chunks > steps) chunks = steps;
    if (chunks > 65535) chunks = 65535;
    *chunk = (int)(ceil_div(steps, chunks) * SDB_STEP);
    *grid = dim3((unsigned)ceil_div(M, *chunk), (unsigned)ceil_div(N, SDB_ROWS), (unsigned)B);
}
}  // namespace pn

PN_EXPORT size_t pn_bn_stats_workspace_bytes(int64_t rows, int C) {
    return rows > 0 && C > 0 ? bn_det_bytes(rows, C) : 0;
}

#define PN_DET_WS(name, need)                                                                                              \
    PN_REQUIRE(workspace, PN_ERR_BAD_ARG, name ": null workspace");                                                          \
    PN_REQUIRE(workspace_bytes >= (need), PN_ERR_BAD_ARG, name ": workspace of %zu bytes, need %zu", workspace_bytes,     \
               (size_t)(need));                                                                                              \
    PN_REQUIRE(((uintptr_t)workspace & 15) == 0, PN_ERR_BAD_ARG, name ": workspace must be 16-byte aligned")

PN_EXPORT int pn_bn_stats_det_f32(const float* y, int64_t ldy, int64_t rows, int C, double* sum, double* sumsq, void* workspace,
                                  size_t workspace_bytes, pn_stream_t stream) {
    PN_REQUIRE(y && sum && sumsq, PN_ERR_BAD_ARG, "pn_bn_stats_det_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && ldy >= C, PN_ERR_BAD_ARG, "pn_bn_stats_det_f32: bad shape");
    PN_DET_WS("pn_bn_stats_det_f32", bn_det_bytes(rows, C));
    dim3 grid;
    int64_t rpb;
    stats_grid(rows, C, &grid, &rpb);
    cudaStream_t st = (cudaStream_t)stream;
    double* part = static_cast<double*>(workspace);
    col_stats_kernel<0, true><<<grid, 32 * ST_LANES, 0, st>>>(y, ldy, rows, C, rpb, nullptr, 0, nullptr, 1, nullptr, nullptr, nullptr,
                                                               nullptr, 0, part, part + (int64_t)grid.x * C);
    col_partials_sum_kernel<<<(unsigned)ceil_div(C, 128), 128, 0, st>>>(part, (int)grid.x, C, sum, sumsq);
    return finish_launch("pn_bn_stats_det_f32");
}

PN_EXPORT int pn_bn_bwd_stats_det_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* dz, int64_t lddz,
                                      const int32_t* argmax, int K, const float* scale, const float* shift, const float* mean,
                                      const float* invstd, int relu, double* s1, double* s2, void* workspace,
                                      size_t workspace_bytes, pn_stream_t stream) {
    PN_REQUIRE(y && dz && scale && shift && mean && invstd && s1 && s2, PN_ERR_BAD_ARG, "pn_bn_bwd_stats_det_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && ldy >= C && lddz >= C, PN_ERR_BAD_ARG, "pn_bn_bwd_stats_det_f32: bad shape");
    PN_REQUIRE(!argmax || (K > 0 && rows % K == 0), PN_ERR_BAD_ARG, "pn_bn_bwd_stats_det_f32: rows must be a multiple of K");
    PN_DET_WS("pn_bn_bwd_stats_det_f32", bn_det_bytes(rows, C));
    dim3 grid;
    int64_t rpb;
    stats_grid(rows, C, &grid, &rpb);
    cudaStream_t st = (cudaStream_t)stream;
    double* p1 = static_cast<double*>(workspace);
    double* p2 = p1 + (int64_t)grid.x * C;
    if (argmax)
        col_stats_kernel<2, true><<<grid, 32 * ST_LANES, 0, st>>>(y, ldy, rows, C, rpb, dz, lddz, argmax, K, scale, shift, mean,
                                                                   invstd, relu, p1, p2);
    else
        col_stats_kernel<1, true><<<grid, 32 * ST_LANES, 0, st>>>(y, ldy, rows, C, rpb, dz, lddz, nullptr, 1, scale, shift, mean,
                                                                   invstd, relu, p1, p2);
    col_partials_sum_kernel<<<(unsigned)ceil_div(C, 128), 128, 0, st>>>(p1, (int)grid.x, C, s1, s2);
    return finish_launch("pn_bn_bwd_stats_det_f32");
}

PN_EXPORT int pn_bn_eval_bwd_det_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* dz, int64_t lddz,
                                     const int32_t* argmax, int K, const float* scale, const float* shift, const float* mean,
                                     const float* invstd, int relu, double* s1, double* s2, float* dy, int64_t lddy, float* dgamma,
                                     float* dbeta, void* workspace, size_t workspace_bytes, pn_stream_t stream) {
    PN_REQUIRE(y && dz && scale && shift && mean && invstd && s1 && s2 && dy, PN_ERR_BAD_ARG,
               "pn_bn_eval_bwd_det_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && ldy >= C && lddz >= C && lddy >= C, PN_ERR_BAD_ARG, "pn_bn_eval_bwd_det_f32: bad shape");
    PN_REQUIRE(!argmax || (K > 0 && rows % K == 0), PN_ERR_BAD_ARG, "pn_bn_eval_bwd_det_f32: rows must be a multiple of K");
    PN_DET_WS("pn_bn_eval_bwd_det_f32", bn_det_bytes(rows, C));
    dim3 grid;
    int64_t rpb;
    stats_grid(rows, C, &grid, &rpb);
    cudaStream_t st = (cudaStream_t)stream;
    double* p1 = static_cast<double*>(workspace);
    double* p2 = p1 + (int64_t)grid.x * C;
    if (argmax)
        bn_eval_bwd_kernel<true, true><<<grid, 32 * ST_LANES, 0, st>>>(y, ldy, rows, C, rpb, dz, lddz, argmax, K, scale, shift, mean,
                                                                      invstd, relu, p1, p2, dy, lddy);
    else
        bn_eval_bwd_kernel<false, true><<<grid, 32 * ST_LANES, 0, st>>>(y, ldy, rows, C, rpb, dz, lddz, nullptr, 1, scale, shift,
                                                                       mean, invstd, relu, p1, p2, dy, lddy);
    col_partials_sum_kernel<<<(unsigned)ceil_div(C, 128), 128, 0, st>>>(p1, (int)grid.x, C, s1, s2);
    if (dgamma || dbeta) bn_eval_bwd_finalize_kernel<<<(unsigned)ceil_div(C, 128), 128, 0, st>>>(s1, s2, C, dgamma, dbeta);
    return finish_launch("pn_bn_eval_bwd_det_f32");
}

PN_EXPORT size_t pn_grad_weight_f32_workspace_bytes(int64_t rows, int cout, int cin) {
    if (rows <= 0 || cout <= 0 || cin <= 0) return 0;
    int64_t splits, rps;
    grad_weight_f32_shape(rows, cout, cin, &splits, &rps);
    return sizeof(float) * (size_t)splits * ((size_t)cout * cin + cout);
}

// Launch the deterministic slab sum of the weight gradients (also used by grad_tc.cu).
int pn::grad_weight_slab_sum(const float* ws, int64_t splits, int64_t bias_parts, int cout, int cin, float* dw, int64_t lddw, float* db,
                         cudaStream_t st) {
    slab_sum_kernel<<<ew_blocks((int64_t)cout * cin + cout, 256), 256, 0, st>>>(ws, (int)splits, (int)bias_parts, cout, cin, dw, lddw,
                                                                                db);
    return finish_launch("grad weight slab sum");
}

PN_EXPORT int pn_grad_weight_det_f32(const float* dy, int64_t lddy, const float* x, int64_t ldx, int64_t rows, int cout, int cin,
                                     float* dw, int64_t lddw, float* db, void* workspace, size_t workspace_bytes,
                                     pn_stream_t stream) {
    PN_REQUIRE(dy && x && dw, PN_ERR_BAD_ARG, "pn_grad_weight_det_f32: null pointer");
    PN_REQUIRE(rows > 0 && cout > 0 && cin > 0 && lddy >= cout && ldx >= cin && lddw >= cin, PN_ERR_BAD_ARG,
               "pn_grad_weight_det_f32: bad shape");
    PN_DET_WS("pn_grad_weight_det_f32", pn_grad_weight_f32_workspace_bytes(rows, cout, cin));
    int64_t splits, rps;
    grad_weight_f32_shape(rows, cout, cin, &splits, &rps);
    PN_REQUIRE(splits <= 65535, PN_ERR_UNSUPPORTED, "pn_grad_weight_det_f32: too many row splits");
    int vec_ok = 0;
    if (((uintptr_t)dy % 16 == 0) && (lddy % 4 == 0)) vec_ok |= 1;
    if (((uintptr_t)x % 16 == 0) && (ldx % 4 == 0)) vec_ok |= 2;
    cudaStream_t st = (cudaStream_t)stream;
    float* ws = static_cast<float*>(workspace);
    float* wsb = ws + splits * (int64_t)cout * cin;
    dim3 grid((unsigned)ceil_div(cout, 64), (unsigned)ceil_div(cin, 64), (unsigned)splits);
    grad_weight_kernel<64, 64, 16, 4, 4, true><<<grid, 256, 0, st>>>(dy, lddy, x, ldx, rows, rps, cout, cin, ws, cin,
                                                                      db ? wsb : nullptr, vec_ok);
    const int e = finish_launch("pn_grad_weight_det_f32");
    if (e != PN_OK) return e;
    return grad_weight_slab_sum(ws, splits, splits, cout, cin, dw, lddw, db, st);
}

PN_EXPORT int pn_group_bwd_det_f32(const float* dgrouped, int64_t ldg, int col0, int D, const int32_t* offsets,
                                   const int32_t* slots, int B, int N, float* dfeat, pn_stream_t stream) {
    PN_REQUIRE(dgrouped && offsets && slots && dfeat, PN_ERR_BAD_ARG, "pn_group_bwd_det_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && D > 0 && col0 >= 0 && ldg >= col0 + D, PN_ERR_BAD_ARG, "pn_group_bwd_det_f32: bad shape");
    return csr_pull(dgrouped, ldg, col0, D, 1, nullptr, offsets, slots, (int64_t)B * N, dfeat, (cudaStream_t)stream);
}

PN_EXPORT int pn_group_bwd_xyz_det_f32(const float* dgrouped, int64_t ldg, int col0, const int64_t* idx, const int32_t* offsets,
                                       const int32_t* slots, int B, int N, int S, int K, float* dxyz, float* dnew_xyz,
                                       pn_stream_t stream) {
    PN_REQUIRE(dgrouped && idx && offsets && slots && dxyz, PN_ERR_BAD_ARG, "pn_group_bwd_xyz_det_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && S > 0 && K > 0 && col0 >= 0 && ldg >= col0 + 3, PN_ERR_BAD_ARG,
               "pn_group_bwd_xyz_det_f32: bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    if (dnew_xyz) {
        const int64_t groups = (int64_t)B * S;
        group_bwd_xyz_kernel<false><<<ew_blocks(groups * 32, 256), 256, 0, st>>>(dgrouped, ldg, col0, idx, N, S, K, groups, dxyz,
                                                                                 dnew_xyz);
        const int e = finish_launch("pn_group_bwd_xyz_det_f32");
        if (e != PN_OK) return e;
    }
    return csr_pull(dgrouped, ldg, col0, 3, 1, nullptr, offsets, slots, (int64_t)B * N, dxyz, st);
}

PN_EXPORT int pn_three_interpolate_bwd_det_f32(const float* dx, int64_t ldx, int D1, int D2, const float* weight,
                                               const int32_t* offsets, const int32_t* slots, int B, int N, int S, float* dpoints1,
                                               float* dpoints2, pn_stream_t stream) {
    PN_REQUIRE(dx && weight && offsets && slots && dpoints2 && (D1 == 0 || dpoints1), PN_ERR_BAD_ARG,
               "pn_three_interpolate_bwd_det_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && S > 0 && D1 >= 0 && D2 > 0 && ldx >= D1 + D2, PN_ERR_BAD_ARG,
               "pn_three_interpolate_bwd_det_f32: bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    if (D1 > 0) {
        const int64_t total = (int64_t)B * N * D1;
        three_interpolate_bwd_kernel<false><<<ew_blocks(total, 256), 256, 0, st>>>(dx, ldx, D1, 0, nullptr, nullptr, N, S, total,
                                                                                   dpoints1, nullptr);
        const int e = finish_launch("pn_three_interpolate_bwd_det_f32");
        if (e != PN_OK) return e;
    }
    return csr_pull(dx, ldx, D1, D2, 3, weight, offsets, slots, (int64_t)B * S, dpoints2, st);
}

PN_EXPORT int pn_three_interpolate_bwd_xyz_det_f32(const float* dx, int64_t ldx, int D1, int D2, const int64_t* idx,
                                                   const float* weight, const float* points2, int64_t p2B, int64_t p2S, int64_t p2C,
                                                   const float* xyz1, int64_t aB, int64_t aN, int64_t aC, const float* xyz2,
                                                   int64_t bB, int64_t bS, int64_t bC, int B, int N, int S, const int32_t* offsets,
                                                   const int32_t* slots, float* workspace, float* dpoints1, float* dpoints2,
                                                   float* dxyz1, float* dxyz2, pn_stream_t stream) {
    PN_REQUIRE(dx && idx && weight && points2 && xyz1 && xyz2 && offsets && slots && workspace && dpoints2 && dxyz1 && dxyz2 &&
                   (D1 == 0 || dpoints1),
               PN_ERR_BAD_ARG, "pn_three_interpolate_bwd_xyz_det_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && D1 >= 0 && D2 > 0 && ldx >= D1 + D2, PN_ERR_BAD_ARG,
               "pn_three_interpolate_bwd_xyz_det_f32: bad shape");
    PN_REQUIRE(S >= 3, PN_ERR_BAD_ARG, "pn_three_interpolate_bwd_xyz_det_f32: need S >= 3 (got %d)", S);
    const int64_t rows = (int64_t)B * N;
    const bool vec = D1 % 4 == 0 && D2 % 4 == 0 && ldx % 4 == 0 && p2C == 1 && p2S % 4 == 0 && p2B % 4 == 0 &&
                     ((uintptr_t)dx & 15) == 0 && ((uintptr_t)points2 & 15) == 0 && ((uintptr_t)dpoints1 & 15) == 0;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = (unsigned)ew_blocks(rows * 32, 256);
    if (vec)
        three_interpolate_bwd_xyz_kernel<true, true><<<grid, 256, 0, st>>>(dx, ldx, D1, D2, idx, weight, points2, p2B, p2S, p2C, xyz1,
                                                                          aB, aN, aC, xyz2, bB, bS, bC, N, S, rows, dpoints1,
                                                                          dpoints2, dxyz1, workspace);
    else
        three_interpolate_bwd_xyz_kernel<false, true><<<grid, 256, 0, st>>>(dx, ldx, D1, D2, idx, weight, points2, p2B, p2S, p2C,
                                                                           xyz1, aB, aN, aC, xyz2, bB, bS, bC, N, S, rows, dpoints1,
                                                                           dpoints2, dxyz1, workspace);
    int e = finish_launch("pn_three_interpolate_bwd_xyz_det_f32");
    if (e != PN_OK) return e;
    e = csr_pull(dx, ldx, D1, D2, 3, weight, offsets, slots, (int64_t)B * S, dpoints2, st);
    if (e != PN_OK) return e;
    return csr_pull(workspace, 3, 0, 3, 1, nullptr, offsets, slots, (int64_t)B * S, dxyz2, st);
}

PN_EXPORT size_t pn_cross_entropy_workspace_bytes(int64_t rows) {
    return rows > 0 ? sizeof(double) * (2 + (size_t)ew_blocks(rows, 256)) : 0;
}

PN_EXPORT int pn_cross_entropy_det_f32(const float* x, int64_t ldx, const int64_t* target, int64_t rows, int C, void* workspace,
                                       size_t workspace_bytes, float* loss, float* dx, int64_t lddx, float grad_scale,
                                       pn_stream_t stream) {
    PN_REQUIRE(x && target && loss, PN_ERR_BAD_ARG, "pn_cross_entropy_det_f32: null pointer");
    PN_REQUIRE(rows > 0 && C > 0 && ldx >= C && (!dx || lddx >= C), PN_ERR_BAD_ARG, "pn_cross_entropy_det_f32: bad shape");
    PN_DET_WS("pn_cross_entropy_det_f32", pn_cross_entropy_workspace_bytes(rows));
    cudaStream_t st = (cudaStream_t)stream;
    double* ws = static_cast<double*>(workspace);     // [sum, count, block partials]
    cudaError_t e = cudaMemsetAsync(ws, 0, 2 * sizeof(double), st);
    if (e != cudaSuccess) {
        set_error("pn_cross_entropy_det_f32: %s", cudaGetErrorString(e));
        return (int)e;
    }
    const unsigned blocks = ew_blocks(rows, 256);
    label_count_kernel<<<blocks, 256, 0, st>>>(target, rows, ws + 1);      // integers in fp64: exact in any order
    cross_entropy_kernel<true><<<blocks, 256, 0, st>>>(x, ldx, target, rows, C, ws + 2, ws + 1, dx, lddx, grad_scale);
    ordered_sum_kernel<<<1, 32, 0, st>>>(ws + 2, blocks, ws);
    loss_finalize_kernel<<<1, 1, 0, st>>>(ws, ws + 1, loss);
    return finish_launch("pn_cross_entropy_det_f32");
}

PN_EXPORT size_t pn_chamfer_workspace_bytes(int B, int N) {
    return B > 0 && N > 0 ? sizeof(double) * (size_t)B * (size_t)ceil_div(N, CH_TILE) : 0;
}

PN_EXPORT int pn_chamfer_det_f32(const float* p1, int64_t aB, int64_t aN, int64_t aC, const float* p2, int64_t bB, int64_t bN,
                                 int64_t bC, int B, int N, int M, int D, float* per_point, double* total, int32_t* argmin,
                                 void* workspace, size_t workspace_bytes, pn_stream_t stream) {
    PN_REQUIRE(p1 && p2 && total, PN_ERR_BAD_ARG, "pn_chamfer_det_f32: null pointer");
    PN_REQUIRE(B > 0 && B <= 65535 && N > 0 && M > 0 && D > 0 && D <= CH_MAXD, PN_ERR_BAD_ARG,
               "pn_chamfer_det_f32: bad sizes (D <= 8)");
    PN_DET_WS("pn_chamfer_det_f32", pn_chamfer_workspace_bytes(B, N));
    cudaStream_t st = (cudaStream_t)stream;
    double* part = static_cast<double*>(workspace);
    dim3 grid((unsigned)ceil_div(N, CH_TILE), (unsigned)B);
    if (argmin)
        chamfer_kernel<true, true><<<grid, CH_TILE, 0, st>>>(p1, aB, aN, aC, p2, bB, bN, bC, N, M, D, per_point, part, argmin);
    else
        chamfer_kernel<false, true><<<grid, CH_TILE, 0, st>>>(p1, aB, aN, aC, p2, bB, bN, bC, N, M, D, per_point, part, nullptr);
    ordered_sum_kernel<<<1, 32, 0, st>>>(part, (int64_t)grid.x * grid.y, total);
    return finish_launch("pn_chamfer_det_f32");
}

PN_EXPORT int pn_chamfer_bwd_det_f32(const float* p1, int64_t aB, int64_t aN, int64_t aC, const float* p2, int64_t bB, int64_t bN,
                                     int64_t bC, int B, int N, int M, int D, const int32_t* argmin, const float* g_total,
                                     float scale, const int32_t* offsets, const int32_t* slots, float* workspace, float* dp1,
                                     float* dp2, pn_stream_t stream) {
    PN_REQUIRE(p1 && p2 && argmin && g_total && (dp1 || dp2), PN_ERR_BAD_ARG, "pn_chamfer_bwd_det_f32: null pointer");
    PN_REQUIRE(!dp2 || (offsets && slots && workspace), PN_ERR_BAD_ARG, "pn_chamfer_bwd_det_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && M > 0 && D > 0 && D <= CH_MAXD, PN_ERR_BAD_ARG, "pn_chamfer_bwd_det_f32: bad sizes (D <= 8)");
    const int64_t total = (int64_t)B * N;
    cudaStream_t st = (cudaStream_t)stream;
    if (!dp2) {      // nothing is scattered: the default kernel is deterministic already
        chamfer_bwd_kernel<<<ew_blocks(total, 256), 256, 0, st>>>(p1, aB, aN, aC, p2, bB, bN, bC, N, M, D, total, argmin, g_total,
                                                                 scale, dp1, nullptr);
        return finish_launch("pn_chamfer_bwd_det_f32");
    }
    chamfer_bwd_kernel<true><<<ew_blocks(total, 256), 256, 0, st>>>(p1, aB, aN, aC, p2, bB, bN, bC, N, M, D, total, argmin, g_total,
                                                                   scale, dp1, workspace);
    const int e = finish_launch("pn_chamfer_bwd_det_f32");
    if (e != PN_OK) return e;
    return csr_pull(workspace, D, 0, D, 1, nullptr, offsets, slots, (int64_t)B * M, dp2, st);
}

PN_EXPORT size_t pn_square_distance_bwd_det_workspace_bytes(int B, int N, int M) {
    if (B <= 0 || N <= 0 || M <= 0) return 0;
    int chunk;
    dim3 grid;
    sqdist_bwd_shape(B, N, M, &chunk, &grid);
    return sizeof(float) * 4 * ((size_t)(1 + grid.x) * B * N + (size_t)(1 + grid.y) * B * M);
}

PN_EXPORT int pn_square_distance_bwd_det_f32(const float* g, int64_t gB, int64_t gN, const float* src, int64_t aB, int64_t aN,
                                             int64_t aC, const float* dst, int64_t bB, int64_t bN, int64_t bC, int B, int N, int M,
                                             void* workspace, size_t workspace_bytes, float* dsrc, float* ddst, pn_stream_t stream) {
    PN_REQUIRE(g && src && dst && (dsrc || ddst), PN_ERR_BAD_ARG, "pn_square_distance_bwd_det_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && M > 0, PN_ERR_BAD_ARG, "pn_square_distance_bwd_det_f32: B, N, M must be positive");
    PN_REQUIRE(B <= 65535 && ceil_div(N, SDB_ROWS) <= 65535, PN_ERR_UNSUPPORTED,
               "pn_square_distance_bwd_det_f32: B <= 65535 and N <= %d", 65535 * SDB_ROWS);
    PN_REQUIRE(gB >= 0 && gN >= 0, PN_ERR_BAD_ARG, "pn_square_distance_bwd_det_f32: negative stride of g");
    PN_DET_WS("pn_square_distance_bwd_det_f32", pn_square_distance_bwd_det_workspace_bytes(B, N, M));
    int chunk;
    dim3 grid;
    sqdist_bwd_shape(B, N, M, &chunk, &grid);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nr = (int64_t)B * N, nc = (int64_t)B * M;
    float* rws = static_cast<float*>(workspace);       // [B,N,4] sums, then [B,M,4] sums, then the per-CTA slots
    float* cws = rws + nr * 4;
    float* rpart = cws + nc * 4;                        // [grid.x, B, N, 4]
    float* cpart = rpart + (int64_t)grid.x * nr * 4;    // [grid.y, B, M, 4]
    const bool vec = ((uintptr_t)g & 15) == 0 && gN % 4 == 0 && (B == 1 || gB % 4 == 0);
    const bool rows = dsrc != nullptr, cols = ddst != nullptr;
    auto kern = vec ? (rows ? (cols ? sqdist_bwd_kernel<true, true, true, true> : sqdist_bwd_kernel<true, true, false, true>)
                            : sqdist_bwd_kernel<true, false, true, true>)
                    : (rows ? (cols ? sqdist_bwd_kernel<false, true, true, true> : sqdist_bwd_kernel<false, true, false, true>)
                            : sqdist_bwd_kernel<false, false, true, true>);
    kern<<<grid, SDB_WARPS * 32, 0, st>>>(g, gB, gN, src, aB, aN, aC, dst, bB, bN, bC, N, M, chunk, rpart, cpart);
    if (rows)
        sqdist_partials_sum_kernel<<<ew_blocks(nr, 256), 256, 0, st>>>(reinterpret_cast<const float4*>(rpart), (int)grid.x, nr,
                                                                       reinterpret_cast<float4*>(rws));
    if (cols)
        sqdist_partials_sum_kernel<<<ew_blocks(nc, 256), 256, 0, st>>>(reinterpret_cast<const float4*>(cpart), (int)grid.y, nc,
                                                                       reinterpret_cast<float4*>(cws));
    sqdist_bwd_finish_kernel<<<ew_blocks(nr + nc, 256), 256, 0, st>>>(src, aB, aN, aC, dst, bB, bN, bC, B, N, M,
                                                                     reinterpret_cast<const float4*>(rws),
                                                                     reinterpret_cast<const float4*>(cws), dsrc, ddst);
    return finish_launch("pn_square_distance_bwd_det_f32");
}
