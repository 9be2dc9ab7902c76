// common.cuh -- shared helpers for libpn12_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "pn12_b200.h"

#define PN_EXPORT extern "C" __attribute__((visibility("default")))

namespace pn {

// Thread-local description of the last failure; read through pn_last_error_string().
void set_error(const char* fmt, ...);

inline int finish_launch(const char* what) {
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) {
        cudaGetLastError();  // clear the sticky launch error
        set_error("%s: CUDA launch failed: %s", what, cudaGetErrorString(e));
        return (int)e;
    }
    return PN_OK;
}

#define PN_REQUIRE(cond, code, ...)      \
    do {                                 \
        if (!(cond)) {                   \
            pn::set_error(__VA_ARGS__);  \
            return (code);               \
        }                                \
    } while (0)

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Layout of the per-cloud bucket workspace of pn_ball_grid_build_f32 (ball_grid.cu): bytes per cloud and the offset of the
// cell-sorted float4 (x, y, z, original index) records, for kernels of other files that walk the cloud in bucket order.
size_t ball_grid_cloud_bytes(int N);
size_t ball_grid_sorted_offset();

// Launch with the extended API (dynamic shared memory above 48 KB was enabled by the caller via cudaFuncSetAttribute).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// Squared norm exactly as torch.sum(p ** 2, -1) evaluates it on three components:
// ((x*x + y*y) + z*z), each operation rounded to fp32, no FMA contraction.
__device__ __forceinline__ float sqnorm3(float x, float y, float z) {
    return __fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z));
}

// square_distance of the reference (pointnet_util.py:37-39) in its CPU rounding sequence:
//   dot = fma(az,bz, fma(ay,by, ax*bx));  d = ((-2*dot) + |a|^2) + |b|^2
// (-2*dot is exact, so fma(-2, dot, sa) rounds exactly like (-2*dot) + sa.)
__device__ __forceinline__ float sqdist_expand(float ax, float ay, float az, float sa, float bx, float by,
                                               float bz, float sb) {
    const float dot = __fmaf_rn(az, bz, __fmaf_rn(ay, by, __fmul_rn(ax, bx)));
    return __fadd_rn(__fmaf_rn(-2.0f, dot, sa), sb);
}

// FPS distance of the reference (pointnet_util.py:80): sum((p - c) ** 2) = ((dx*dx + dy*dy) + dz*dz).
__device__ __forceinline__ float sqdist_diff(float px, float py, float pz, float cx, float cy, float cz) {
    const float dx = __fsub_rn(px, cx), dy = __fsub_rn(py, cy), dz = __fsub_rn(pz, cz);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// Packed fp32 pairs: add / mul / fma .rn.f32x2 (FADD2 / FMUL2 / FFMA2) round each half exactly like the scalar .rn form,
// two operations per instruction.  ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (it does not for the scalar
// .rn forms), which changes the rounding: a product that feeds a sum must be unpacked and summed with the scalar _rn
// intrinsics, unless the rounding wanted is that of the fma (as in sqdist_expand).
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) {
    asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

// sqdist_diff for two points at once (8 arithmetic instructions instead of 16); n* = the negated centroid broadcast to
// both halves (p + (-c) == p - c)
__device__ __forceinline__ void sqdist_diff2(unsigned long long px, unsigned long long py, unsigned long long pz,
                                             unsigned long long ncx, unsigned long long ncy, unsigned long long ncz, float& d0,
                                             float& d1) {
    const unsigned long long dx = add2(px, ncx), dy = add2(py, ncy), dz = add2(pz, ncz);
    const unsigned long long xx = mul2(dx, dx), yy = mul2(dy, dy), zz = mul2(dz, dz);
    float x0, x1, y0, y1, z0, z1;      // the sums on the unpacked halves: packed, they would contract into FFMA2
    unpack2(xx, x0, x1);
    unpack2(yy, y0, y1);
    unpack2(zz, z0, z1);
    d0 = __fadd_rn(__fadd_rn(x0, y0), z0);
    d1 = __fadd_rn(__fadd_rn(x1, y1), z1);
}

}  // namespace pn
