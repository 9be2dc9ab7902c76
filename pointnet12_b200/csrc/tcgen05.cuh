// tcgen05.cuh -- the PTX of the tensor-core kernels (mlp_tc.cu, gemm_tc.cu, grad_tc.cu) and of the mbarrier exchange of
// fps.cu, and the only place that knows the encodings they rely on: the UMMA instruction and shared-memory descriptors,
// the bf16 hi/lo split of an fp32 operand and the three-product MMA issue.  The encodings were pinned on hardware with
// tools/probes/tc_probe.cu (DESIGN.md section 5), which keeps its own copy on purpose.  sm_100a only.
#pragma once
#include <cuda_bf16.h>

namespace pn {
namespace tc {

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// after the barriers of a CTA are initialised, before any other thread (or peer CTA, or the async proxy) uses them
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// generic-proxy stores to shared memory -> visible to the MMA (async proxy)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    unsigned done = 0;
    while (!done) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------ bulk copy
// global -> shared on the TMA engine, completion counted in bytes on `bar` (bytes: a multiple of 16)
__device__ __forceinline__ void bulk_load(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
// `bytes` in pieces of at most 32 KB, all completing on one barrier, whose expected byte count is set first.  (`bytes` by
// reference: where it is a field of a kernel's parameter struct it is then re-read after each copy, as the loop written out
// in the kernel did, and the kernel's code does not change.)
__device__ __forceinline__ void bulk_load_pieces(unsigned dst, const unsigned char* src, const unsigned& bytes, unsigned bar) {
    mbar_arrive_expect_tx(bar, bytes);
    for (unsigned off = 0; off < bytes; off += 32768u) {
        const unsigned n = bytes - off < 32768u ? bytes - off : 32768u;
        bulk_load(dst + off, src + off, n, bar);
    }
}

// ------------------------------------------------------------------------------------------------ tcgen05
// one lane of a converged warp (the instruction sequence around it stays warp-uniform, so descriptors and barrier
// addresses are computed in uniform registers instead of being moved there lane by lane)
__device__ __forceinline__ bool elect() {
    unsigned p;
    asm volatile("{ .reg .pred q; elect.sync _|q, 0xffffffff; selp.u32 %0, 1, 0, q; }" : "=r"(p));
    return p != 0;
}
// whole warp: `cols` (a power of two >= 32) TMEM columns, base address written to *slot in shared memory
__device__ __forceinline__ void tmem_alloc(unsigned* slot, unsigned cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(unsigned taddr, unsigned cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols));
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// arrives on `bar` once the MMAs this thread issued before have completed
__device__ __forceinline__ void commit(unsigned bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 columns: r[j] = column j of the thread's lane
__device__ __forceinline__ void ld32(unsigned taddr, unsigned (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 16 lanes x 32 columns: r[4m + 2rb + c] = row t/4 + 8rb, column 8m + 2(t%4) + c
__device__ __forceinline__ void ld_16x256_x4(unsigned taddr, unsigned (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.16x256b.x4.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 32 lanes x 16 columns
__device__ __forceinline__ void st16(unsigned taddr, const unsigned (&r)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
                 "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
                 "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
                 : "memory");
}
// 16 lanes x 8 columns: thread t provides {row t/4: columns 2(t%4), 2(t%4)+1; row t/4 + 8: the same columns}
// (pinned on hardware with tools/probes/st_shape_probe.cu)
__device__ __forceinline__ void st_16x256(unsigned taddr, unsigned a0, unsigned a1, unsigned b0, unsigned b1) {
    asm volatile("tcgen05.st.sync.aligned.16x256b.x1.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(a0), "r"(a1), "r"(b0), "r"(b1) : "memory");
}

// ------------------------------------------------------------------------------------------------ descriptors
// Instruction descriptor of kind::f16: D fp32 (bit 4), A and B bf16 (bits 7, 10), both K-major, N / 8 at bit 17, M / 16 at bit 24.
__host__ __device__ constexpr unsigned idesc_bf16_f32(unsigned m, unsigned n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
// Shared-memory descriptor of a K-major operand without swizzle, built from core matrices of 8 rows x 16 bytes:
// start address (bits 0-13), leading byte offset 128 B = the next 8 K values (bits 16-29), stride byte offset `sbo` = the
// next 8 rows (bits 32-45), all in 16-byte units, and the version bit 46.  As two 32-bit halves, for loops that keep the
// descriptor in uniform registers and advance the start address in the low half:
__host__ __device__ constexpr unsigned sdesc_hi32(unsigned sbo) { return ((sbo >> 4) & 0x3FFF) | (1u << 14); }
__host__ __device__ constexpr unsigned sdesc_lo32(unsigned addr) { return (((128u >> 4) & 0x3FFF) << 16) | ((addr >> 4) & 0x3FFF); }
// ... and as a 64-bit base (everything but the address) that sdesc() completes
__host__ __device__ constexpr unsigned long long sdesc_base(unsigned sbo) {
    return ((unsigned long long)sdesc_hi32(sbo) << 32) | (unsigned long long)sdesc_lo32(0);
}
__device__ __forceinline__ unsigned long long sdesc(unsigned long long base, unsigned addr) {
    return base | (unsigned long long)((addr >> 4) & 0x3FFF);
}

// ------------------------------------------------------------------------------------------------ MMA issue
// D (TMEM) = A * B^T (+ D if acc != 0), kind::f16, A from shared memory (given by its descriptor) ...
__device__ __forceinline__ void mma(unsigned d, unsigned long long a, unsigned long long b, unsigned idesc, unsigned acc) {
    asm volatile("{ .reg .pred q; setp.ne.b32 q, %4, 0; tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, q; }" ::"r"(d), "l"(a),
                 "l"(b), "r"(idesc), "r"(acc)
                 : "memory");
}
// ... or from TMEM (given by its address)
__device__ __forceinline__ void mma(unsigned d, unsigned a, unsigned long long b, unsigned idesc, unsigned acc) {
    asm volatile("{ .reg .pred q; setp.ne.b32 q, %4, 0; tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, q; }" ::"r"(d), "r"(a),
                 "l"(b), "r"(idesc), "r"(acc)
                 : "memory");
}
// fp32 parity from bf16 operands: a*b ~ a_hi*b_hi + a_hi*b_lo + a_lo*b_hi (the dropped a_lo*b_lo is ~2^-18 relative).
// split = false issues a_hi*b_hi only (plain bf16).  A: shared-memory descriptors or TMEM addresses, as for mma().
template <typename A>
__device__ __forceinline__ void mma_bf16x3(unsigned d, A a_hi, A a_lo, unsigned long long b_hi, unsigned long long b_lo, unsigned idesc,
                                           unsigned acc, bool split = true) {
    mma(d, a_hi, b_hi, idesc, acc);
    if (split) {
        mma(d, a_hi, b_lo, idesc, 1u);
        mma(d, a_lo, b_hi, idesc, 1u);
    }
}

// ------------------------------------------------------------------------------------------------ bf16 hi / lo split
// hi = rn(v), lo = rn(v - hi) for a pair (a, b), packed as bf16x2 with a -- the even k -- in the low half
__device__ __forceinline__ void split_bf16x2(float a, float b, unsigned& hi, unsigned& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);      // cvt.rn.bf16x2.f32: two conversions per instruction
    hi = *reinterpret_cast<const unsigned*>(&h);
    const __nv_bfloat162 l = __floats2bfloat162_rn(a - __uint_as_float(hi << 16), b - __uint_as_float(hi & 0xFFFF0000u));
    lo = *reinterpret_cast<const unsigned*>(&l);
}
// 8 consecutive k -> 8 bf16 hi + 8 bf16 lo, one 16-byte shared-memory store each (a row of a core matrix)
__device__ __forceinline__ void store_split8(unsigned char* hi_img, unsigned char* lo_img, unsigned off, const float (&v)[8]) {
    unsigned h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) split_bf16x2(v[2 * j], v[2 * j + 1], h[j], l[j]);
    *reinterpret_cast<uint4*>(hi_img + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo_img + off) = make_uint4(l[0], l[1], l[2], l[3]);
}
// 32 consecutive k -> 16 packed hi words + 16 lo words, stored at TMEM addresses t_hi and t_lo (an A operand in TMEM)
__device__ __forceinline__ void store_split32(unsigned t_hi, unsigned t_lo, const float (&v)[32]) {
    unsigned hi[16], lo[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) split_bf16x2(v[2 * j], v[2 * j + 1], hi[j], lo[j]);
    st16(t_hi, hi);
    st16(t_lo, lo);
}

// ------------------------------------------------------------------------------------------------ warp column reduction
// Steps W, W/2, .., STOP of a butterfly that reduces columns held one row per lane (v[c] = column c of the lane's row) with
// `op`: a step combines the W columns a lane keeps with those of lane ^ W and halves the columns it is responsible for.
//   W = 16, STOP = 1: lane j ends with column j, reduced over the warp, in v[0] (31 shuffles instead of 32 x 5).
//   W = 8, STOP = 1: the same for columns v[0..15] over each half-warp: lane j ends with column j % 16.
//   W = 16, STOP = S: lane j ends with columns (j & (32 - S)) + i, i < S, in v[i], reduced over the lanes that share j % S;
//   steps S/2 .. 1 on v[0..S-1] (possibly in another type) finish the reduction.
template <int W, int STOP, typename T, typename Op>
__device__ __forceinline__ void col_butterfly(T (&v)[32], int lane, Op op) {
    if constexpr (W >= STOP) {
        const bool up = (lane & W) != 0;
#pragma unroll
        for (int i = 0; i < W; ++i) {
            const T send = up ? v[i] : v[i + W];
            const T keep = up ? v[i + W] : v[i];
            v[i] = op(keep, __shfl_xor_sync(0xffffffffu, send, W));
        }
        col_butterfly<W / 2, STOP>(v, lane, op);
    }
}

}  // namespace tc
}  // namespace pn
