// fps.cu -- farthest-point sampling (reference: model/pointnet_util.py:63-84).
//
// One thread-block CLUSTER per cloud.  The cloud is split into contiguous chunks, one per CTA; every
// thread keeps PTS points (x, y, z, running min-distance) in registers for the whole kernel, so an
// iteration touches no global memory at all.  Per iteration:
//   1. each thread updates its PTS running distances against the current centroid and tracks its
//      best (distance, index);
//   2. warp arg-max with two REDUX instructions (max over the distance bits -- distances are >= 0, so
//      unsigned order equals float order -- then min over the indices that attain it);
//   3. one __syncthreads, then every warp redundantly reduces the per-warp winners (no second barrier);
//   4. cluster exchange: the CTA's winner (packed key + its coordinates) is stored into every peer's
//      shared memory through DSMEM, one barrier.cluster, then all threads pick the cluster winner.
// Slots are double-buffered by iteration parity so that one barrier per level and iteration is enough.
//
// fps_async_kernel (the default for clusters) removes both barriers from the loop: every WARP pushes its
// own winner (distance bits, index, x, y, z = 20 bytes) straight into a slot of every CTA of the cluster with
// st.async, whose completion is counted in bytes on the RECEIVER's mbarrier (complete_tx); each warp then
// waits on its CTA's local mbarrier, reads the CL*NW slots (one or two per lane) and reduces them with the
// same two-REDUX arg-max.  One-way DSMEM latency instead of store + barrier round trip, no __syncthreads.
//
// Bit-exactness: distance = ((dx*dx + dy*dy) + dz*dz) with explicit _rn intrinsics (no FMA
// contraction), running min, ties resolved to the lowest point index -- as torch.max does on CPU.
#include <cooperative_groups.h>

#include <type_traits>

#include "common.cuh"
#include "tcgen05.cuh"

namespace cg = cooperative_groups;

namespace pn {

constexpr int kMaxCluster = 16;
constexpr unsigned kNoIndex = 0xFFFFFFFFu;

struct __align__(32) FpsMsg {
    unsigned long long key;  // (distance bits << 32) | ~index : max key = max distance, then min index
    float x, y, z;
    float pad[3];
};

constexpr int kFpsSmemHeader = 2 * kMaxCluster * (int)sizeof(FpsMsg) + 2 * 32 * (int)sizeof(uint2) + 64;   // + two mbarriers (async exchange)

// the address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ unsigned map_to_cta(unsigned addr, unsigned rank) {
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}

template <int THREADS, int PTS, bool CLUSTER>
__global__ void __launch_bounds__(THREADS, 1)
fps_kernel(const float* __restrict__ xyz, int64_t sB, int64_t sN, int64_t sC, int N, int npoint,
           const int64_t* __restrict__ start, int64_t* __restrict__ out, unsigned long long* seq, int chunk, int async_x) {
    constexpr int NW = THREADS / 32;
    extern __shared__ __align__(32) unsigned char smem_raw[];
    FpsMsg* cl_slots = reinterpret_cast<FpsMsg*>(smem_raw);                                   // [2][16]
    uint2* warp_slots = reinterpret_cast<uint2*>(smem_raw + 2 * kMaxCluster * sizeof(FpsMsg));  // [2][32]
    unsigned long long* xbar = reinterpret_cast<unsigned long long*>(smem_raw + kFpsSmemHeader - 64);   // [2], async exchange
    float* sx = reinterpret_cast<float*>(smem_raw + kFpsSmemHeader);
    float* sy = sx + chunk;
    float* sz = sy + chunk;

    unsigned CL = 1, rank = 0;
    if constexpr (CLUSTER) {
        cg::cluster_group cluster = cg::this_cluster();
        CL = cluster.num_blocks();
        rank = cluster.block_rank();
    }
    const int b = blockIdx.x / CL;
    const float* __restrict__ p = xyz + (int64_t)b * sB;
    const int base = rank * chunk;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    float x[PTS], y[PTS], z[PTS], d[PTS];
#pragma unroll
    for (int k = 0; k < PTS; ++k) {
        const int li = tid + k * THREADS;
        const int j = base + li;
        const bool ok = li < chunk && j < N;
        x[k] = ok ? p[(int64_t)j * sN] : 0.0f;
        y[k] = ok ? p[(int64_t)j * sN + sC] : 0.0f;
        z[k] = ok ? p[(int64_t)j * sN + 2 * sC] : 0.0f;
        d[k] = ok ? 1e10f : -2.0f;  // -2 marks an empty slot: never selected, never updated
        if (li < chunk) {
            sx[li] = x[k];
            sy[li] = y[k];
            sz[li] = z[k];
        }
    }
    int far = (int)start[b];
    float cx = p[(int64_t)far * sN], cy = p[(int64_t)far * sN + sC], cz = p[(int64_t)far * sN + 2 * sC];
    if constexpr (CLUSTER) {
        if (async_x && tid == 0) {
            tc::mbar_init(tc::smem_u32(&xbar[0]), 1);
            tc::mbar_init(tc::smem_u32(&xbar[1]), 1);
            tc::mbar_init_fence();
        }
        __syncthreads();
        cg::this_cluster().sync();  // peers must be resident (and their barriers initialised) before DSMEM stores
    } else {
        __syncthreads();
    }

    int64_t* __restrict__ o = out + (int64_t)b * npoint;
    for (int i = 0; i < npoint; ++i) {
        if (rank == 0 && tid == 0) {
            o[i] = far;
            // progress feed for consumers running beside this kernel: index and "valid" flag in ONE 8-byte store, so a
            // reader that sees the flag has the index (no fence in this latency-critical loop)
            if (seq) *reinterpret_cast<volatile unsigned long long*>(seq + (int64_t)b * npoint + i) = ((unsigned long long)(unsigned)far << 32) | 1ull;
        }
        float bv = -1.0f;
        int bk = 0;
#pragma unroll
        for (int k = 0; k < PTS; ++k) {
            const float dd = sqdist_diff(x[k], y[k], z[k], cx, cy, cz);
            d[k] = fminf(d[k], dd);
            if (d[k] > bv) {  // strict: the lowest index wins inside a thread (k ascending = index ascending)
                bv = d[k];
                bk = k;
            }
        }
        const unsigned vb = __float_as_uint(fmaxf(bv, 0.0f));
        const unsigned gi = bv < 0.0f ? kNoIndex : (unsigned)(base + tid + bk * THREADS);
        const unsigned wm = __reduce_max_sync(0xffffffffu, vb);
        const unsigned wi = __reduce_min_sync(0xffffffffu, vb == wm ? gi : kNoIndex);
        const int par = i & 1;
        unsigned bm, bi;
        if constexpr (NW > 1) {
            if (lane == 0) warp_slots[par * 32 + warp] = make_uint2(wm, wi);
            __syncthreads();
            const uint2 s = lane < NW ? warp_slots[par * 32 + lane] : make_uint2(0u, kNoIndex);
            bm = __reduce_max_sync(0xffffffffu, s.x);
            bi = __reduce_min_sync(0xffffffffu, s.x == bm ? s.y : kNoIndex);
        } else {
            bm = wm;
            bi = wi;
        }
        if constexpr (!CLUSTER) {
            far = (int)bi;
            cx = sx[far];
            cy = sy[far];
            cz = sz[far];
        } else {
            cg::cluster_group cluster = cg::this_cluster();
            if (async_x) {
                // CTA winner -> every CTA of the cluster with st.async, completion counted in bytes on the RECEIVER's mbarrier:
                // a one-way DSMEM store instead of store + barrier.cluster round trip (1.76 -> ~0.8 us per iteration at 16 CTAs)
                const unsigned l_bar = tc::smem_u32(&xbar[par]);
                if (tid == 0) tc::mbar_arrive_expect_tx(l_bar, CL * 20u);
                if (warp == 0 && lane < (int)CL) {
                    const unsigned long long key = ((unsigned long long)bm << 32) | (unsigned long long)(~bi);
                    const int li = bi == kNoIndex ? 0 : (int)bi - base;
                    const unsigned r_slot = map_to_cta(tc::smem_u32(&cl_slots[par * kMaxCluster + rank]), lane);
                    const unsigned r_bar = map_to_cta(l_bar, lane);
                    asm volatile(
                        "st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(r_slot),
                        "r"((unsigned)(key & 0xFFFFFFFFull)), "r"((unsigned)(key >> 32)), "r"(__float_as_uint(sx[li])),
                        "r"(__float_as_uint(sy[li])), "r"(r_bar)
                        : "memory");
                    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(r_slot + 16),
                                 "r"(__float_as_uint(sz[li])), "r"(r_bar)
                                 : "memory");
                }
                tc::mbar_wait(l_bar, (unsigned)((i >> 1) & 1));
            } else {
            if (warp == 0 && lane < (int)CL) {
                FpsMsg m;
                m.key = ((unsigned long long)bm << 32) | (unsigned long long)(~bi);
                const int li = bi == kNoIndex ? 0 : (int)bi - base;
                m.x = sx[li];
                m.y = sy[li];
                m.z = sz[li];
                m.pad[0] = m.pad[1] = m.pad[2] = 0.0f;
                FpsMsg* dst = cluster.map_shared_rank(&cl_slots[par * kMaxCluster + rank], lane);
                *dst = m;
            }
            cluster.sync();
            }
            unsigned long long best = 0ull;
            int bc = 0;
            for (int c = 0; c < (int)CL; ++c) {
                const unsigned long long k = cl_slots[par * kMaxCluster + c].key;
                if (k > best) {
                    best = k;
                    bc = c;
                }
            }
            far = (int)(~(unsigned)(best & 0xFFFFFFFFull));
            const FpsMsg& w = cl_slots[par * kMaxCluster + bc];
            cx = w.x;
            cy = w.y;
            cz = w.z;
        }
    }
    if constexpr (CLUSTER) {
        if (async_x) cg::this_cluster().sync();  // nobody leaves while a peer may still be storing into its shared memory
    }
}

// ------------------------------------------------------------------------------------------------
// st.async + mbarrier exchange
struct __align__(32) FpsSlot {
    unsigned val, idx;  // distance bits, point index
    float x, y, z;
    float pad[3];
};
constexpr int kMaxSlots = 64;
constexpr int kSlotBytes = 20;  // bytes actually transmitted per slot (v4.b32 + b32)
constexpr int kAsyncSmemHeader = 64 + 2 * kMaxSlots * (int)sizeof(FpsSlot);

// ZT: every CTA also keeps the z coordinate of the WHOLE cloud in shared memory (4 N bytes), so a winner travels as
// one 16-byte st.async (distance, index, x, y) instead of two (z is looked up locally by index): half the remote
// writes per iteration on the receiving barriers.
template <int NW, int PTS, bool ZT>
__global__ void __launch_bounds__(NW * 32, 1)
fps_async_kernel(const float* __restrict__ xyz, int64_t sB, int64_t sN, int64_t sC, int N, int npoint,
                 const int64_t* __restrict__ start, int64_t* __restrict__ out, unsigned long long* seq, int chunk) {
    constexpr int THREADS = NW * 32;
    extern __shared__ __align__(32) unsigned char smem_raw[];
    unsigned long long* mbar = reinterpret_cast<unsigned long long*>(smem_raw);          // [2]
    FpsSlot* slots = reinterpret_cast<FpsSlot*>(smem_raw + 64);                            // [2][kMaxSlots]
    float* sx = reinterpret_cast<float*>(smem_raw + kAsyncSmemHeader);
    float* sy = sx + chunk;
    float* sz = sy + chunk;
    float* zt = sz + chunk;   // [N] when ZT

    cg::cluster_group cluster = cg::this_cluster();
    const unsigned CL = cluster.num_blocks();
    const unsigned rank = cluster.block_rank();
    const int nslot = (int)CL * NW;
    const int b = blockIdx.x / CL;
    const float* __restrict__ p = xyz + (int64_t)b * sB;
    const int base = rank * chunk;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    static_assert(PTS % 2 == 0, "points are processed in packed pairs");
    unsigned long long xp[PTS / 2], yp[PTS / 2], zp[PTS / 2];
    float d[PTS];
#pragma unroll
    for (int k = 0; k < PTS; k += 2) {
        float x[2], y[2], z[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int li = tid + (k + u) * THREADS;
            const int j = base + li;
            const bool ok = li < chunk && j < N;
            x[u] = ok ? p[(int64_t)j * sN] : 0.0f;
            y[u] = ok ? p[(int64_t)j * sN + sC] : 0.0f;
            z[u] = ok ? p[(int64_t)j * sN + 2 * sC] : 0.0f;
            d[k + u] = ok ? 1e10f : -2.0f;
            if (li < chunk) {
                sx[li] = x[u];
                sy[li] = y[u];
                sz[li] = z[u];
            }
        }
        xp[k / 2] = pack2(x[0], x[1]);
        yp[k / 2] = pack2(y[0], y[1]);
        zp[k / 2] = pack2(z[0], z[1]);
    }
    if constexpr (ZT) {
        for (int i = tid; i < N; i += THREADS) zt[i] = p[(int64_t)i * sN + 2 * sC];
    }
    if (tid == 0) {
        tc::mbar_init(tc::smem_u32(&mbar[0]), 1);
        tc::mbar_init(tc::smem_u32(&mbar[1]), 1);
        tc::mbar_init_fence();
    }
    int far = (int)start[b];
    far = min(max(far, 0), N - 1);
    float cx = p[(int64_t)far * sN], cy = p[(int64_t)far * sN + sC], cz = p[(int64_t)far * sN + 2 * sC];
    __syncthreads();
    cluster.sync();  // barriers initialised and peers resident before any st.async

    // remote addresses this lane sends to (lane < CL: CTA `lane`); parity 1 lives at a fixed offset
    const unsigned my_slot = rank * NW + warp;
    const unsigned dst_cta = lane < (int)CL ? lane : 0;
    const unsigned r_slot0 = map_to_cta(tc::smem_u32(&slots[my_slot]), dst_cta);
    const unsigned r_bar0 = map_to_cta(tc::smem_u32(&mbar[0]), dst_cta);
    const unsigned l_bar0 = tc::smem_u32(&mbar[0]);
    constexpr unsigned kParSlotOff = kMaxSlots * sizeof(FpsSlot), kParBarOff = sizeof(unsigned long long);

    int64_t* __restrict__ o = out + (int64_t)b * npoint;
    for (int i = 0; i < npoint; ++i) {
        const int par = i & 1;
        if (rank == 0 && tid == 0) {
            o[i] = far;
            // progress feed for consumers running beside this kernel: index and "valid" flag in ONE 8-byte store, so a
            // reader that sees the flag has the index (no fence in this latency-critical loop)
            if (seq) *reinterpret_cast<volatile unsigned long long*>(seq + (int64_t)b * npoint + i) = ((unsigned long long)(unsigned)far << 32) | 1ull;
        }
        if (i == npoint - 1) break;  // the last arg-max would never be used
        if (tid == 0)
            tc::mbar_arrive_expect_tx(l_bar0 + par * kParBarOff, (unsigned)(nslot * (ZT ? 16 : kSlotBytes)));
        float bv = -1.0f;
        int bk = 0;
        const unsigned long long ncx = pack2(-cx, -cx), ncy = pack2(-cy, -cy), ncz = pack2(-cz, -cz);
#pragma unroll
        for (int k = 0; k < PTS; k += 2) {
            float d0, d1;
            sqdist_diff2(xp[k / 2], yp[k / 2], zp[k / 2], ncx, ncy, ncz, d0, d1);
            d[k] = fminf(d[k], d0);
            if (d[k] > bv) {
                bv = d[k];
                bk = k;
            }
            d[k + 1] = fminf(d[k + 1], d1);
            if (d[k + 1] > bv) {
                bv = d[k + 1];
                bk = k + 1;
            }
        }
        const unsigned vb = __float_as_uint(fmaxf(bv, 0.0f));
        const unsigned gi = bv < 0.0f ? kNoIndex : (unsigned)(base + tid + bk * THREADS);
        const unsigned wm = __reduce_max_sync(0xffffffffu, vb);
        const unsigned wi = __reduce_min_sync(0xffffffffu, vb == wm ? gi : kNoIndex);
        if (lane < (int)CL) {
            const int li = wi == kNoIndex ? 0 : (int)wi - base;
            const float mx = sx[li], my = sy[li];
            const unsigned r_slot = r_slot0 + par * kParSlotOff, r_bar = r_bar0 + par * kParBarOff;
            asm volatile(
                "st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(
                    r_slot),
                "r"(wm), "r"(wi), "r"(__float_as_uint(mx)), "r"(__float_as_uint(my)), "r"(r_bar)
                : "memory");
            if constexpr (!ZT) {
                const float mz = sz[li];
                asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(
                                 r_slot + 16),
                             "r"(__float_as_uint(mz)), "r"(r_bar)
                             : "memory");
            }
        }
        tc::mbar_wait(l_bar0 + par * kParBarOff, (unsigned)((i >> 1) & 1));
        // reduce the CL*NW slots: one or two per lane
        unsigned sv = 0u, si = kNoIndex;
        float px = 0.f, py = 0.f, pz = 0.f;
        if (lane < nslot) {
            const FpsSlot& s0 = slots[par * kMaxSlots + lane];
            sv = s0.val; si = s0.idx; px = s0.x; py = s0.y;
            if constexpr (!ZT) pz = s0.z;
        }
        if (lane + 32 < nslot) {
            const FpsSlot& s1 = slots[par * kMaxSlots + lane + 32];
            if (s1.val > sv || (s1.val == sv && s1.idx < si)) {
                sv = s1.val; si = s1.idx; px = s1.x; py = s1.y;
                if constexpr (!ZT) pz = s1.z;
            }
        }
        const unsigned bm = __reduce_max_sync(0xffffffffu, sv);
        const unsigned bi = __reduce_min_sync(0xffffffffu, sv == bm ? si : kNoIndex);
        const unsigned who = __ballot_sync(0xffffffffu, sv == bm && si == bi);
        const int src = __ffs(who) - 1;
        far = (int)bi;
        cx = __shfl_sync(0xffffffffu, px, src);
        cy = __shfl_sync(0xffffffffu, py, src);
        if constexpr (ZT) cz = zt[min(bi, (unsigned)(N - 1))];
        else cz = __shfl_sync(0xffffffffu, pz, src);
    }
    cluster.sync();  // nobody leaves while a peer may still be storing into its shared memory
}

// ------------------------------------------------------------------------------------------------
// Bucket-pruned sampling (exact).  With several batches in flight (runtime.GraphedSemSeg depth > 1) what counts is the SM
// time a sampling launch occupies, not its latency: fps_async_kernel keeps the cloud in registers, which caps a CTA at
// ~6000 points (4 CTAs = 4 SMs per cloud of 24000) and has every thread update every point in every iteration.  This kernel
// reads the cloud in BUCKET order (the cell-sorted float4 (x, y, z, original index) records pn_ball_grid_build_f32 makes
// anyway for the ball query), so a warp's PTS * 32 consecutive points are spatially compact, keeps them in SHARED memory
// (16 B per point: 12288 points per CTA, two CTAs per cloud) and only the running distances in registers, and skips a warp's
// whole update when the new centroid cannot change any of its distances:
//     lb = ((ddx*ddx + ddy*ddy) + ddz*ddz),  ddx = max(lo.x - c.x, c.x - hi.x, 0), ...   (the warp's bounding box)
// is evaluated with the same rounding sequence as the distance itself; IEEE rounding is monotone, so lb <= d(p, c) for every
// point p of the box in fp32, and lb >= max_p mindist(p) implies min(mindist(p), d(p, c)) == mindist(p) for all of them:
// the update is the identity and the warp's cached (max, arg-max) stays valid.  After the first ~50 centroids a new centroid
// touches 10-20 % of the warps, so four warps share a scheduler at the cost of one.  The result is bit-identical to the
// reference: ties are resolved to the lowest ORIGINAL index (carried in the record, compared explicitly, because storage
// order is no longer index order).  Exchange between the CTAs: st.async + mbarrier as in fps_async_kernel (no z table).
template <int NW, int PTS>
__global__ void __launch_bounds__(NW * 32, NW == 8 ? 2 : 1)
fps_pruned_kernel(const float* __restrict__ xyz, int64_t sB, int64_t sN, int64_t sC, const unsigned char* __restrict__ grid_ws,
                  size_t ws_stride, size_t sorted_off, int N, int npoint, const int64_t* __restrict__ start,
                  int64_t* __restrict__ out, unsigned long long* seq, int no_prune) {
    static_assert(PTS % 2 == 0, "points are processed in packed pairs");
    constexpr int CAP = NW * PTS * 32, NQ = PTS / 2;
    extern __shared__ __align__(32) unsigned char smem_raw[];
    unsigned long long* mbar = reinterpret_cast<unsigned long long*>(smem_raw);          // [2]
    FpsSlot* slots = reinterpret_cast<FpsSlot*>(smem_raw + 64);                            // [2][kMaxSlots]
    // the CTA's points, two per pair of 16-byte records so that the packed fp32x2 operands need no shuffling:
    //   rec[((warp * NQ + q) * 2 + 0) * 32 + lane] = (x_a, x_b, y_a, y_b)      a = point 2q, b = point 2q + 1 of the lane
    //   rec[((warp * NQ + q) * 2 + 1) * 32 + lane] = (z_a, z_b, index_a, index_b)
    float4* rec = reinterpret_cast<float4*>(smem_raw + kAsyncSmemHeader);                  // [CAP]

    cg::cluster_group cluster = cg::this_cluster();
    const unsigned CL = cluster.num_blocks();
    const unsigned rank = cluster.block_rank();
    const int nslot = (int)CL * NW;
    const int b = blockIdx.x / CL;
    const float* __restrict__ p = xyz + (int64_t)b * sB;
    const float4* __restrict__ sorted = reinterpret_cast<const float4*>(grid_ws + (size_t)b * ws_stride + sorted_off);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float4* wrec = rec + (size_t)warp * NQ * 2 * 32 + lane;        // this lane's records: wrec[(q * 2 + h) * 32]
    const int g0 = (int)rank * CAP + warp * PTS * 32;              // the warp's run inside the cloud's bucket order

    float d[PTS];
    float lo[3] = {3.0e38f, 3.0e38f, 3.0e38f}, hi[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        float4 v[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int j = g0 + (2 * q + u) * 32 + lane;
            const bool ok = j < N;
            v[u] = make_float4(0.f, 0.f, 0.f, __int_as_float(-1));           // empty slot: index 0xFFFFFFFF
            if (ok) v[u] = sorted[j];
            d[2 * q + u] = ok ? 1e10f : -2.0f;                               // -2: never selected, never updated
            if (ok) {
                lo[0] = fminf(lo[0], v[u].x); hi[0] = fmaxf(hi[0], v[u].x);
                lo[1] = fminf(lo[1], v[u].y); hi[1] = fmaxf(hi[1], v[u].y);
                lo[2] = fminf(lo[2], v[u].z); hi[2] = fmaxf(hi[2], v[u].z);
            }
        }
        wrec[(q * 2 + 0) * 32] = make_float4(v[0].x, v[1].x, v[0].y, v[1].y);
        wrec[(q * 2 + 1) * 32] = make_float4(v[0].z, v[1].z, v[0].w, v[1].w);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c)
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            lo[c] = fminf(lo[c], __shfl_xor_sync(0xffffffffu, lo[c], o));
            hi[c] = fmaxf(hi[c], __shfl_xor_sync(0xffffffffu, hi[c], o));
        }
    const bool warp_empty = g0 >= N;
    if (tid == 0) {
        tc::mbar_init(tc::smem_u32(&mbar[0]), 1);
        tc::mbar_init(tc::smem_u32(&mbar[1]), 1);
        tc::mbar_init_fence();
    }
    int far = (int)start[b];
    far = min(max(far, 0), N - 1);
    float cx = p[(int64_t)far * sN], cy = p[(int64_t)far * sN + sC], cz = p[(int64_t)far * sN + 2 * sC];
    __syncthreads();
    cluster.sync();  // barriers initialised and peers resident before any st.async

    const unsigned my_slot = rank * NW + warp;
    const unsigned dst_cta = lane < (int)CL ? lane : 0;
    const unsigned r_slot0 = map_to_cta(tc::smem_u32(&slots[my_slot]), dst_cta);
    const unsigned r_bar0 = map_to_cta(tc::smem_u32(&mbar[0]), dst_cta);
    const unsigned l_bar0 = tc::smem_u32(&mbar[0]);
    constexpr unsigned kParSlotOff = kMaxSlots * sizeof(FpsSlot), kParBarOff = sizeof(unsigned long long);

    // the warp's cached winner: (distance bits, original index, coordinates); valid while no distance of the warp changes
    float wmax = warp_empty ? -1.0f : 1e10f;     // max of the warp's running distances (as a float, for the box test)
    unsigned wm = 0u, wi = kNoIndex;
    float wx = 0.f, wy = 0.f, wz = 0.f;

    int64_t* __restrict__ o = out + (int64_t)b * npoint;
    for (int i = 0; i < npoint; ++i) {
        const int par = i & 1;
        if (rank == 0 && tid == 0) {
            o[i] = far;
            if (seq) *reinterpret_cast<volatile unsigned long long*>(seq + (int64_t)b * npoint + i) = ((unsigned long long)(unsigned)far << 32) | 1ull;
        }
        if (i == npoint - 1) break;  // the last arg-max would never be used
        if (tid == 0)
            tc::mbar_arrive_expect_tx(l_bar0 + par * kParBarOff, (unsigned)(nslot * kSlotBytes));
        // lower bound of the distance from the new centroid to any point of the warp's box, in the distance's own rounding
        const float ddx = fmaxf(fmaxf(__fsub_rn(lo[0], cx), __fsub_rn(cx, hi[0])), 0.0f);
        const float ddy = fmaxf(fmaxf(__fsub_rn(lo[1], cy), __fsub_rn(cy, hi[1])), 0.0f);
        const float ddz = fmaxf(fmaxf(__fsub_rn(lo[2], cz), __fsub_rn(cz, hi[2])), 0.0f);
        const float lb = __fadd_rn(__fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy)), __fmul_rn(ddz, ddz));
        if (lb < wmax || (no_prune && !warp_empty)) {   // warp-uniform
            const unsigned long long ncx = pack2(-cx, -cx), ncy = pack2(-cy, -cy), ncz = pack2(-cz, -cz);
            float bv = -2.0f;
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                const float4 xy = wrec[(q * 2 + 0) * 32];
                const float4 zi = wrec[(q * 2 + 1) * 32];
                float d0, d1;
                sqdist_diff2(pack2(xy.x, xy.y), pack2(xy.z, xy.w), pack2(zi.x, zi.y), ncx, ncy, ncz, d0, d1);
                d[2 * q] = fminf(d[2 * q], d0);
                d[2 * q + 1] = fminf(d[2 * q + 1], d1);
                bv = fmaxf(bv, fmaxf(d[2 * q], d[2 * q + 1]));
            }
            const unsigned vb = __float_as_uint(fmaxf(bv, 0.0f));
            wm = __reduce_max_sync(0xffffffffu, vb);
            // the lowest ORIGINAL index among the points that attain the warp's maximum (ties are resolved by index, as
            // torch.max does in index order; storage order is bucket order): only the few lanes that hold the maximum look
            unsigned cand = kNoIndex;
            int kb = 0;
            if (bv >= 0.0f && vb == wm) {
#pragma unroll
                for (int k = 0; k < PTS; ++k) {
                    if (d[k] == bv) {
                        const float4 zi = wrec[((k >> 1) * 2 + 1) * 32];
                        const unsigned ov = __float_as_uint((k & 1) ? zi.w : zi.z);
                        if (ov < cand) {
                            cand = ov;
                            kb = k;
                        }
                    }
                }
            }
            wi = __reduce_min_sync(0xffffffffu, cand);
            const unsigned who = __ballot_sync(0xffffffffu, cand == wi && cand != kNoIndex);
            const int src = who ? __ffs(who) - 1 : 0;
            const float4 xy = wrec[((kb >> 1) * 2 + 0) * 32];
            const float4 zi = wrec[((kb >> 1) * 2 + 1) * 32];
            wx = __shfl_sync(0xffffffffu, (kb & 1) ? xy.y : xy.x, src);
            wy = __shfl_sync(0xffffffffu, (kb & 1) ? xy.w : xy.z, src);
            wz = __shfl_sync(0xffffffffu, (kb & 1) ? zi.y : zi.x, src);
            wmax = __uint_as_float(wm);
        }
        if (lane < (int)CL) {
            const unsigned r_slot = r_slot0 + par * kParSlotOff, r_bar = r_bar0 + par * kParBarOff;
            asm volatile(
                "st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(
                    r_slot),
                "r"(wm), "r"(wi), "r"(__float_as_uint(wx)), "r"(__float_as_uint(wy)), "r"(r_bar)
                : "memory");
            asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(r_slot + 16),
                         "r"(__float_as_uint(wz)), "r"(r_bar)
                         : "memory");
        }
        tc::mbar_wait(l_bar0 + par * kParBarOff, (unsigned)((i >> 1) & 1));
        // reduce the CL*NW slots: one or two per lane
        unsigned sv = 0u, si = kNoIndex;
        float px = 0.f, py = 0.f, pz = 0.f;
        if (lane < nslot) {
            const FpsSlot& s0 = slots[par * kMaxSlots + lane];
            sv = s0.val; si = s0.idx; px = s0.x; py = s0.y; pz = s0.z;
        }
        if (lane + 32 < nslot) {
            const FpsSlot& s1 = slots[par * kMaxSlots + lane + 32];
            if (s1.val > sv || (s1.val == sv && s1.idx < si)) {
                sv = s1.val; si = s1.idx; px = s1.x; py = s1.y; pz = s1.z;
            }
        }
        const unsigned bm = __reduce_max_sync(0xffffffffu, sv);
        const unsigned bi = __reduce_min_sync(0xffffffffu, sv == bm ? si : kNoIndex);
        const unsigned who = __ballot_sync(0xffffffffu, sv == bm && si == bi);
        const int src = __ffs(who) - 1;
        far = (int)bi;
        cx = __shfl_sync(0xffffffffu, px, src);
        cy = __shfl_sync(0xffffffffu, py, src);
        cz = __shfl_sync(0xffffffffu, pz, src);
    }
    cluster.sync();  // nobody leaves while a peer may still be storing into its shared memory
}

// Per-call launch configuration (from pn_launch_opts) and, for pn_fps_launch_info, where to report the launch shape.
struct FpsCfg {
    int cluster = 0, threads = 0;
    int exchange = 0;       // 0 auto (st.async where possible), 1 barrier.cluster, 2 st.async
    bool no_ztable = false; // exchange 3: st.async without the per-CTA z table
    bool query_only = false;
    bool block_async = true;   // cluster form of the block-level kernel: st.async exchange (false: barrier.cluster, exchange = 1)
    int* ctas = nullptr;
    size_t* smem = nullptr;
};

template <typename Kern>
static int launch_cluster_kernel(Kern kern, const char* what, int CL, int threads, size_t smem, const FpsCfg& cfg_, const float* xyz,
                                 int64_t sB, int64_t sN, int64_t sC, int B, int N, int npoint, const int64_t* start, int64_t* out,
                                 unsigned long long* seq, int chunk, cudaStream_t stream) {
    if (cfg_.ctas) *cfg_.ctas = B * CL;
    if (cfg_.smem) *cfg_.smem = smem;
    if (cfg_.query_only) return PN_OK;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess && CL > 8) e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("pn_fps_f32: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
        return (int)e;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(B * CL));
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    if (CL > 1) {
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)CL;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
    }
    if constexpr (std::is_invocable_v<Kern, const float*, int64_t, int64_t, int64_t, int, int, const int64_t*, int64_t*, unsigned long long*, int, int>)
        e = cudaLaunchKernelEx(&cfg, kern, xyz, sB, sN, sC, N, npoint, start, out, seq, chunk, cfg_.block_async ? 1 : 0);
    else
        e = cudaLaunchKernelEx(&cfg, kern, xyz, sB, sN, sC, N, npoint, start, out, seq, chunk);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("pn_fps_f32: launch of %s failed (cluster=%d threads=%d smem=%zu): %s", what, CL, threads, smem,
                  cudaGetErrorString(e));
        return (int)e;
    }
    return PN_OK;
}

#define PN_FPS_ARGS fc, xyz, sB, sN, sC, B, N, npoint, start, out, seq, chunk, stream

template <int THREADS>
static int dispatch_barrier(int pts, int CL, const FpsCfg& fc, const float* xyz, int64_t sB, int64_t sN, int64_t sC, int B, int N, int npoint,
                            const int64_t* start, int64_t* out, unsigned long long* seq, int chunk, cudaStream_t stream) {
    const size_t smem = (size_t)kFpsSmemHeader + (size_t)chunk * 3 * sizeof(float);
#define PN_FPS_CASE(P)                                                                                              \
    if (pts <= P)                                                                                                   \
        return CL > 1 ? launch_cluster_kernel(fps_kernel<THREADS, P, true>, "fps_kernel", CL, THREADS, smem, PN_FPS_ARGS) \
                      : launch_cluster_kernel(fps_kernel<THREADS, P, false>, "fps_kernel", CL, THREADS, smem, PN_FPS_ARGS)
    PN_FPS_CASE(1);
    PN_FPS_CASE(2);
    PN_FPS_CASE(4);
    PN_FPS_CASE(8);
    if constexpr (THREADS <= 512) {
        PN_FPS_CASE(16);
    }
#undef PN_FPS_CASE
    set_error("pn_fps_f32: %d points per thread at %d threads exceeds the register-resident limit", pts, THREADS);
    return PN_ERR_UNSUPPORTED;
}

template <int NW>
static int dispatch_async(int pts, int CL, const FpsCfg& fc, const float* xyz, int64_t sB, int64_t sN, int64_t sC, int B, int N, int npoint,
                          const int64_t* start, int64_t* out, unsigned long long* seq, int chunk, cudaStream_t stream) {
    const size_t smem0 = (size_t)kAsyncSmemHeader + (size_t)chunk * 3 * sizeof(float);
    const bool zt = !fc.no_ztable && smem0 + (size_t)N * sizeof(float) <= 200 * 1024;
    const size_t smem = smem0 + (zt ? (size_t)N * sizeof(float) : 0);
#define PN_FPS_CASE(P)                                                                                                       \
    if (pts <= P)                                                                                                            \
        return zt ? launch_cluster_kernel(fps_async_kernel<NW, P, true>, "fps_async_kernel", CL, NW * 32, smem, PN_FPS_ARGS) \
                  : launch_cluster_kernel(fps_async_kernel<NW, P, false>, "fps_async_kernel", CL, NW * 32, smem, PN_FPS_ARGS)
    PN_FPS_CASE(4);
    PN_FPS_CASE(8);
    PN_FPS_CASE(12);
    PN_FPS_CASE(16);
    PN_FPS_CASE(24);
    PN_FPS_CASE(32);
    if constexpr (NW == 8) {   // 256 threads own the whole register file: 2 CTAs x 48 points hold a 24000-point cloud
        PN_FPS_CASE(48);
    }
#undef PN_FPS_CASE
    set_error("pn_fps_f32: %d points per thread at %d warps exceeds the register-resident limit", pts, NW);
    return PN_ERR_UNSUPPORTED;
}

}  // namespace pn

static int fps_cfg_from_opts(const pn_launch_opts* o, pn::FpsCfg* fc) {
    if (!o) return PN_OK;
    const int cluster_size = o->fps_cluster, threads = o->fps_threads, exchange = o->fps_exchange;
    const bool cl_ok = cluster_size == 0 || cluster_size == 1 || cluster_size == 2 || cluster_size == 3 || cluster_size == 4 ||
                       cluster_size == 8 || cluster_size == 16;
    const bool th_ok = threads == 0 || threads == 64 || threads == 128 || threads == 256 || threads == 512 ||
                       threads == 1024;
    PN_REQUIRE(cl_ok && th_ok && exchange >= 0 && exchange <= 3, PN_ERR_BAD_ARG,
               "pn_launch_opts: fps_cluster in {0,1,2,3,4,8,16}, fps_threads in {0,64..1024}, fps_exchange in {0,1,2,3}");
    fc->cluster = cluster_size;
    fc->threads = threads;
    fc->exchange = exchange == 3 ? 2 : exchange;
    fc->no_ztable = exchange == 3;
    fc->block_async = exchange != 1;
    return PN_OK;
}

static int fps_dispatch(const pn::FpsCfg& fc, const float* xyz, int64_t sB, int64_t sN, int64_t sC, int B, int N, int npoint,
                        const int64_t* start, int64_t* out, unsigned long long* seq, pn_stream_t stream_);

PN_EXPORT int pn_fps_f32(const float* xyz, int64_t sB, int64_t sN, int64_t sC, int B, int N, int npoint,
                         const int64_t* start, int64_t* out, const pn_launch_opts* opts, pn_stream_t stream_) {
    PN_REQUIRE(xyz && start && out, PN_ERR_BAD_ARG, "pn_fps_f32: null pointer");
    pn::FpsCfg fc;
    if (int rc = fps_cfg_from_opts(opts, &fc)) return rc;
    return fps_dispatch(fc, xyz, sB, sN, sC, B, N, npoint, start, out, nullptr, stream_);
}

PN_EXPORT int pn_fps_progress_f32(const float* xyz, int64_t sB, int64_t sN, int64_t sC, int B, int N, int npoint,
                                  const int64_t* start, int64_t* out, uint64_t* progress, const pn_launch_opts* opts,
                                  pn_stream_t stream_) {
    PN_REQUIRE(xyz && start && out && progress, PN_ERR_BAD_ARG, "pn_fps_progress_f32: null pointer");
    pn::FpsCfg fc;
    if (int rc = fps_cfg_from_opts(opts, &fc)) return rc;
    return fps_dispatch(fc, xyz, sB, sN, sC, B, N, npoint, start, out, reinterpret_cast<unsigned long long*>(progress), stream_);
}

PN_EXPORT int pn_fps_sorted_f32(const float* xyz, int64_t sB, int64_t sN, int64_t sC, const void* grid, size_t grid_bytes, int B,
                                int N, int npoint, const int64_t* start, int64_t* out, uint64_t* progress, const pn_launch_opts* opts,
                                pn_stream_t stream_) {
    using namespace pn;
    PN_REQUIRE(xyz && grid && start && out, PN_ERR_BAD_ARG, "pn_fps_sorted_f32: null pointer");
    PN_REQUIRE(B > 0 && N > 0 && npoint > 0, PN_ERR_BAD_ARG, "pn_fps_sorted_f32: B, N, npoint must be positive (got %d, %d, %d)", B, N,
               npoint);
    PN_REQUIRE(grid_bytes >= pn_ball_grid_bytes(B, N), PN_ERR_BAD_ARG, "pn_fps_sorted_f32: grid buffer too small");
    // 32 warps x 12 points per lane (default), or (tuning hook, fps_threads = 512) 16 warps x 24 points per lane
    // (both hold 12288 points per CTA; beyond two CTAs per cloud only the 16-warp shape keeps cluster x warps <= 64 slots)
    int NW = ((opts && opts->fps_threads == 512) || N > 2 * 12288) ? 16 : 32;
    if (opts && opts->fps_threads == 256 && N <= 8 * 6144) NW = 8;       // 8 warps x 24 points: 6144 per CTA, two CTAs fit one SM
    const int PTS = NW == 32 ? 12 : 24;
    const int CAP = NW * PTS * 32;
    const int CL = (int)ceil_div(N, CAP);
    PN_REQUIRE(CL <= 64 / NW, PN_ERR_UNSUPPORTED, "pn_fps_sorted_f32: N=%d exceeds %d (%d CTAs of %d points)", N, 64 / NW * CAP, 64 / NW, CAP);
    const int no_prune = (opts && opts->fps_exchange == 1) ? 1 : 0;      // tuning hook: every warp updates every iteration
    auto launch = [&](auto kern) -> int {
        const size_t smem = (size_t)kAsyncSmemHeader + (size_t)CAP * sizeof(float4);
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_error("pn_fps_sorted_f32: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
            return (int)e;
        }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(B * CL));
        cfg.blockDim = dim3((unsigned)(NW * 32));
        cfg.dynamicSmemBytes = smem;
        cfg.stream = (cudaStream_t)stream_;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)CL;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        e = cudaLaunchKernelEx(&cfg, kern, xyz, sB, sN, sC, static_cast<const unsigned char*>(grid), ball_grid_cloud_bytes(N),
                               ball_grid_sorted_offset(), N, npoint, start, out, reinterpret_cast<unsigned long long*>(progress),
                               no_prune);
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_error("pn_fps_sorted_f32: launch failed (cluster=%d smem=%zu): %s", CL, smem, cudaGetErrorString(e));
            return (int)e;
        }
        return PN_OK;
    };
    return NW == 32 ? launch(fps_pruned_kernel<32, 12>) : (NW == 16 ? launch(fps_pruned_kernel<16, 24>) : launch(fps_pruned_kernel<8, 24>));
}

PN_EXPORT int pn_fps_launch_info(int B, int N, int npoint, const pn_launch_opts* opts, int* ctas, size_t* smem_bytes) {
    PN_REQUIRE(ctas && smem_bytes, PN_ERR_BAD_ARG, "pn_fps_launch_info: null pointer");
    pn::FpsCfg fc;
    if (int rc = fps_cfg_from_opts(opts, &fc)) return rc;
    fc.query_only = true;
    fc.ctas = ctas;
    fc.smem = smem_bytes;
    *ctas = 0;
    *smem_bytes = 0;
    return fps_dispatch(fc, reinterpret_cast<const float*>(16), 3 * (int64_t)N, 1, N, B, N, npoint,
                        reinterpret_cast<const int64_t*>(16), reinterpret_cast<int64_t*>(16), nullptr, nullptr);
}

static int fps_dispatch(const pn::FpsCfg& fc, const float* xyz, int64_t sB, int64_t sN, int64_t sC, int B, int N, int npoint,
                        const int64_t* start, int64_t* out, unsigned long long* seq, pn_stream_t stream_) {
    using namespace pn;
    PN_REQUIRE(B > 0 && N > 0 && npoint > 0, PN_ERR_BAD_ARG, "pn_fps_f32: B, N, npoint must be positive (got %d, %d, %d)", B,
               N, npoint);
    cudaStream_t stream = (cudaStream_t)stream_;
    int CL = fc.cluster;
    if (CL == 0) {
        if (N <= 3072) CL = 1;
        else if (N <= 6144) CL = 2;
        else if (N <= 12288) CL = 4;
        else if (N <= 65536) CL = 8;   // 8 x 256 threads x 32 points; clusters of 16 are placed one per GPC at best and were
        else CL = 16;                  // measured slower wherever 8 CTAs can hold the cloud (N = 32768: 1.07 vs 0.56 ms)
    }
    const int chunk = (int)ceil_div(N, CL);
    // st.async exchange: clusters only, at most 64 slots (cluster size x warps) and 32 points per thread
    bool use_async = CL > 1 && fc.exchange != 1;
    int threads = fc.threads;
    if (use_async) {
        if (threads == 0) threads = (chunk <= 4096 && CL * 4 <= kMaxSlots) ? 128 : 256;
        const int nw = threads / 32;
        if (threads > 256 || CL * nw > kMaxSlots || ceil_div(chunk, threads) > (threads == 256 ? 48 : 32)) {
            PN_REQUIRE(fc.exchange != 2, PN_ERR_UNSUPPORTED,
                       "pn_fps_f32: st.async exchange needs cluster*warps <= 64, threads <= 256 and <= 32 (48 at 256 threads) points per thread "
                       "(N=%d cluster=%d threads=%d)", N, CL, threads);
            use_async = false;
            threads = fc.threads;
        }
    }
    if (use_async) {
        const int pts = (int)ceil_div(chunk, threads);
        PN_REQUIRE((size_t)kAsyncSmemHeader + (size_t)chunk * 12 <= 227 * 1024, PN_ERR_UNSUPPORTED,
                   "pn_fps_f32: N=%d needs %d points per CTA at cluster size %d; shared memory holds 19000", N, chunk, CL);
        switch (threads) {
            case 64: return dispatch_async<2>(pts, CL, PN_FPS_ARGS);
            case 128: return dispatch_async<4>(pts, CL, PN_FPS_ARGS);
            default: return dispatch_async<8>(pts, CL, PN_FPS_ARGS);
        }
    }
    if (threads == 0) threads = N <= 128 ? 64 : N <= 512 ? 128 : N <= 2048 ? 256 : 512;
    const int pts = (int)ceil_div(chunk, threads);
    PN_REQUIRE((size_t)kFpsSmemHeader + (size_t)chunk * 12 <= 227 * 1024, PN_ERR_UNSUPPORTED,
               "pn_fps_f32: N=%d needs %d points per CTA at cluster size %d; shared memory holds 19200", N, chunk, CL);
    switch (threads) {
        case 64: return dispatch_barrier<64>(pts, CL, PN_FPS_ARGS);
        case 128: return dispatch_barrier<128>(pts, CL, PN_FPS_ARGS);
        case 256: return dispatch_barrier<256>(pts, CL, PN_FPS_ARGS);
        case 512: return dispatch_barrier<512>(pts, CL, PN_FPS_ARGS);
        default: return dispatch_barrier<1024>(pts, CL, PN_FPS_ARGS);
    }
}
