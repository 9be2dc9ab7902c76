/*
 * pn12_b200.h -- C ABI of libpn12_b200.so: hand-written sm_100a CUDA kernels for the PointNet /
 * PointNet++ forward hot path of Jiang-Muyun/PointNet12.
 *
 * The reference has no FFI layer (it is pure Python/PyTorch); this header IS the native boundary the
 * new build creates underneath the reference's Python API (SURVEY.md section 8b).  Every entry point
 * names the reference function it replaces (file:line into the reference repo).  The Python binding a
 * maintainer adds on the reference side is shown in INTEGRATION.md.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  All pointers are DEVICE pointers unless noted.
 *   - The caller owns every buffer; the library never allocates, frees or synchronises.
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous and capturable in a
 *     CUDA graph.  Entry points are stateless and re-entrant: the library keeps no mutable process-wide settings;
 *     everything that tunes a launch travels with the call in a pn_launch_opts (NULL = defaults).
 *   - Point clouds are addressed point-major through ELEMENT strides (sB, sN, sC): element (b, n, c)
 *     lives at base[b*sB + n*sN + c*sC].  This covers the permuted [B,3,N] views the reference passes
 *     around (model/pointnet_util.py:184) as well as contiguous [B,N,3].
 *   - Feature matrices are row-major [rows, C] with a leading dimension (ld*, in elements).
 *   - Indices are int64 at the boundary, as in the reference.
 *   - Return value: 0 on success; negative pn_status on bad arguments; positive = cudaError_t of
 *     the launch.  pn_last_error_string() describes the last failure on the calling thread.
 *     Nothing is printed and nothing throws.
 *   - pointnet12_b200/_native.py builds its ctypes bindings by reading the declarations below, so they use only
 *     int, int32_t, int64_t, size_t and float by value, pointers (bound as void*), typedefs and structs of these (array
 *     fields sized by an integer #define), enums, and the return types int, size_t and const char*; any other spelling
 *     makes that module's import fail.
 */
#ifndef PN12_B200_H
#define PN12_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* pn_stream_t; /* cudaStream_t */

enum pn_status {
    PN_OK = 0,
    PN_ERR_BAD_ARG = -1,     /* null pointer, non-positive size, inconsistent shape */
    PN_ERR_UNSUPPORTED = -2, /* size outside what the kernels were built for */
    PN_ERR_ALIGNMENT = -3,   /* pointer / leading dimension not aligned as documented */
    PN_ERR_DEVICE = -4       /* not an sm_100 device */
};

/* Library identification: version = major*10000 + minor*100 + patch. */
int pn_version(void);
const char* pn_last_error_string(void);
/* Queries the current device; fails with PN_ERR_DEVICE unless compute capability is 10.x. */
int pn_device_check(int* sm_count, int* cc_major, int* cc_minor);

/* Per-call launch options of the sampling and fused-chain entry points (a HOST struct, read during the call; NULL or
 * all zeros = defaults).  They replace the process-wide setters of ABI 0.3: two threads can run different precisions
 * or launch shapes at the same time.
 *   mlp_passes    0 or 3 = all three split-bf16 products, fp32 parity (~1e-5 relative); 1 = only a_hi * w_hi, i.e. plain
 *                 bf16 inputs with fp32 accumulation -- a third of the tensor-core work (config C4).  Same packed blob.
 *   mlp_engine    0 = automatic (chains whose packed weights fit in shared memory run on the resident-weight kernel,
 *                 larger chains stream their weights through a ring), 1 = always stream, 2 = resident or fail;
 *                 +4 = row-per-thread producers only (no coalesced quad producer), +8 = no N-slicing of single-layer
 *                 chains, +16 = 8-warp streaming CTAs only.  For benchmarks and tests.
 *   reserved_sms  SMs the resident-weight launches (one persistent CTA per SM) leave to kernels of other streams.
 *   tile_counter  (device pointer or NULL) ONE zeroed uint32 owned by the caller and not shared with a launch that may
 *                 run at the same time: the resident-weight kernel then hands out its 128-row tiles through this
 *                 counter instead of a static round-robin, so CTAs that get their SM late (another stream's kernels
 *                 hold it) only take what is left; the kernel resets the counter to zero before it ends.
 *   mlp_debug     profiling hook: device buffer of 4 * 64 * 32 int64 (or NULL); CTA 0 of a resident-weight launch records
 *                 clock64() per phase: [group][tile round % 64][tile start, producer done, then per layer: MMA issue
 *                 start, MMAs issued, accumulator ready, epilogue done; last: tile done].
 *   fps_cluster / fps_threads / fps_exchange
 *                 force the cluster size (1,2,3,4,8,16), threads per CTA (64..1024) and the intra-cluster exchange of
 *                 pn_fps_f32 (1 = DSMEM store + barrier.cluster, 2 = st.async + mbarrier, 3 = the same without the per-CTA
 *                 z table, i.e. two st.async per winner instead of one); 0 = automatic. */
typedef struct pn_launch_opts {
    int mlp_passes;
    int mlp_engine;
    int reserved_sms;
    int fps_cluster;
    int fps_threads;
    int fps_exchange;
    uint32_t* tile_counter;
    void* mlp_debug;
} pn_launch_opts;

/* farthest_point_sample (model/pointnet_util.py:63-84).
 * xyz [B,N,3] via strides; start_idx [B] = the torch.randint draw of :75 (made by the caller on the
 * CPU generator, then copied to the device); out_idx [B,npoint].
 * Distances are ((dx*dx + dy*dy) + dz*dz) in fp32 without fused multiply-add, running minimum,
 * arg-max with the lowest index winning ties -- bit-exact with the reference.
 * One thread-block cluster per cloud; coordinates and running distances stay in registers; the
 * per-iteration arg-max is exchanged between the CTAs with st.async + mbarrier (no barrier in the loop).
 * Limits: N <= 131072. */
int pn_fps_f32(const float* xyz, int64_t sB, int64_t sN, int64_t sC, int B, int N, int npoint,
               const int64_t* start_idx, int64_t* out_idx, const pn_launch_opts* opts, pn_stream_t stream);

/* square_distance (model/pointnet_util.py:19-40): out[b,i,j] = ((-2*dot) + |src_i|^2) + |dst_j|^2
 * with dot = fma(z,z', fma(y,y', x*x')), i.e. the fp32 rounding sequence of the reference's CPU path.
 * out is contiguous [B,N,M].  Provided for API completeness; the hot path never materialises it. */
int pn_square_distance_f32(const float* src, int64_t aB, int64_t aN, int64_t aC, const float* dst, int64_t bB,
                           int64_t bN, int64_t bC, int B, int N, int M, float* out, pn_stream_t stream);
/* Backward of square_distance (model/pointnet_util.py:19-40; dist = -2 src dst^T + |src|^2 + |dst|^2) for g = dL/ddist [B,N,M]
 * (batch stride gB >= 0, row stride gN >= 0, unit column stride; 16-byte aligned rows take the vector path):
 *   dsrc[b,n] = 2 (sum_m g[b,n,m]) src[b,n] - 2 sum_m g[b,n,m] dst[b,m]
 *   ddst[b,m] = 2 (sum_n g[b,n,m]) dst[b,m] - 2 sum_n g[b,n,m] src[b,n]
 * the two terms formed apart and subtracted last, as torch's autograd adds the sum and matmul backwards.  g is read once:
 * row and column sums come from the same pass (fp32, column sums accumulated with atomics, so the last bits depend on
 * the order).  src / dst via element strides like pn_square_distance_f32; dsrc [B,N,3] / ddst [B,M,3] contiguous,
 * written; either may be NULL (that side is skipped).  workspace: 16-byte aligned fp32 scratch of 4*B*(N+M) floats,
 * zeroed here.  Limits: B <= 65535, N <= 4194240. */
int pn_square_distance_bwd_f32(const float* g, int64_t gB, int64_t gN, const float* src, int64_t aB, int64_t aN, int64_t aC,
                               const float* dst, int64_t bB, int64_t bN, int64_t bC, int B, int N, int M, float* workspace,
                               float* dsrc, float* ddst, pn_stream_t stream);

/* query_ball_point (model/pointnet_util.py:87-107).
 * out_idx [B,S,nsample]: the first nsample indices j (ascending) with NOT(sqdist(new_xyz_s, xyz_j) >
 * radius2), padded with the first hit; rows without any hit are filled with N (as the reference
 * would).  radius2 = (float)(radius**2).  Membership uses the square_distance formula above. */
int pn_ball_query_f32(const float* xyz, int64_t xB, int64_t xN, int64_t xC, const float* new_xyz, int64_t qB,
                      int64_t qN, int64_t qC, int B, int N, int S, float radius2, int nsample,
                      int64_t* out_idx, pn_stream_t stream);

/* query_ball_point through a uniform-grid bucket pass (same result as pn_ball_query_f32, bit for bit).
 * pn_ball_grid_build_f32 depends on xyz and the radius only (not on the centroids), so a caller can run it
 * beside farthest-point sampling: per cloud it computes the bounding box, picks a cell size >= radius (plus
 * slack for the fp32 rounding of the membership formula) and counting-sorts the points by cell into
 * (x, y, z, original index) records.  grid: caller-owned, 16-byte aligned device buffer of
 * pn_ball_grid_bytes(B, N) bytes.
 * pn_ball_query_grid_f32: one warp per centroid; when the 27 neighbouring cells hold at most `threshold`
 * points they are all tested and the hits are ordered through a shared-memory bitmap over original indices,
 * otherwise the ball is dense and the ordered scan over the raw cloud stops after a short prefix.
 * threshold: 0 = automatic (~sqrt(64 N)), negative = always scan, INT_MAX = always use the cells.
 * done (may be NULL): [B, S] flags of rows that are already complete (see pn_ball_query_stream_f32) and are skipped.
 * Limits: N <= 1048576. */
size_t pn_ball_grid_bytes(int B, int N);
/* The bucket-sorted point order stored in a grid built by pn_ball_grid_build_f32, as (pointer, element stride, batch
 * stride) in int32 elements: order[b*bstride + r*estride] = original index of the r-th point of cloud b in cell order. */
int pn_ball_grid_order(const void* grid, int N, const int32_t** order, int64_t* estride, int64_t* bstride);
int pn_ball_grid_build_f32(const float* xyz, int64_t xB, int64_t xN, int64_t xC, int B, int N, float radius2,
                           void* grid, size_t grid_bytes, pn_stream_t stream);
int pn_ball_query_grid_f32(const float* xyz, int64_t xB, int64_t xN, int64_t xC, const float* new_xyz, int64_t qB,
                           int64_t qN, int64_t qC, int B, int N, int S, float radius2, int nsample,
                           const void* grid, size_t grid_bytes, int threshold, const int32_t* done, int64_t* out_idx,
                           pn_stream_t stream);

/* query_ball_point fed by a RUNNING farthest-point-sampling kernel.  pn_fps_progress_f32 is pn_fps_f32 that also
 * publishes every centroid the moment it is chosen (progress [B, npoint], zeroed by the caller before the launch:
 * one 8-byte word per centroid, index << 32 | 1).  pn_ball_query_stream_f32, launched on ANOTHER stream once the grid
 * is built, runs `ctas` persistent CTAs (a multiple of B; the caller sizes it to the SMs sampling leaves idle, see
 * pn_fps_launch_info, and passes min_smem_bytes so large that a CTA cannot share an SM with a sampling CTA), polls
 * the feed and writes out_idx rows plus done[b, s] = 1 as centroids appear, for the centroids s < s_end (the last few
 * are better left to the follow-up kernel, which has the whole GPU).  A CTA whose wait exceeds 3 ms gives up.
 * The caller then runs pn_ball_query_grid_f32 with the same `done` array after sampling: it computes whatever is
 * not done -- normally nothing -- so the result never depends on the two kernels having run side by side.
 * Limits: N <= 32768. */
int pn_fps_progress_f32(const float* xyz, int64_t sB, int64_t sN, int64_t sC, int B, int N, int npoint,
                        const int64_t* start_idx, int64_t* out_idx, uint64_t* progress, const pn_launch_opts* opts,
                        pn_stream_t stream);
/* farthest_point_sample over a cloud whose bucket workspace exists already (pn_ball_grid_build_f32 with any radius): the same
 * result as pn_fps_f32, bit for bit, computed with bucket pruning -- the cloud is read in cell order, so a warp's points are
 * spatially compact, and a warp skips its whole distance update whenever the lower bound of the new centroid's distance to the
 * warp's bounding box (evaluated with the distance's own fp32 rounding sequence, which is monotone) is not below the largest
 * running distance of the warp.  Points live in shared memory (16 B each, 12288 per CTA): 2 CTAs per cloud of 24000 points
 * instead of 4-8, for callers that keep several batches in flight and care about SM time rather than latency.
 * xyz / strides: the cloud the grid was built from (only the start points are read from it).  progress: as in
 * pn_fps_progress_f32, or NULL.  opts (tuning hooks): fps_threads = 512 -> 16 warps x 24 points per lane instead of 32 x 12,
 * fps_exchange = 1 -> no pruning.  Limits: N <= 49152. */
int pn_fps_sorted_f32(const float* xyz, int64_t sB, int64_t sN, int64_t sC, const void* grid, size_t grid_bytes, int B, int N,
                      int npoint, const int64_t* start_idx, int64_t* out_idx, uint64_t* progress, const pn_launch_opts* opts,
                      pn_stream_t stream);
/* Launch shape pn_fps_f32 would use for (B, N, npoint, opts): CTAs in the grid and dynamic shared memory per CTA. */
int pn_fps_launch_info(int B, int N, int npoint, const pn_launch_opts* opts, int* ctas, size_t* smem_bytes);
int pn_ball_query_stream_f32(const float* xyz, int64_t xB, int64_t xN, int64_t xC, const uint64_t* progress, int B, int N,
                             int S, int s_end, float radius2, int nsample, const void* grid, size_t grid_bytes, int ctas,
                             size_t min_smem_bytes, int32_t* done, int64_t* out_idx, pn_stream_t stream);

/* index_points (model/pointnet_util.py:43-60): out[b,m,:] = points[b, idx[b,m], :].
 * points [B,N,C] via strides, idx [B,M], out contiguous [B,M,C]. */
int pn_index_points_f32(const float* points, int64_t pB, int64_t pN, int64_t pC, int B, int N, int C,
                        const int64_t* idx, int64_t M, float* out, pn_stream_t stream);

/* Gather + recentre + concat of sample_and_group (model/pointnet_util.py:127-131, order
 * [xyz_rel, feat]) or of PointNetSetAbstractionMsg.forward (:243-247, msg_order=1: [feat, xyz_rel]).
 * feat may be NULL (D = 0).  out rows are (b,s,k) with 3+D channels and leading dimension ldo. */
int pn_group_f32(const float* xyz, int64_t xB, int64_t xN, int64_t xC, const float* feat, int64_t fB,
                 int64_t fN, int64_t fC, int D, const float* new_xyz, int64_t qB, int64_t qN, int64_t qC,
                 const int64_t* idx, int B, int N, int S, int K, int msg_order, float* out, int64_t ldo,
                 pn_stream_t stream);

/* One layer of a shared MLP: 1x1 Conv2d/Conv1d/Linear with BatchNorm already folded into (w, bias),
 * optional ReLU (model/pointnet_util.py:195-197, :253-255, :310-312; pointnet2.py:172-173;
 * pointnet.py passim).  y[b][r][co] = act(sum_ci x[b][r][ci] * w[b][co][ci] + bias[co]).
 * x rows have leading dimension ldx, batch stride x_bstride (elements); w is [cout,cin] row-major
 * with batch stride w_bstride (0 = shared; non-zero for the per-cloud transforms applied with
 * torch.bmm in pointnet.py:105-107); bias may be NULL, bias_bstride != 0 gives every batch item its
 * own bias (the global-feature half of PointNetSeg's 1088->512 conv folded per cloud,
 * pointnet.py:128-131, 247).  fp32 FMA accumulation. */
int pn_linear_f32(const float* x, int64_t ldx, int64_t x_bstride, const float* w, int64_t w_bstride,
                  const float* bias, int64_t bias_bstride, int relu, int B, int64_t rows, int cin, int cout,
                  float* y, int64_t ldy, int64_t y_bstride, pn_stream_t stream);

/* torch.max(new_points, 2)[0] (model/pointnet_util.py:199, :256) and the global max over points of
 * pointnet.py:35,74,122: y[g,:] = max over the K consecutive rows g*K .. g*K+K-1 of x. */
int pn_group_max_f32(const float* x, int64_t ldx, int64_t groups, int K, int C, float* y, int64_t ldy,
                     pn_stream_t stream);

/* 3-NN search + inverse-distance weights of PointNetFeaturePropagation.forward
 * (model/pointnet_util.py:295-300): idx [B,N,3] = the three sources with the smallest
 * sqdist(xyz1_n, xyz2_s) (ties: lowest index), weight [B,N,3] = (1/max(d,1e-10)) normalised. */
int pn_three_nn_f32(const float* xyz1, int64_t aB, int64_t aN, int64_t aC, const float* xyz2, int64_t bB,
                    int64_t bN, int64_t bC, int B, int N, int S, int64_t* idx, float* weight,
                    pn_stream_t stream);

/* The same 3-NN search as pn_three_nn_f32 (identical idx / weight, ties included), as an exact branch-and-bound:
 * pn_three_nn_blocks_build_f32 Morton-sorts the S <= 8192 coarse points of every cloud into blocks of 16 or 32 with
 * bounding boxes (blocks: caller-owned, opaque, 16-byte aligned, pn_three_nn_blocks_bytes(B, S) bytes); in
 * pn_three_nn_blocks_f32 one warp serves 32 fine points, visits the blocks nearest-first and stops when the nearest
 * unvisited block is farther than the warp's worst third-neighbour distance.  order (may be NULL): processing order
 * of the fine points as in pn_fp_mlp_bf16x3 -- pass the bucket order of the fine cloud (pn_ball_grid_order) so that
 * the 32 points of a warp are spatial neighbours and the pruning bites.  background = 1 caps the grid at ~3 small
 * CTAs per SM (persistent over the fine points) so that the search can run beside the kernels of another stream
 * without taking their registers / shared memory. */
size_t pn_three_nn_blocks_bytes(int B, int S);
int pn_three_nn_blocks_build_f32(const float* xyz2, int64_t bB, int64_t bN, int64_t bC, int B, int S, void* blocks,
                                 size_t blocks_bytes, pn_stream_t stream);
int pn_three_nn_blocks_f32(const float* xyz1, int64_t aB, int64_t aN, int64_t aC, const int32_t* order,
                           int64_t order_es, int64_t order_bs, const void* blocks, size_t blocks_bytes, int B, int N,
                           int S, int background, int64_t* idx, float* weight, pn_stream_t stream);

/* Weighted gather of model/pointnet_util.py:301 fused with the concat of :303-307:
 * out[b,n,0:D1] = points1[b,n,:] (skipped when points1 == NULL), out[b,n,D1:D1+D2] =
 * sum_k points2[b, idx[b,n,k], :] * weight[b,n,k].  out rows have leading dimension ldo. */
int pn_three_interpolate_f32(const float* points1, int64_t p1B, int64_t p1N, int64_t p1C, int D1,
                             const float* points2, int64_t p2B, int64_t p2N, int64_t p2C, int D2, int S,
                             const int64_t* idx, const float* weight, int B, int N, float* out, int64_t ldo,
                             int64_t o_bstride, pn_stream_t stream);

/* F.log_softmax over the channels of each row (pointnet2.py:174; pointnet.py:251). */
int pn_log_softmax_f32(const float* x, int64_t ldx, int64_t rows, int C, float* y, int64_t ldy,
                       pn_stream_t stream);
/* pred.argmax(-1) of the reference's evaluation loop (pcdseg.py:75) over rows of C <= 256 scores: one uint8 label per row,
 * the first maximum wins (torch.argmax).  What an evaluation loop needs of the [B, N, classes] log-probabilities: moving the
 * labels to the host instead costs 1 byte per point instead of 4 * classes. */
int pn_argmax_labels_u8(const float* x, int64_t ldx, int64_t rows, int C, uint8_t* labels, pn_stream_t stream);

/* ---- fused shared-MLP chains on the tensor cores (tcgen05 + TMEM), fp32 parity by 3-pass split bf16 ----
 * A chain is up to PN_MLP_MAX_LAYERS layers  y = act(x * w^T + bias)  with BatchNorm already folded into
 * (w, bias); relu[l] selects the activation.  Hidden layers are limited to 256 channels, the last layer to 1024.
 * The weights are pre-packed once (pn_mlp_pack_bf16x3) into a device blob of pn_mlp_blob_bytes() bytes:
 * per layer the bf16 hi and lo images in the UMMA shared-memory layout, then the fp32 bias table.
 * Products are computed as a_hi*w_hi + a_hi*w_lo + a_lo*w_hi with fp32 accumulation (relative error ~1e-5). */
#define PN_MLP_MAX_LAYERS 6
typedef struct pn_mlp_desc {
    int nlayers;
    int cin[PN_MLP_MAX_LAYERS];
    int cout[PN_MLP_MAX_LAYERS];
    int relu[PN_MLP_MAX_LAYERS];
} pn_mlp_desc;

/* Size of the packed blob; 0 (and an error string) if the chain is not supported. */
size_t pn_mlp_blob_bytes(const pn_mlp_desc* desc);
/* Warp groups (2 or 4) of the resident-weight kernel if the chain's packed weights fit in shared memory (and its layers in
 * the tile shapes of that kernel), else 0: the chain then streams its weights through a ring for every row tile.  A caller
 * with many row tiles can split such a chain into parts that do fit (the intermediate rows cost far less HBM traffic than
 * re-reading the weights per tile). */
int pn_mlp_resident_groups(const pn_mlp_desc* desc);
/* w[l]: device pointer to [cout[l], cin[l]] row-major fp32; bias[l]: device pointer or NULL.  The arrays w and
 * bias themselves live in HOST memory.  blob: 128-byte aligned device buffer. */
int pn_mlp_pack_bf16x3(const pn_mlp_desc* desc, const float* const* w, const float* const* bias, void* blob,
                       pn_stream_t stream);
/* The same with transposed[l] != 0 (host array, may be NULL) marking layers whose w[l] points to the TRANSPOSE of the
 * layer's weight, i.e. a row-major [cin[l], cout[l]] matrix.  The training step packs W^T this way for the input-gradient
 * GEMM dx = dy W (backward of a 1x1 conv) without materialising the transpose. */
int pn_mlp_pack_t_bf16x3(const pn_mlp_desc* desc, const float* const* w, const float* const* bias, const int* transposed,
                         void* blob, pn_stream_t stream);

/* Output modes of the fused chains. */
enum pn_mlp_out { PN_MLP_OUT_ROWS = 0, PN_MLP_OUT_MAX32 = 1, PN_MLP_OUT_LOG_SOFTMAX = 2 };

/* Plain rows: y = chain(x) for x [rows, cin[0]] (leading dimension ldx).  out_mode ROWS: y [rows, cout];
 * MAX32: y [rows/32, cout] = max over each run of 32 rows; LOG_SOFTMAX: y [rows, cout] log-probabilities.
 * (The per-point conv chains of model/pointnet.py.) */
int pn_mlp_rows_bf16x3(const pn_mlp_desc* desc, const void* blob, const float* x, int64_t ldx, int64_t rows,
                       int out_mode, float* y, int64_t ldy, const pn_launch_opts* opts, pn_stream_t stream);

/* One whole set-abstraction level after sampling (model/pointnet_util.py:127-131 + :194-199, or the MSG
 * branch :243-256 with msg_order = 1): gather + recentre + concat straight into the tensor-core operand,
 * the conv+BN+ReLU chain, and the max over the nsample rows of each group.  nsample = 16 or 32: out [B*S, cout_last]
 * rows with leading dimension ldo.  nsample = 32 m (64, 128, ...): the kernel pools runs of 32 rows, out has B*S*m rows
 * and the caller reduces every m consecutive rows (pn_group_max_f32).  Arguments as pn_group_f32. */
int pn_sa_mlp_max_bf16x3(const pn_mlp_desc* desc, const void* blob, const float* xyz, int64_t xB, int64_t xN,
                         int64_t xC, const float* feat, int64_t fB, int64_t fN, int64_t fC, int D,
                         const float* new_xyz, int64_t qB, int64_t qN, int64_t qC, const int64_t* idx, int B, int N,
                         int S, int K, int msg_order, float* out, int64_t ldo, const pn_launch_opts* opts,
                         pn_stream_t stream);
/* The same with the output mode chosen by the caller: PN_MLP_OUT_MAX32 as above, or PN_MLP_OUT_ROWS to keep the
 * [B*S*K, cout_last] rows (used when a level with few row tiles runs layer by layer: single-layer chains are
 * N-sliced over gridDim.y so that they fill the GPU). */
int pn_sa_mlp_bf16x3(const pn_mlp_desc* desc, const void* blob, const float* xyz, int64_t xB, int64_t xN,
                     int64_t xC, const float* feat, int64_t fB, int64_t fN, int64_t fC, int D,
                     const float* new_xyz, int64_t qB, int64_t qN, int64_t qC, const int64_t* idx, int B, int N,
                     int S, int K, int msg_order, int out_mode, float* out, int64_t ldo, const pn_launch_opts* opts,
                     pn_stream_t stream);

/* One feature-propagation level after the 3-NN search (model/pointnet_util.py:301-312): weighted gather of
 * the three coarse rows + skip concat straight into the tensor-core operand, then the conv+BN+ReLU chain.
 * With out_mode LOG_SOFTMAX and the segmentation head appended to the chain (pointnet2.py:172-175) the
 * log-probabilities [B, N, classes] are written directly.  out rows (b, n) have leading dimension ldo and
 * must be contiguous over the batch.  Arguments as pn_three_interpolate_f32.
 * relu_in = 1 (needs points1 == NULL): ReLU is applied to the interpolated channels before the chain.  This is how
 * a caller folds the level's FIRST layer into the coarse level -- interpolation is linear and its weights sum
 * to one, so conv(interp(p2)) + b == interp(conv(p2) + b): the caller runs that layer once over the S coarse
 * points (pn_mlp_rows_bf16x3, no ReLU), passes the result as points2 and drops the layer from the chain.
 * order (may be NULL): a permutation of the N points of every cloud -- tile row r of cloud b handles point
 * order[b*order_bs + r*order_es] (strides in int32 elements).  The result is the same; with a spatially sorted order
 * (pn_ball_grid_order) the rows of a warp share their three coarse neighbours and the gather hits in L1.
 * residual (may be NULL; chains of >= 2 layers): rows [B*N, ldr] added to the FIRST layer's pre-activation.  This is how
 * a caller takes the skip half of that layer off the critical path -- W [p1 ; interp] = W_a p1 + W_b interp: it computes
 * W_a p1 early (pn_mlp_rows_bf16x3, no bias, no ReLU; ldr = cout[0] rounded up to 32, 16-byte aligned), passes points1 =
 * NULL, D1 = 0 and a chain whose first layer holds only W_b. */
int pn_fp_mlp_bf16x3(const pn_mlp_desc* desc, const void* blob, const float* points1, int64_t p1B, int64_t p1N,
                     int64_t p1C, int D1, const float* points2, int64_t p2B, int64_t p2N, int64_t p2C, int D2, int S,
                     const int64_t* idx, const float* weight, int relu_in, const int32_t* order, int64_t order_es,
                     int64_t order_bs, const float* residual, int64_t ldr, int B, int N, int out_mode, float* out,
                     int64_t ldo, const pn_launch_opts* opts, pn_stream_t stream);

/* ================================================================================================================
 * Training step of PointNet2SemSeg (SURVEY.md section 8, row f-1; reference pcdseg.py:157-186) and evaluation
 * metrics (row f-2; pcdseg.py:58-97).  In train mode BatchNorm uses the statistics of the current batch, so a
 * layer is  pn_linear_f32 -> pn_bn_stats_f32 -> pn_bn_finalize_f32 -> pn_bn_act(_max)_f32  and every layer's
 * pre-normalisation output y is kept for the backward pass.  All matrices are row-major [rows, C] fp32 with a
 * leading dimension; the per-channel accumulators (sum, sumsq, s1, s2) are fp64 and must be ZEROED by the caller.
 * ================================================================================================================ */

/* Column sums of y and y*y in fp64 (nn.BatchNorm1d/2d in training mode, model/pointnet_util.py:196, :311,
 * pointnet2.py:172: the batch mean / biased variance over every row of the layer).  Atomically ADDED to sum / sumsq. */
int pn_bn_stats_f32(const float* y, int64_t ldy, int64_t rows, int C, double* sum, double* sumsq, pn_stream_t stream);
/* mean = sum/n, var = sumsq/n - mean^2 (biased), invstd = 1/sqrt(var+eps), scale = gamma*invstd, shift = beta -
 * mean*scale; running_mean/var (may be NULL) updated with `momentum` and the UNBIASED variance as torch does,
 * num_batches_tracked (may be NULL) incremented. */
int pn_bn_finalize_f32(const double* sum, const double* sumsq, int64_t n, int C, const float* gamma, const float* beta,
                       float eps, float momentum, float* running_mean, float* running_var,
                       int64_t* num_batches_tracked, float* scale, float* shift, float* mean, float* invstd,
                       pn_stream_t stream);
/* z = act(y*scale + shift)  (F.relu(bn(conv(x))), model/pointnet_util.py:197, :312). */
int pn_bn_act_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* scale, const float* shift, int relu,
                  float* z, int64_t ldz, pn_stream_t stream);
/* The same followed by torch.max over the K rows of each group (model/pointnet_util.py:199): out [groups, C],
 * argmax [groups, C] int32 = the first row of the group attaining the maximum (where the gradient is routed). */
int pn_bn_act_max_f32(const float* y, int64_t ldy, int64_t groups, int K, int C, const float* scale,
                      const float* shift, int relu, float* out, int64_t ldo, int32_t* argmax, pn_stream_t stream);
/* Backward of act(bn(y)), first pass: g = dz * [y*scale+shift > 0], xhat = (y-mean)*invstd; s1 += sum g,
 * s2 += sum g*xhat (fp64).  argmax != NULL: dz is the POOLED gradient [rows/K, C] and g[r] = dz[r/K] where
 * argmax[r/K] == r%K, 0 elsewhere (backward of torch.max). */
int pn_bn_bwd_stats_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* dz, int64_t lddz,
                        const int32_t* argmax, int K, const float* scale, const float* shift, const float* mean,
                        const float* invstd, int relu, double* s1, double* s2, pn_stream_t stream);
/* Second pass: dy = gamma*invstd*(g - s1/rows - xhat*s2/rows); dgamma += s2, dbeta += s1 (may be NULL; accumulated like
 * dw / db, so the caller zeroes them or passes the parameter's gradient buffer). */
int pn_bn_bwd_apply_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* dz, int64_t lddz,
                        const int32_t* argmax, int K, const float* scale, const float* shift, const float* mean,
                        const float* invstd, int relu, const double* s1, const double* s2, float* dy, int64_t lddy,
                        float* dgamma, float* dbeta, pn_stream_t stream);
/* Backward of act(bn(y)) when BatchNorm normalises with FIXED statistics (eval mode: scale, shift, mean, invstd from the
 * running mean / variance), in one pass: g = dz * [y*scale+shift > 0] (relu; argmax != NULL: routed from the pooled
 * gradient as in pn_bn_bwd_stats_f32), dy = scale*g, s1 += sum g, s2 += sum g*xhat with xhat = (y-mean)*invstd (fp64,
 * zeroed by the caller), then dgamma += s2, dbeta += s1 (either may be NULL; accumulated like pn_bn_bwd_apply_f32). */
int pn_bn_eval_bwd_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* dz, int64_t lddz,
                       const int32_t* argmax, int K, const float* scale, const float* shift, const float* mean,
                       const float* invstd, int relu, double* s1, double* s2, float* dy, int64_t lddy, float* dgamma,
                       float* dbeta, pn_stream_t stream);
/* Weight gradient of a 1x1 conv: dw[co,ci] += sum_r dy[r,co]*x[r,ci], db[co] += sum_r dy[r,co] (db may be NULL).
 * Split over the rows, accumulated with fp32 atomics: dw / db must be zeroed (or hold a gradient to add to). */
int pn_grad_weight_f32(const float* dy, int64_t lddy, const float* x, int64_t ldx, int64_t rows, int cout, int cin,
                       float* dw, int64_t lddw, float* db, pn_stream_t stream);
/* The same on the tensor cores (tcgen05, both operands from shared memory, 3-pass split bf16 with fp32 accumulation =
 * fp32 parity like the forward chains): a CTA owns a 128 x 128 tile of dw in TMEM and a slab of rows, converts dy / x to
 * bf16 hi + lo on the fly straight into the UMMA K-major layout, and adds its tile to dw with fp32 atomics. */
int pn_grad_weight_bf16x3(const float* dy, int64_t lddy, const float* x, int64_t ldx, int64_t rows, int cout, int cin,
                          float* dw, int64_t lddw, float* db, pn_stream_t stream);
/* The same with f(x) = act(x*x_scale[ci] + x_shift[ci]) applied to the x operand while it is loaded: the normalise + ReLU
 * of the layer that produced x, for a forward that kept only that layer's pre-normalisation output (pn_train_gemm_bf16x3). */
int pn_grad_weight_bn_bf16x3(const float* dy, int64_t lddy, const float* x, int64_t ldx, const float* x_scale,
                             const float* x_shift, int x_relu, int64_t rows, int cout, int cin, float* dw, int64_t lddw,
                             float* db, pn_stream_t stream);
/* One layer of the training forward (or the input-gradient GEMM of its backward) on the tensor cores with BatchNorm fused
 * on both sides: y[r,n] = sum_k f(x[r,k]) * W[n,k] + bias[n], f(v) = act(v*in_scale[k] + in_shift[k]) (in_scale NULL:
 * identity) = the normalise + ReLU of the PREVIOUS layer applied on load; col_sum / col_sumsq (fp64, may be NULL, ADDED to)
 * = the column sums of y and y*y for THIS layer's batch statistics (then pn_bn_finalize_f32).  w is [cout, cin] row-major,
 * or with w_transposed != 0 the transpose of a row-major [cin, cout] matrix (dx = dy W reads W that way).  3-pass split
 * bf16 with fp32 accumulation (fp32 parity).  Weights stay resident in shared memory: pn_train_gemm_supported(cin, cout)
 * tells whether the layer fits (cout <= 256, padded cin*cout*4 <= 128 KB); wider layers use pn_mlp_rows_bf16x3. */
int pn_train_gemm_supported(int cin, int cout);
/* w_scratch: caller-owned device buffer of pn_train_gemm_scratch_bytes(cin, cout) bytes, 128-byte aligned: the call first
 * converts the weights into it (bf16 hi + lo in the kernel's shared-memory layout), then every CTA fetches that image.
 * w == NULL: w_scratch already holds the image -- pn_train_pack_many converts the weights of MANY layers (a table of
 * pn_train_pack_item in DEVICE memory; `transposed` as w_transposed) in one launch, e.g. once per training iteration. */
typedef struct pn_train_pack_item {
    const float* w; /* [cout, cin] row-major, or its transpose [cin, cout] when transposed != 0 */
    void* out;      /* pn_train_gemm_scratch_bytes(cin, cout) bytes, 128-byte aligned */
    int cin, cout, transposed, reserved;
} pn_train_pack_item;
int pn_train_pack_many(const pn_train_pack_item* items, int n_items, int max_cin, int max_cout, pn_stream_t stream);
size_t pn_train_gemm_scratch_bytes(int cin, int cout);
int pn_train_gemm_bf16x3(const float* x, int64_t ldx, int64_t rows, int cin, const float* in_scale, const float* in_shift,
                         int in_relu, const float* w, int w_transposed, const float* bias, int cout, float* y, int64_t ldy,
                         double* col_sum, double* col_sumsq, void* w_scratch, pn_stream_t stream);
/* The input-gradient GEMM of the backward pass with the NEXT reduction fused into its epilogue: dz = dy W (w / w_transposed
 * as above; dz is the gradient w.r.t. the activated output of the layer below) and, from that layer's pre-normalisation
 * output prev_y [rows, cout] and batch constants, s1 += sum_r g, s2 += sum_r g*xhat with g = dz * [prev_y*scale+shift > 0],
 * xhat = (prev_y - mean)*invstd -- exactly what pn_bn_bwd_stats_f32 would compute in a pass of its own over dz and prev_y
 * (s1, s2: fp64 [cout], zeroed by the caller; then pn_bn_bwd_apply_f32). */
int pn_train_gemm_bnbwd_bf16x3(const float* dy, int64_t lddy, int64_t rows, int cin, const float* w, int w_transposed, int cout,
                               float* dz, int64_t lddz, const float* prev_y, int64_t ld_prev, const float* prev_scale,
                               const float* prev_shift, const float* prev_mean, const float* prev_invstd, double* s1, double* s2,
                               void* w_scratch, pn_stream_t stream);
/* The same input-gradient GEMM when the layer below normalises with FIXED statistics (eval-mode BatchNorm: its scale, shift,
 * mean, invstd from the running statistics): no batch coupling, so the epilogue stores that layer's dy_prev = scale*g
 * (g = (dy W) * [prev_y*scale+shift > 0]) instead of dy W -- exactly what pn_bn_eval_bwd_f32 would write in a pass of its own
 * -- adds sum g / sum g*xhat to s1 / s2 (fp64 [cout], zeroed by the caller), then dgamma += s2, dbeta += s1 (either may be
 * NULL). */
int pn_train_gemm_bneval_bf16x3(const float* dy, int64_t lddy, int64_t rows, int cin, const float* w, int w_transposed, int cout,
                                float* dy_prev, int64_t ld_dy_prev, const float* prev_y, int64_t ld_prev, const float* prev_scale,
                                const float* prev_shift, const float* prev_mean, const float* prev_invstd, double* s1, double* s2,
                                float* dgamma, float* dbeta, void* w_scratch, pn_stream_t stream);
/* out [cols, rows] = in [rows, cols]^T (the weight of the input-gradient GEMM dx = dy W = pn_linear_f32(dy, W^T)). */
int pn_transpose_f32(const float* in, int rows, int cols, float* out, pn_stream_t stream);
/* Backward of the gather of sample_and_group (model/pointnet_util.py:128-131): dfeat[b, idx[b,s,k], :] +=
 * dgrouped[(b,s,k), col0 : col0+D].  dfeat contiguous [B,N,D], zeroed by the caller.  (xyz carries no gradient.) */
int pn_group_bwd_f32(const float* dgrouped, int64_t ldg, int col0, int D, const int64_t* idx, int B, int N, int S,
                     int K, float* dfeat, pn_stream_t stream);
/* Backward of pn_three_interpolate_f32 (model/pointnet_util.py:301-307): dpoints1 [B,N,D1] = dx[:, :D1];
 * dpoints2[b, idx[b,n,k], :] += weight[b,n,k] * dx[(b,n), D1:].  dpoints2 contiguous [B,S,D2], zeroed by the caller. */
int pn_three_interpolate_bwd_f32(const float* dx, int64_t ldx, int D1, int D2, const int64_t* idx, const float* weight,
                                 int B, int N, int S, float* dpoints1, float* dpoints2, pn_stream_t stream);
/* Coordinate gradient of the gather + recentre of sample_and_group (model/pointnet_util.py:127-131; MSG :243-247; group-all
 * :151-156): dxyz[b, idx[b,s,k], :] += dgrouped[(b,s,k), col0 : col0+3] (the xyz_rel columns: col0 = 0 in sample_and_group
 * order, D in MSG order) and, for the in-place recentring, dnew_xyz[b,s,:] = -sum_k dgrouped[(b,s,k), col0 : col0+3]
 * (written; dnew_xyz = NULL for group-all, which is not recentred).  dxyz contiguous [B,N,3], zeroed by the caller;
 * dnew_xyz contiguous [B,S,3]. */
int pn_group_bwd_xyz_f32(const float* dgrouped, int64_t ldg, int col0, const int64_t* idx, int B, int N, int S, int K,
                         float* dxyz, float* dnew_xyz, pn_stream_t stream);
/* pn_three_interpolate_bwd_f32 plus the gradient w.r.t. the coordinates of both clouds, through the 3-NN weights of
 * model/pointnet_util.py:295-300 (dists = square_distance(xyz1, xyz2); dists[dists < 1e-10] = 1e-10; weight = 1/dists,
 * normalised).  points2 [B,S,D2] and xyz1 [B,N,3] / xyz2 [B,S,3] (element strides, like pn_three_nn_f32) are the forward's
 * inputs; the distances are recomputed with the 3-NN kernels' rounding sequence, so the clamp decision and 1/d are the
 * forward's.  A clamped distance passes no gradient.  dxyz1 [B,N,3] is written; dpoints2 [B,S,D2] and dxyz2 [B,S,3]
 * (contiguous) are accumulated into buffers the caller zeroed.  Needs S >= 3 (S == 1 is a broadcast without coordinate
 * gradient; S == 2 has no 3-NN forward). */
int pn_three_interpolate_bwd_xyz_f32(const float* dx, int64_t ldx, int D1, int D2, const int64_t* idx, const float* weight,
                                     const float* points2, int64_t p2B, int64_t p2S, int64_t p2C, const float* xyz1, int64_t aB,
                                     int64_t aN, int64_t aC, const float* xyz2, int64_t bB, int64_t bS, int64_t bC, int B, int N,
                                     int S, float* dpoints1, float* dpoints2, float* dxyz1, float* dxyz2, pn_stream_t stream);
/* ---- Deterministic variants (torch.use_deterministic_algorithms) -------------------------------------------------------
 * The same results as the entry points above, with every floating-point sum taken in an order that depends only on the
 * shapes and the device's SM count: two calls on the same inputs give bitwise-equal outputs.  Column / slab / block partials go
 * to a caller-provided workspace (16-byte aligned, at least the bytes the matching *_workspace_bytes helper returns; 0 there
 * means bad sizes) and are added in block order; scatter-adds go through an inverse index (CSR) built by pn_csr_build and are
 * pulled per destination in ascending slot order.  Accumulating outputs (sum, s1, dw, db, dgamma, ...) keep their semantics:
 * the ordered total is added to them once. */
size_t pn_bn_stats_workspace_bytes(int64_t rows, int C);
int pn_bn_stats_det_f32(const float* y, int64_t ldy, int64_t rows, int C, double* sum, double* sumsq, void* workspace,
                        size_t workspace_bytes, pn_stream_t stream);
int pn_bn_bwd_stats_det_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* dz, int64_t lddz,
                            const int32_t* argmax, int K, const float* scale, const float* shift, const float* mean,
                            const float* invstd, int relu, double* s1, double* s2, void* workspace, size_t workspace_bytes,
                            pn_stream_t stream);
/* (workspace: pn_bn_stats_workspace_bytes(rows, C)) */
int pn_bn_eval_bwd_det_f32(const float* y, int64_t ldy, int64_t rows, int C, const float* dz, int64_t lddz,
                           const int32_t* argmax, int K, const float* scale, const float* shift, const float* mean,
                           const float* invstd, int relu, double* s1, double* s2, float* dy, int64_t lddy, float* dgamma,
                           float* dbeta, void* workspace, size_t workspace_bytes, pn_stream_t stream);
/* Weight gradients: workspace = one fp32 tile per row slab (about SMs x the tile for the tensor-core engine). */
size_t pn_grad_weight_f32_workspace_bytes(int64_t rows, int cout, int cin);
size_t pn_grad_weight_bf16x3_workspace_bytes(int64_t rows, int cout, int cin);
int pn_grad_weight_det_f32(const float* dy, int64_t lddy, const float* x, int64_t ldx, int64_t rows, int cout, int cin,
                           float* dw, int64_t lddw, float* db, void* workspace, size_t workspace_bytes, pn_stream_t stream);
int pn_grad_weight_det_bf16x3(const float* dy, int64_t lddy, const float* x, int64_t ldx, int64_t rows, int cout, int cin,
                              float* dw, int64_t lddw, float* db, void* workspace, size_t workspace_bytes, pn_stream_t stream);
int pn_grad_weight_bn_det_bf16x3(const float* dy, int64_t lddy, const float* x, int64_t ldx, const float* x_scale,
                                 const float* x_shift, int x_relu, int64_t rows, int cout, int cin, float* dw, int64_t lddw,
                                 float* db, void* workspace, size_t workspace_bytes, pn_stream_t stream);
/* Inverse index of a gather: slot i (of B * slots_per_batch) names destination key(i) = (i / slots_per_batch) * n_dst +
 * clamp(idx[i], 0, n_dst - 1) (idx int32 or int64, idx_bits = 32 / 64).  offsets int32 [B*n_dst + 1]: the slots of key k are
 * slots[offsets[k] .. offsets[k+1]), in ascending order (slots int32 [n_slots]).  A stable radix sort of the keys: no limit on
 * how many slots one destination has.  workspace: pn_csr_workspace_bytes(n_slots, B * n_dst), 4-byte aligned. */
size_t pn_csr_workspace_bytes(int64_t n_slots, int64_t n_keys);
int pn_csr_build(const void* idx, int idx_bits, int64_t n_slots, int64_t slots_per_batch, int n_dst, int B, void* workspace,
                 size_t workspace_bytes, int32_t* offsets, int32_t* slots, pn_stream_t stream);
/* out[k, c] (contiguous [n_dst, D], written) = sum over the slots s of k in ascending order, sequentially in fp32 from 0, of
 * (weight ? weight[s] : 1) * src[(s / div) * ld + col0 + c]  -- what np.add.at accumulates. */
int pn_csr_pull_f32(const float* src, int64_t ld, int col0, int D, int div, const float* weight, const int32_t* offsets,
                    const int32_t* slots, int64_t n_dst, float* out, pn_stream_t stream);
/* pn_group_bwd_f32 through the CSR of idx (slots_per_batch = S*K, n_dst = N): dfeat [B,N,D] is written. */
int pn_group_bwd_det_f32(const float* dgrouped, int64_t ldg, int col0, int D, const int32_t* offsets, const int32_t* slots, int B,
                         int N, float* dfeat, pn_stream_t stream);
/* pn_group_bwd_xyz_f32 through the same CSR: dxyz [B,N,3] is written. */
int pn_group_bwd_xyz_det_f32(const float* dgrouped, int64_t ldg, int col0, const int64_t* idx, const int32_t* offsets,
                             const int32_t* slots, int B, int N, int S, int K, float* dxyz, float* dnew_xyz, pn_stream_t stream);
/* pn_three_interpolate_bwd_f32 through the CSR of the 3-NN idx (slots_per_batch = N*3, n_dst = S): dpoints2 is written. */
int pn_three_interpolate_bwd_det_f32(const float* dx, int64_t ldx, int D1, int D2, const float* weight, const int32_t* offsets,
                                     const int32_t* slots, int B, int N, int S, float* dpoints1, float* dpoints2,
                                     pn_stream_t stream);
/* pn_three_interpolate_bwd_xyz_f32 through the same CSR; workspace: fp32 [B*N*9] (the per-slot terms of dxyz2).  dpoints2
 * and dxyz2 are written. */
int pn_three_interpolate_bwd_xyz_det_f32(const float* dx, int64_t ldx, int D1, int D2, const int64_t* idx, const float* weight,
                                         const float* points2, int64_t p2B, int64_t p2S, int64_t p2C, const float* xyz1,
                                         int64_t aB, int64_t aN, int64_t aC, const float* xyz2, int64_t bB, int64_t bS,
                                         int64_t bC, int B, int N, int S, const int32_t* offsets, const int32_t* slots,
                                         float* workspace, float* dpoints1, float* dpoints2, float* dxyz1, float* dxyz2,
                                         pn_stream_t stream);
/* pn_cross_entropy_f32 with the loss summed per block and the blocks added in order; workspace replaces loss_sum. */
size_t pn_cross_entropy_workspace_bytes(int64_t rows);
int pn_cross_entropy_det_f32(const float* x, int64_t ldx, const int64_t* target, int64_t rows, int C, void* workspace,
                             size_t workspace_bytes, float* loss, float* dx, int64_t lddx, float grad_scale, pn_stream_t stream);
/* pn_chamfer_f32 (argmin NULL) or pn_chamfer_argmin_f32 with the total summed per block, blocks in order; total is written. */
size_t pn_chamfer_workspace_bytes(int B, int N);
int pn_chamfer_det_f32(const float* p1, int64_t aB, int64_t aN, int64_t aC, const float* p2, int64_t bB, int64_t bN, int64_t bC,
                       int B, int N, int M, int D, float* per_point, double* total, int32_t* argmin, void* workspace,
                       size_t workspace_bytes, pn_stream_t stream);
/* pn_chamfer_bwd_f32 through the CSR of argmin (int32, slots_per_batch = N, n_dst = M); workspace: fp32 [B*N*D].  dp2 is
 * written. */
int pn_chamfer_bwd_det_f32(const float* p1, int64_t aB, int64_t aN, int64_t aC, const float* p2, int64_t bB, int64_t bN,
                           int64_t bC, int B, int N, int M, int D, const int32_t* argmin, const float* g_total, float scale,
                           const int32_t* offsets, const int32_t* slots, float* workspace, float* dp1, float* dp2,
                           pn_stream_t stream);
/* pn_square_distance_bwd_f32 with one workspace slot per column chunk (rows) and per row tile (columns), added in order. */
size_t pn_square_distance_bwd_det_workspace_bytes(int B, int N, int M);
int pn_square_distance_bwd_det_f32(const float* g, int64_t gB, int64_t gN, const float* src, int64_t aB, int64_t aN, int64_t aC,
                                   const float* dst, int64_t bB, int64_t bN, int64_t bC, int B, int N, int M, void* workspace,
                                   size_t workspace_bytes, float* dsrc, float* ddst, pn_stream_t stream);
/* nn.Dropout(p) in training mode (pointnet2.py:172): y = x*keep/(1-p).  mask_in (bytes, dense [rows*C]) != NULL:
 * keep = mask_in -- also the backward pass.  Otherwise keep ~ Bernoulli(1-p) from a Philox4x32-10 stream keyed by
 * seed_offset[0] with counter offset seed_offset[1] (DEVICE memory, so a replayed CUDA graph sees fresh values) and
 * is written to mask_out (may be NULL). */
int pn_dropout_f32(const float* x, int64_t ldx, int64_t rows, int C, float p, const uint64_t* seed_offset,
                   const uint8_t* mask_in, uint8_t* mask_out, float* y, int64_t ldy, pn_stream_t stream);
/* nn.CrossEntropyLoss()(x^T, target) as pcdseg.py:177-178 applies it to the network's log-probabilities:
 * loss = mean_r (logsumexp(x_r) - x_r[target_r]); dx (may be NULL) = (softmax(x_r) - onehot) * grad_scale / n.
 * Rows with target -100 (ignore_index) are left out of the mean and get dx = 0; n counts the other rows (all rows
 * ignored: loss = NaN, like torch).  Any other target outside [0, C) makes the loss and that row of dx NaN.
 * loss_sum: two fp64 scratch words (sum, n), loss: one fp32 word (both device). */
int pn_cross_entropy_f32(const float* x, int64_t ldx, const int64_t* target, int64_t rows, int C, double* loss_sum,
                         float* loss, float* dx, int64_t lddx, float grad_scale, pn_stream_t stream);
/* Backward of F.log_softmax (pointnet2.py:174): dx = dy - exp(y)*sum_c dy, y = the log-probabilities. */
int pn_log_softmax_bwd_f32(const float* dy, int64_t lddy, const float* y, int64_t ldy, int64_t rows, int C, float* dx,
                           int64_t lddx, pn_stream_t stream);
/* torch.optim.Adam(lr, betas, eps, weight_decay) of pcdseg.py:136-141 on one flat fp32 buffer: g = grad*grad_scale +
 * weight_decay*p; m, v updated; p -= lr/(1-beta1^step) * m / (sqrt(v)/sqrt(1-beta2^step) + eps).  step >= 1.
 * grad_scale = 1/world_size after a summing all-reduce. */
int pn_adam_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                float beta2, float eps, float weight_decay, int64_t step, float grad_scale, pn_stream_t stream);
/* The same update with the learning rate (*lr) and the step count (*step, incremented first: start it at 0) in DEVICE
 * memory, so that a captured CUDA graph replays with the current values. */
int pn_adam_dev_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, const float* lr,
                    int64_t* step, float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                    pn_stream_t stream);
/* test_kitti_semseg's inner loop (pcdseg.py:72-83) without host round trips: pred (may be NULL) [rows] = argmax over
 * the C <= 64 classes; counts int64 [3C+1] (overwritten) = per class intersection | predicted | target, then the
 * number of correct points. */
int pn_seg_metrics_f32(const float* logp, int64_t ldx, const int64_t* target, int64_t rows, int C, int64_t* pred,
                       int64_t* counts, pn_stream_t stream);
/* Folds one batch's counts into the running totals as the reference's Python does: ious[c] += (U == 0 ? 1 : I/U)
 * (double division rounded to fp32, added in fp32), count[c] += 1, acc_sum += correct/points (fp64), batches += 1. */
int pn_seg_metrics_accumulate(const int64_t* counts, int C, int64_t points, float* ious, uint32_t* count,
                              double* acc_sum, int64_t* batches, pn_stream_t stream);

/* ================================================================================================================
 * Raw SemanticKITTI scans -> network input (SURVEY.md section 8, row f-3): Semantic_KITTI_Utils.get
 * (data_utils/kitti_utils.py:183-227) + SemKITTI_Loader.__getitem__ (data_utils/SemKITTI_Loader.py:91-115).
 * points: B scans concatenated, float32 x 4 per point (x, y, z, reflectance: the .bin wire format), 16-byte aligned;
 * raw_label: uint32 per point (.label: semantic id in the low 16 bits); offsets: int64 [B+1] (device) = first point of
 * every scan; lut: uint8 [lut_size] = the learning_map of config/semantic-kitti.yaml as a table (ids beyond it -> 0).
 * ================================================================================================================ */
size_t pn_scan_workspace_bytes(int B, int64_t max_points);
/* Keep flag per point -- learning_map[label] != 0 (kitti_utils.py:213-218) and, with inview != 0, the field-of-view
 * test of points_basic_filter (:262-280): h_lo < atan2(y, x) < h_hi, v_lo < atan2(z, sqrt(x^2+y^2+z^2)) < v_hi in fp32
 * (the caller passes the bounds as the fp32 values of -/+40 deg and -/+20 deg in radians) and |x|,|y|,|z|,d < 10000 --
 * then an ORDER-PRESERVING compaction: kept[offsets[b] + i] = index inside scan b of its i-th kept point,
 * kept_count[b] = how many.  max_points (host) = the longest scan, for the grid size. */
int pn_scan_filter_f32(const float* points, const uint32_t* raw_label, const int64_t* offsets, int B, int64_t max_points,
                       const uint8_t* lut, int lut_size, int inview, float h_lo, float h_hi, float v_lo, float v_hi,
                       int32_t* kept, int32_t* kept_count, void* workspace, size_t workspace_bytes, pn_stream_t stream);
/* out [B, 4, npoints] (channel-major, what PointNet2SemSeg.forward takes after pcdseg.py:167's transpose) and labels
 * int64 [B, npoints] (learning_map[label] - 1): point j of scan b is kept point choice[b*npoints + j] of that scan
 * (np.random.choice(length, npoints, replace=True), SemKITTI_Loader.py:110-113), normalised and clipped
 * (pcd_normalize, :23-30) plus noise[(offsets[b] + i)*4 .. +3] (pcd_jitter, :17-21: one fp32 4-vector per KEPT point,
 * already scaled and clipped by the caller; NULL = none).  choice == NULL: indices, and with sigma > 0 the jitter
 * clip(sigma*N(0,1), -clip, clip), are drawn from the Philox4x32-10 stream seed_offset = {seed, offset} (device memory). */
int pn_scan_sample_f32(const float* points, const uint32_t* raw_label, const int64_t* offsets, int B, const uint8_t* lut,
                       int lut_size, const int32_t* kept, const int32_t* kept_count, int npoints, const int64_t* choice,
                       const float* noise, float sigma, float clip, const uint64_t* seed_offset, float* out,
                       int64_t* labels, pn_stream_t stream);

/* ---- row f-4 helpers ------------------------------------------------------------------------------------------- */
/* chamfer_batch / chamfer_non_batch (model/chamfer.py:7-53): per_point [B,N] (may be NULL) = min_m ||p1[b,n] - p2[b,m]||_2,
 * *total (fp64, device, overwritten) = their sum; the reference divides by B.  Clouds via strides, D <= 8 coordinates. */
int pn_chamfer_f32(const float* p1, int64_t aB, int64_t aN, int64_t aC, const float* p2, int64_t bB, int64_t bN, int64_t bC,
                   int B, int N, int M, int D, float* per_point, double* total, pn_stream_t stream);
/* pn_chamfer_f32 that also writes argmin [B,N] (int32, device) = the index m of the nearest p2 point, the first of equal
 * minima (torch's min(dim) on the CPU), for the backward pass; per_point and *total are pn_chamfer_f32's. */
int pn_chamfer_argmin_f32(const float* p1, int64_t aB, int64_t aN, int64_t aC, const float* p2, int64_t bB, int64_t bN,
                          int64_t bC, int B, int N, int M, int D, float* per_point, double* total, int32_t* argmin,
                          pn_stream_t stream);
/* Backward of chamfer_batch / chamfer_non_batch (model/chamfer.py:7-53: norm -> min -> sum): per p1 point, r = p1[b,n] -
 * p2[b,a] with a = argmin[b,n] of pn_chamfer_argmin_f32, d = ||r|| recomputed in the forward's rounding sequence,
 * c = (*g_total) * scale / d, and 0 where d == 0 (torch's norm backward).  dp1 [B,N,D] = c r (written);
 * dp2[b,a] -= c r into a contiguous [B,M,D] buffer the caller zeroed (fp32 atomics).  Either output may be NULL.
 * g_total: the fp32 gradient of the loss (device); scale = 1/B for chamfer_batch, 1 for chamfer_non_batch.  D <= 8. */
int pn_chamfer_bwd_f32(const float* p1, int64_t aB, int64_t aN, int64_t aC, const float* p2, int64_t bB, int64_t bN, int64_t bC,
                       int B, int N, int M, int D, const int32_t* argmin, const float* g_total, float scale, float* dp1,
                       float* dp2, pn_stream_t stream);
/* SemKITTI_2_Common.__call__ (data_utils/kitti_utils.py:97-110): y[r, j] = max(x[r, src0[j]], x[r, src1[j]]) for j < n_out
 * (src1[j] == src0[j] for classes that are not merged); src0 / src1 are device int32 [n_out], indices < n_in. */
int pn_class_merge_f32(const float* x, int64_t ldx, int64_t rows, int n_in, int n_out, const int* src0, const int* src1,
                       float* y, pn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PN12_B200_H */
