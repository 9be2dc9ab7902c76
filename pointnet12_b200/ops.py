"""Tensor-level wrappers over the C ABI: allocate outputs with torch, pass raw pointers and strides.

PyTorch is used here for device memory and streams only.  CUDA float32 tensors in, CUDA tensors out;
CPU tensors raise (there is no CPU fallback).  Strided (permuted) point clouds are passed through
unchanged -- the kernels take element strides, like the reference's functions take views.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import List, Optional, Sequence, Tuple

import torch

from . import _native as nv


def _need_cuda(t: torch.Tensor, name: str) -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(
            f"{name} is a {t.device} tensor: pointnet12_b200 runs on CUDA (sm_100a) only and has no CPU fallback")


def _f32(t: torch.Tensor, name: str) -> torch.Tensor:
    _need_cuda(t, name)
    return t if t.dtype == torch.float32 else t.float()


def _i64(t: torch.Tensor, name: str) -> torch.Tensor:
    _need_cuda(t, name)
    t = t if t.dtype == torch.int64 else t.long()
    return t if t.is_contiguous() else t.contiguous()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _cloud(t: torch.Tensor, name: str, channels: Optional[int] = None) -> torch.Tensor:
    t = _f32(t, name)
    if t.dim() != 3:
        raise ValueError(f"{name} must be [B, N, C], got shape {tuple(t.shape)}")
    if channels is not None and t.shape[2] != channels:
        raise ValueError(f"{name} must have {channels} channels in its last dimension, got {t.shape[2]}")
    return t


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class _on_device:
    """Make the tensor's device current for the duration of a launch (no-op in the common case)."""

    def __init__(self, t: torch.Tensor):
        self.idx = t.device.index
        self.ctx = None

    def __enter__(self):
        if self.idx != torch.cuda.current_device():
            self.ctx = torch.cuda.device(self.idx)
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)


def device_check() -> Tuple[int, int, int]:
    import ctypes as C

    sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
    nv.call("pn_device_check", C.byref(sm), C.byref(ma), C.byref(mi))
    return sm.value, ma.value, mi.value


# ------------------------------------------------------------------------------------------------
# Launch options.  The C ABI keeps no process-wide settings: everything that tunes a launch travels with the call in a
# pn_launch_opts.  Here the settings live in a process-wide default plus a per-THREAD override (`options(...)`), so two
# Python threads can run, say, the fp32-parity and the single-pass bf16 precision at the same time.
_tls = threading.local()
_DEFAULTS = {
    "precision": "bf16x3",      # 'bf16x3' | 'bf16' | 'fp32'  (set_mlp_mode)
    "mlp_engine": 0,            # pn_launch_opts.mlp_engine flags (set_mlp_engine)
    "reserved_sms": 0,          # SMs the resident-weight chain launches leave to other streams
    "fps_config": (0, 0, 0),    # (cluster size, threads per CTA, exchange) of pn_fps_f32; 0 = automatic
    "mlp_debug": None,          # device pointer of the chain timeline buffer
    "tile_counters": None,      # TileCounters: resident chains draw their tiles dynamically (see TileCounters)
    "fps1_config": None,        # launch shape of the LEVEL-1 sampling of PointNet2SemSeg (None = automatic); PN12_FPS1 overrides
    "stream_ball": True,        # level-1 ball query answered beside the sampling (False: after it); PN12_STREAM_BALL overrides
    "nn1_background": True,     # fp1's 3-NN search on a capped grid (see nn1_background)
    "reserve_level2": True,     # sa1 / sa2 leave the level-2 sampling's SMs out of their grids
    "host_out_slices": None,    # batch slices of the last level when the output goes to the host (None: HOST_OUT_SLICES)
    "fps1_sorted": None,        # level-1 sampling through the bucket-pruned kernel (fps_sorted) with this config; PN12_FPS1_SORTED overrides
}


def _opt(name: str):
    return getattr(_tls, name, _DEFAULTS[name])


class options:
    """with ops.options(precision="bf16", fps_config=(4, 256, 2)): ...  -- overrides for the calling thread only."""

    def __init__(self, **kw):
        for k in kw:
            if k not in _DEFAULTS:
                raise TypeError(f"unknown option {k!r}; known: {sorted(_DEFAULTS)}")
        if "precision" in kw and kw["precision"] not in ("bf16x3", "bf16", "fp32"):
            raise ValueError("precision must be 'bf16x3', 'bf16' or 'fp32'")
        self.kw, self.old = kw, {}

    def __enter__(self):
        missing = object()
        for k, v in self.kw.items():
            self.old[k] = getattr(_tls, k, missing)
            setattr(_tls, k, v)
        self.missing = missing
        return self

    def __exit__(self, *exc):
        for k, v in self.old.items():
            if v is self.missing:
                delattr(_tls, k)
            else:
                setattr(_tls, k, v)


class TileCounters:
    """A pool of zeroed uint32 words for pn_launch_opts.tile_counter.  Inside `with ops.options(tile_counters=pool)`
    every resident-weight chain launch takes the next word and hands out its row tiles through it (dynamic scheduling):
    CTAs whose SM is held by another stream's kernel when the launch begins only take what is left.  The kernel resets
    its word before it ends, so a captured CUDA graph can be replayed; launches that may run at the same time must not
    share a word, hence one pool per graph."""

    def __init__(self, device, n: int = 64):
        self.buf = torch.zeros((n,), dtype=torch.int32, device=device)
        self.used = 0

    def take(self) -> int:
        if self.used >= self.buf.numel():
            raise RuntimeError("TileCounters: pool exhausted")
        self.used += 1
        return self.buf.data_ptr() + 4 * (self.used - 1)


def _launch_opts(dynamic_tiles: bool = False, fps_config=None) -> "nv.LaunchOpts":
    o = nv.LaunchOpts()
    o.mlp_passes = 1 if _opt("precision") == "bf16" else 3
    o.mlp_engine = _opt("mlp_engine")
    o.reserved_sms = _opt("reserved_sms")
    o.fps_cluster, o.fps_threads, o.fps_exchange = fps_config if fps_config is not None else _opt("fps_config")
    o.mlp_debug = _opt("mlp_debug")
    pool = _opt("tile_counters")
    o.tile_counter = pool.take() if (dynamic_tiles and pool is not None) else None
    return o


def fps_set_config(cluster_size: int = 0, threads: int = 0, exchange: int = 0) -> None:
    """Tuning hook (process default): cluster size, threads per CTA, exchange (1 = barrier.cluster, 2 = st.async, 3 = st.async
    without the z table); 0 = automatic.  Per thread / per call: options(fps_config=...) / fps(..., config=...)."""
    _DEFAULTS["fps_config"] = (int(cluster_size), int(threads), int(exchange))


# ------------------------------------------------------------------------------------------------
def fps(xyz: torch.Tensor, npoint: int, start_idx: torch.Tensor, progress: Optional[torch.Tensor] = None,
        config: Optional[Tuple[int, int, int]] = None) -> torch.Tensor:
    """farthest_point_sample (pointnet_util.py:63-84); start_idx [B] int64 on the device.
    progress: a ZEROED int64 [B, npoint] tensor -> the kernel also publishes every centroid as it is chosen
    (index << 32 | 1), for consumers running beside it (ball_query_stream).
    config: (cluster size, threads per CTA, exchange) for this call (default: options / fps_set_config; 0 = automatic)."""
    xyz = _cloud(xyz, "xyz", 3)
    B, N, _ = xyz.shape
    start_idx = _i64(start_idx, "start_idx")
    if start_idx.shape != (B,):
        raise ValueError(f"start_idx must have shape ({B},), got {tuple(start_idx.shape)}")
    out = torch.empty((B, int(npoint)), dtype=torch.int64, device=xyz.device)
    lo = _launch_opts(fps_config=config)
    with _on_device(xyz):
        if progress is None:
            nv.call("pn_fps_f32", xyz.data_ptr(), *xyz.stride(), B, N, int(npoint), start_idx.data_ptr(), out.data_ptr(),
                    C.byref(lo), _stream(), tag=(B, N, int(npoint)))
        else:
            if progress.shape != (B, int(npoint)) or progress.dtype != torch.int64 or not progress.is_contiguous():
                raise ValueError("progress must be a contiguous int64 [B, npoint] tensor")
            nv.call("pn_fps_progress_f32", xyz.data_ptr(), *xyz.stride(), B, N, int(npoint), start_idx.data_ptr(),
                    out.data_ptr(), progress.data_ptr(), C.byref(lo), _stream(), tag=(B, N, int(npoint)))
    return out


def fps_sorted(xyz: torch.Tensor, grid: "BallGrid", npoint: int, start_idx: torch.Tensor,
               progress: Optional[torch.Tensor] = None, config: Optional[Tuple[int, int, int]] = None) -> torch.Tensor:
    """farthest_point_sample with bucket pruning (pn_fps_sorted_f32): identical indices to fps(), computed from the cell-sorted
    copy of the cloud inside `grid` (any radius); 2 CTAs per cloud of up to 24576 points.  For throughput (several batches in
    flight), not latency."""
    xyz = _cloud(xyz, "xyz", 3)
    B, N, _ = xyz.shape
    if (grid.B, grid.N) != (B, N):
        raise ValueError("grid was built for another cloud shape")
    start_idx = _i64(start_idx, "start_idx")
    if start_idx.shape != (B,):
        raise ValueError(f"start_idx must have shape ({B},), got {tuple(start_idx.shape)}")
    out = torch.empty((B, int(npoint)), dtype=torch.int64, device=xyz.device)
    with _on_device(xyz):
        nv.call("pn_fps_sorted_f32", xyz.data_ptr(), *xyz.stride(), grid.buf.data_ptr(), grid.nbytes, B, N, int(npoint),
                start_idx.data_ptr(), out.data_ptr(), _p(progress), C.byref(_launch_opts(fps_config=config)), _stream(),
                tag=(B, N, int(npoint)))
    return out


FPS_SORTED_MAX_POINTS = 4 * 16 * 24 * 32


def fps_launch_info(B: int, N: int, npoint: int, config: Optional[Tuple[int, int, int]] = None) -> Tuple[int, int]:
    """(CTAs, dynamic shared memory per CTA) of the sampling launch for this shape."""
    ctas, smem = C.c_int(), C.c_size_t()
    lo = _launch_opts(fps_config=config)
    nv.check(nv.lib().pn_fps_launch_info(int(B), int(N), int(npoint), C.byref(lo), C.byref(ctas), C.byref(smem)),
             "pn_fps_launch_info")
    return ctas.value, smem.value


# Skip half of an FP level's first layer computed early on a side stream (PointNetFeaturePropagation.skip_ahead).  Measured at
# C2: fp4 40 -> 35, fp3 34 -> 31 us, but the three extra launches contend with sa3 / sa4 and the step got 15 us SLOWER
# (0.890 vs 0.875 ms), so it is off by default.
FP_SKIP_AHEAD = os.environ.get("PN12_FP_SKIP_AHEAD", "0") != "0"
FP1_BUCKET_ORDER = os.environ.get("PN12_FP1_ORDER", "0") != "0"   # fp1 walks the fine points in bucket order (helped the row-per-thread gather: 195 -> 183 us; with the quad producer it costs 0.6 %: scattered index / output rows)
HOST_OUT_SLICES = int(os.environ.get("PN12_HOST_OUT_SLICES", "8"))   # batch slices of the last level when the output goes to the host
def stream_ball_query() -> bool:      # PN12_STREAM_BALL=0: the level-1 ball query runs after sampling instead of beside it
    v = os.environ.get("PN12_STREAM_BALL", "")
    return (v != "0") if v else bool(_opt("stream_ball"))


STREAM_BALL_MIN_FREE_SMS = 32    # SMs the sampling launch must leave idle for the streamed ball query to be worth it
# Tuning knobs of the level-1 stage (read per forward, so a benchmark can sweep them inside one process):
#   PN12_FPS1="cluster,threads,exchange"  launch shape of the level-1 sampling (default: automatic = 8 CTAs x 4 warps per cloud)
#   PN12_STREAM_BALL_CTAS=n               persistent CTAs of the streamed ball query (default: every SM sampling leaves idle)
#   PN12_STREAM_BALL_SHARE=1              let those CTAs share an SM with a sampling CTA (default: shared memory sized to forbid it)
def fps1_config() -> Optional[Tuple[int, int, int]]:
    v = os.environ.get("PN12_FPS1", "")
    return tuple(int(t) for t in v.split(",")) if v else _opt("fps1_config")


def nn1_background() -> bool:
    """fp1's 3-NN block search on a capped grid (~3 small CTAs per SM) so that the chains of the critical path find room beside
    it (one batch at a time), or on its full grid (option / PN12_NN1_BACKGROUND=0)."""
    v = os.environ.get("PN12_NN1_BACKGROUND", "")
    return (v != "0") if v else bool(_opt("nn1_background"))


def reserve_level2_sms() -> bool:
    """sa1 / sa2 leave the SMs of the concurrent level-2 sampling out of their persistent grids (PN12_RESERVE_L2=0: do not)."""
    v = os.environ.get("PN12_RESERVE_L2", "")
    return (v != "0") if v else bool(_opt("reserve_level2"))


def host_out_slices() -> int:
    v = _opt("host_out_slices")
    return HOST_OUT_SLICES if v is None else int(v)


def fps1_sorted() -> Optional[Tuple[int, int, int]]:
    v = os.environ.get("PN12_FPS1_SORTED", "")
    if v == "0":
        return None
    return tuple(int(t) for t in v.split(",")) if v else _opt("fps1_sorted")


def stream_ball_ctas(free_sms: int, B: int) -> int:
    v = int(os.environ.get("PN12_STREAM_BALL_CTAS", "0"))
    return (v if v > 0 else free_sms) // B * B


def stream_ball_share() -> bool:
    return os.environ.get("PN12_STREAM_BALL_SHARE", "0") != "0"


STREAM_BALL_TAIL = int(os.environ.get("PN12_STREAM_BALL_TAIL", "0"))    # last centroids per cloud left to the follow-up query (measured at C2: 0 is best, 0.891 vs 0.905-0.918 ms with 16..128)


def ball_query_stream(radius: float, nsample: int, xyz: torch.Tensor, grid: "BallGrid", progress: torch.Tensor,
                      done: torch.Tensor, out: torch.Tensor, ctas: int, min_smem: int, tail: Optional[int] = None) -> None:
    """Answers the ball queries of the centroids a RUNNING fps(..., progress=...) publishes (pn_ball_query_stream_f32);
    call it on another stream than the sampling.  done int32 [B, S] (zeroed), out int64 [B, S, nsample]."""
    xyz = _cloud(xyz, "xyz", 3)
    B, N, _ = xyz.shape
    S = progress.shape[1]
    with _on_device(xyz):
        s_end = max(0, S - (STREAM_BALL_TAIL if tail is None else int(tail)))
        nv.call("pn_ball_query_stream_f32", xyz.data_ptr(), *xyz.stride(), progress.data_ptr(), B, N, S, s_end, float(radius ** 2),
                int(nsample), grid.buf.data_ptr(), grid.nbytes, int(ctas), int(min_smem), done.data_ptr(), out.data_ptr(),
                _stream())


def square_distance(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    """pointnet_util.py:19-40 -> [B, N, M]."""
    src, dst = _cloud(src, "src", 3), _cloud(dst, "dst", 3)
    B, N, _ = src.shape
    M = dst.shape[1]
    out = torch.empty((B, N, M), dtype=torch.float32, device=src.device)
    with _on_device(src):
        nv.call("pn_square_distance_f32", src.data_ptr(), *src.stride(), dst.data_ptr(), *dst.stride(), B, N, M,
                out.data_ptr(), _stream())
    return out


def square_distance_backward(g: torch.Tensor, src: torch.Tensor, dst: torch.Tensor, need_src: bool = True,
                             need_dst: bool = True) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """Backward of square_distance (pn_square_distance_bwd_f32): g [B, N, M] = dL/ddist (any batch and row strides; a
    view whose columns are not contiguous is copied first), src [B, N, 3], dst [B, M, 3] (any strides) -> (dsrc [B, N, 3]
    or None, ddst [B, M, 3] or None), computed for the sides asked for."""
    src, dst = _cloud(src, "src", 3), _cloud(dst, "dst", 3)
    B, N, _ = src.shape
    M = dst.shape[1]
    g = _f32(g, "g")
    if tuple(g.shape) != (B, N, M):
        raise ValueError(f"g must have shape ({B}, {N}, {M}), got {tuple(g.shape)}")
    if not (need_src or need_dst):
        return None, None
    if g.stride(2) != 1 and M > 1:
        g = g.contiguous()
    dsrc = torch.empty((B, N, 3), dtype=torch.float32, device=src.device) if need_src else None
    ddst = torch.empty((B, M, 3), dtype=torch.float32, device=src.device) if need_dst else None
    ws = torch.empty((4 * B * (N + M),), dtype=torch.float32, device=src.device)
    with _on_device(src):
        nv.call("pn_square_distance_bwd_f32", g.data_ptr(), g.stride(0), g.stride(1), src.data_ptr(), *src.stride(),
                dst.data_ptr(), *dst.stride(), B, N, M, ws.data_ptr(), _p(dsrc), _p(ddst), _stream())
    return dsrc, ddst


GRID_MIN_POINTS = 4096     # below this the ordered scan of pn_ball_query_f32 is already short


class BallGrid:
    """Uniform-grid buckets of a batch of clouds for one radius (pn_ball_grid_build_f32).  Depends on xyz and the
    radius only, so it can be built on a side stream while farthest-point sampling runs."""

    def __init__(self, xyz: torch.Tensor, radius: float):
        xyz = _cloud(xyz, "xyz", 3)
        B, N, _ = xyz.shape
        self.B, self.N, self.r2 = B, N, float(radius ** 2)
        self.nbytes = int(nv.lib().pn_ball_grid_bytes(B, N))
        self.buf = torch.empty((self.nbytes,), dtype=torch.uint8, device=xyz.device)
        with _on_device(xyz):
            nv.call("pn_ball_grid_build_f32", xyz.data_ptr(), *xyz.stride(), B, N, self.r2, self.buf.data_ptr(),
                    self.nbytes, _stream())


    def order(self) -> Tuple[int, int, int]:
        """(device pointer, element stride, batch stride) of the bucket-sorted point order, in int32 elements."""
        ptr, es, bs = C.c_void_p(), C.c_int64(), C.c_int64()
        nv.check(nv.lib().pn_ball_grid_order(self.buf.data_ptr(), self.N, C.byref(ptr), C.byref(es), C.byref(bs)),
                 "pn_ball_grid_order")
        return ptr.value, es.value, bs.value


def ball_grid(xyz: torch.Tensor, radius: float) -> BallGrid:
    return BallGrid(xyz, radius)


def ball_query(radius: float, nsample: int, xyz: torch.Tensor, new_xyz: torch.Tensor,
               grid: Optional[BallGrid] = None, method: str = "auto", threshold: Optional[int] = None,
               done: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """query_ball_point (pointnet_util.py:87-107) -> int64 [B, S, nsample].
    method: "auto" (grid buckets for N >= GRID_MIN_POINTS, ordered scan below), "scan" (pn_ball_query_f32),
    "grid" / "grid-cells" / "grid-scan" (pn_ball_query_grid_f32 with the automatic threshold / every query through
    the cells / every query through the per-warp scan).  All return identical indices.
    done / out: int32 [B, S] flags of rows ball_query_stream has already written into `out`; only the others are computed."""
    xyz, new_xyz = _cloud(xyz, "xyz", 3), _cloud(new_xyz, "new_xyz", 3)
    B, N, _ = xyz.shape
    S = new_xyz.shape[1]
    if out is None:
        out = torch.empty((B, S, int(nsample)), dtype=torch.int64, device=xyz.device)
    elif out.shape != (B, S, int(nsample)) or out.dtype != torch.int64 or not out.is_contiguous():
        raise ValueError("out must be a contiguous int64 [B, S, nsample] tensor")
    if done is not None and (method not in ("auto", "grid") or grid is None):
        raise ValueError("done= (rows finished by ball_query_stream) needs the grid method")
    r2 = float(radius ** 2)  # the reference compares against the python scalar radius ** 2 (cast to fp32 by torch)
    if method == "auto":
        method = "grid" if (grid is not None or N >= GRID_MIN_POINTS) else "scan"
    with _on_device(xyz):
        if method == "scan":
            nv.call("pn_ball_query_f32", xyz.data_ptr(), *xyz.stride(), new_xyz.data_ptr(), *new_xyz.stride(), B, N, S,
                    r2, int(nsample), out.data_ptr(), _stream())
            return out
        if method not in ("grid", "grid-cells", "grid-scan"):
            raise ValueError(f"unknown ball query method {method!r}")
        if grid is None:
            grid = BallGrid(xyz, radius)
        elif (grid.B, grid.N) != (B, N) or grid.r2 != r2:
            raise ValueError("grid was built for another cloud shape or radius")
        if threshold is None:
            threshold = {"grid": int(os.environ.get("PN12_BQ_THRESHOLD", "0")), "grid-cells": 2 ** 31 - 1, "grid-scan": -1}[method]
        nv.call("pn_ball_query_grid_f32", xyz.data_ptr(), *xyz.stride(), new_xyz.data_ptr(), *new_xyz.stride(), B, N, S,
                r2, int(nsample), grid.buf.data_ptr(), grid.nbytes, threshold, _p(done), out.data_ptr(), _stream())
    return out


def index_points(points: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """pointnet_util.py:43-60: points [B,N,C], idx [B, ...] -> [B, ..., C]."""
    points = _cloud(points, "points")
    idx = _i64(idx, "idx")
    B, N, Cc = points.shape
    if idx.shape[0] != B:
        raise ValueError("idx and points disagree on the batch size")
    M = idx[0].numel()
    out = torch.empty(tuple(idx.shape) + (Cc,), dtype=torch.float32, device=points.device)
    if M:
        with _on_device(points):
            nv.call("pn_index_points_f32", points.data_ptr(), *points.stride(), B, N, Cc, idx.data_ptr(), M,
                    out.data_ptr(), _stream())
    return out


def group(xyz: torch.Tensor, feat: Optional[torch.Tensor], new_xyz: torch.Tensor, idx: torch.Tensor,
          msg_order: bool, pad4: bool = False) -> torch.Tensor:
    """Gather + recentre + concat (pointnet_util.py:127-131 / :243-247) -> [B, S, K, 3+D].
    pad4: rows are allocated with the channel count rounded up to a multiple of 4 (-> [B, S, K, ld], the data in
    [..., :3+D]) so that the training GEMMs can read them with 16-byte loads."""
    xyz, new_xyz = _cloud(xyz, "xyz", 3), _cloud(new_xyz, "new_xyz", 3)
    idx = _i64(idx, "idx")
    B, N, _ = xyz.shape
    _, S, K = idx.shape
    if feat is not None:
        feat = _cloud(feat, "points")
        D, fs = feat.shape[2], feat.stride()
    else:
        D, fs = 0, (0, 0, 0)
    ld = (3 + D + 3) // 4 * 4 if pad4 else 3 + D
    out = torch.empty((B, S, K, ld), dtype=torch.float32, device=xyz.device)
    with _on_device(xyz):
        nv.call("pn_group_f32", xyz.data_ptr(), *xyz.stride(), _p(feat), *fs, D, new_xyz.data_ptr(), *new_xyz.stride(),
                idx.data_ptr(), B, N, S, K, int(msg_order), out.data_ptr(), ld, _stream())
    return out


def _chamfer_clouds(p1: torch.Tensor, p2: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    p1, p2 = _cloud(p1, "p1"), _cloud(p2, "p2")
    if p1.shape[0] != p2.shape[0] or p1.shape[2] != p2.shape[2]:
        raise ValueError(f"p1 {tuple(p1.shape)} and p2 {tuple(p2.shape)} must agree on the batch size and the coordinates")
    return p1, p2


def chamfer_argmin(p1: torch.Tensor, p2: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """model/chamfer.py:7-53 with the nearest points (pn_chamfer_argmin_f32): p1 [B, N, D], p2 [B, M, D] (any strides,
    D <= 8) -> (total float64 [1] = sum over b, n of min_m ||p1[b,n] - p2[b,m]||, argmin int32 [B, N], the first of equal
    minima)."""
    p1, p2 = _chamfer_clouds(p1, p2)
    B, N, D = p1.shape
    total = torch.empty((1,), dtype=torch.float64, device=p1.device)
    argmin = torch.empty((B, N), dtype=torch.int32, device=p1.device)
    with _on_device(p1):
        nv.call("pn_chamfer_argmin_f32", p1.data_ptr(), *p1.stride(), p2.data_ptr(), *p2.stride(), B, N, p2.shape[1], D, None,
                total.data_ptr(), argmin.data_ptr(), _stream())
    return total, argmin


def chamfer_backward(p1: torch.Tensor, p2: torch.Tensor, argmin: torch.Tensor, g_total: torch.Tensor, scale: float,
                     need_p1: bool = True, need_p2: bool = True) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """Backward of the chamfer sum (pn_chamfer_bwd_f32): argmin of chamfer_argmin, g_total the loss gradient (a one-element
    device tensor) -> (dp1 [B, N, D] or None, dp2 [B, M, D] or None) of scale * g_total * sum_n ||p1[n] - p2[argmin[n]]||."""
    p1, p2 = _chamfer_clouds(p1, p2)
    B, N, D = p1.shape
    M = p2.shape[1]
    _need_cuda(argmin, "argmin")
    if argmin.dtype != torch.int32 or tuple(argmin.shape) != (B, N):
        raise ValueError(f"argmin must be an int32 [{B}, {N}] tensor")
    argmin = argmin.contiguous()
    g = _f32(g_total, "g_total").reshape(-1)
    if g.numel() != 1:
        raise ValueError("g_total must have one element")
    if not (need_p1 or need_p2):
        return None, None
    dp1 = torch.empty((B, N, D), dtype=torch.float32, device=p1.device) if need_p1 else None
    dp2 = torch.zeros((B, M, D), dtype=torch.float32, device=p1.device) if need_p2 else None
    with _on_device(p1):
        nv.call("pn_chamfer_bwd_f32", p1.data_ptr(), *p1.stride(), p2.data_ptr(), *p2.stride(), B, N, M, D, argmin.data_ptr(),
                g.contiguous().data_ptr(), float(scale), _p(dp1), _p(dp2), _stream())
    return dp1, dp2


def _rows(x: torch.Tensor, name: str) -> Tuple[torch.Tensor, int, int, int]:
    """2-D row-major view (rows, C) with unit channel stride -> (tensor, rows, C, ld)."""
    x = _f32(x, name)
    if x.dim() != 2:
        raise ValueError(f"{name} must be 2-D [rows, channels], got {tuple(x.shape)}")
    if x.stride(1) != 1 and x.shape[1] != 1:
        x = x.contiguous()
    ld = x.stride(0) if x.shape[0] > 1 else max(x.stride(0), x.shape[1])
    return x, x.shape[0], x.shape[1], ld


def linear(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], relu: bool,
           out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """y = act(x @ w.T + bias) for x [rows, cin], w [cout, cin] (BatchNorm already folded)."""
    x, rows, cin, ldx = _rows(x, "x")
    w = _f32(w, "w").contiguous()
    cout = w.shape[0]
    if w.shape != (cout, cin):
        raise ValueError(f"weight shape {tuple(w.shape)} does not match input channels {cin}")
    if bias is not None:
        bias = _f32(bias, "bias").contiguous()
    if out is None:
        out = torch.empty((rows, cout), dtype=torch.float32, device=x.device)
    ldy = out.stride(0) if rows > 1 else max(out.stride(0), cout)
    with _on_device(x):
        nv.call("pn_linear_f32", x.data_ptr(), ldx, 0, w.data_ptr(), 0, _p(bias), 0, int(relu), 1, rows, cin, cout,
                out.data_ptr(), ldy, 0, _stream())
    return out


def bmm_points(x: torch.Tensor, trans: torch.Tensor) -> torch.Tensor:
    """torch.bmm(x [B,N,k], trans [B,k,k2]) of pointnet.py:105-107 as a batched linear layer."""
    x = _f32(x, "x").contiguous()
    wt = _f32(trans, "trans").transpose(1, 2).contiguous()        # [B, k2, k]: rows = output channels
    B, N, k = x.shape
    k2 = wt.shape[1]
    out = torch.empty((B, N, k2), dtype=torch.float32, device=x.device)
    with _on_device(x):
        nv.call("pn_linear_f32", x.data_ptr(), k, N * k, wt.data_ptr(), k2 * k, None, 0, 0, B, N, k, k2, out.data_ptr(),
                k2, N * k2, _stream())
    return out


def linear_cloud_bias(x: torch.Tensor, w: torch.Tensor, cloud_bias: torch.Tensor, relu: bool) -> torch.Tensor:
    """y[b,n,:] = act(x[b,n,:] @ w.T + cloud_bias[b,:]) for x [B,N,cin]: shared weights, one bias row per cloud."""
    x = _f32(x, "x").contiguous()
    w = _f32(w, "w").contiguous()
    cloud_bias = _f32(cloud_bias, "cloud_bias").contiguous()
    B, N, cin = x.shape
    cout = w.shape[0]
    if w.shape != (cout, cin) or cloud_bias.shape != (B, cout):
        raise ValueError("linear_cloud_bias: shape mismatch")
    out = torch.empty((B, N, cout), dtype=torch.float32, device=x.device)
    with _on_device(x):
        nv.call("pn_linear_f32", x.data_ptr(), cin, N * cin, w.data_ptr(), 0, cloud_bias.data_ptr(), cout, int(relu), B, N,
                cin, cout, out.data_ptr(), cout, N * cout, _stream())
    return out


def group_max(x: torch.Tensor, K: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """max over each run of K consecutive rows: [G*K, C] -> [G, C] (optionally into a strided `out` view)."""
    x, rows, Cc, ldx = _rows(x, "x")
    if rows % K:
        raise ValueError(f"{rows} rows are not a multiple of K={K}")
    G = rows // K
    if out is None:
        out = torch.empty((G, Cc), dtype=torch.float32, device=x.device)
    elif out.shape != (G, Cc) or out.stride(1) != 1 or out.dtype != torch.float32:
        raise ValueError("out must be a float32 [groups, C] view with unit channel stride")
    ldy = out.stride(0) if G > 1 else max(out.stride(0), Cc)
    with _on_device(x):
        nv.call("pn_group_max_f32", x.data_ptr(), ldx, G, int(K), Cc, out.data_ptr(), ldy, _stream())
    return out


NN_BLOCKS_MIN_EVALS = 1 << 22   # N * S per cloud from which the block search pays for its build
NN_BLOCKS_MAX_S = 8192


def three_nn(xyz1: torch.Tensor, xyz2: torch.Tensor, order: Optional[BallGrid] = None,
             method: str = "auto", background: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """3 nearest sources and normalised inverse-distance weights (pointnet_util.py:295-300).
    method: "scan" (pn_three_nn_f32, all N x S distances), "blocks" (pn_three_nn_blocks_f32: exact branch-and-bound
    over Morton blocks of the coarse cloud) or "auto" (blocks for large N x S when `order`, the bucket order of the
    fine cloud, is available).  Both return identical results.  background: the block search runs on a capped grid
    (~3 small CTAs per SM) so that it can share the GPU with the kernels of another stream."""
    xyz1, xyz2 = _cloud(xyz1, "xyz1", 3), _cloud(xyz2, "xyz2", 3)
    B, N, _ = xyz1.shape
    S = xyz2.shape[1]
    idx = torch.empty((B, N, 3), dtype=torch.int64, device=xyz1.device)
    w = torch.empty((B, N, 3), dtype=torch.float32, device=xyz1.device)
    if method == "auto":
        method = "blocks" if (order is not None and 32 <= S <= NN_BLOCKS_MAX_S and N * S >= NN_BLOCKS_MIN_EVALS) else "scan"
    if method == "blocks":
        if order is not None and (order.B, order.N) != (B, N):
            raise ValueError("order grid was built for another cloud shape")
        optr, oes, obs = order.order() if order is not None else (None, 0, 0)
        nbytes = int(nv.lib().pn_three_nn_blocks_bytes(B, S))
        blocks = torch.empty((nbytes,), dtype=torch.uint8, device=xyz1.device)
        with _on_device(xyz1):
            nv.call("pn_three_nn_blocks_build_f32", xyz2.data_ptr(), *xyz2.stride(), B, S, blocks.data_ptr(), nbytes, _stream())
            nv.call("pn_three_nn_blocks_f32", xyz1.data_ptr(), *xyz1.stride(), optr, oes, obs, blocks.data_ptr(), nbytes, B, N,
                    S, int(bool(background)), idx.data_ptr(), w.data_ptr(), _stream())
        return idx, w
    if method != "scan":
        raise ValueError(f"unknown 3-NN method {method!r}")
    with _on_device(xyz1):
        nv.call("pn_three_nn_f32", xyz1.data_ptr(), *xyz1.stride(), xyz2.data_ptr(), *xyz2.stride(), B, N, S,
                idx.data_ptr(), w.data_ptr(), _stream())
    return idx, w


def three_interpolate(points1: Optional[torch.Tensor], points2: torch.Tensor, idx: torch.Tensor,
                      weight: torch.Tensor) -> torch.Tensor:
    """cat([points1, sum_k points2[idx_k] * weight_k]) (pointnet_util.py:301-307) -> [B, N, D1+D2]."""
    points2 = _cloud(points2, "points2")
    idx = _i64(idx, "idx")
    weight = _f32(weight, "weight").contiguous()
    B, S, D2 = points2.shape
    N = idx.shape[1]
    if points1 is not None:
        points1 = _cloud(points1, "points1")
        D1, s1 = points1.shape[2], points1.stride()
    else:
        D1, s1 = 0, (0, 0, 0)
    out = torch.empty((B, N, D1 + D2), dtype=torch.float32, device=points2.device)
    with _on_device(points2):
        nv.call("pn_three_interpolate_f32", _p(points1), *s1, D1, points2.data_ptr(), *points2.stride(), D2, S,
                idx.data_ptr(), weight.data_ptr(), B, N, out.data_ptr(), D1 + D2, N * (D1 + D2), _stream())
    return out


def log_softmax(x: torch.Tensor) -> torch.Tensor:
    x, rows, Cc, ldx = _rows(x, "x")
    out = torch.empty((rows, Cc), dtype=torch.float32, device=x.device)
    with _on_device(x):
        nv.call("pn_log_softmax_f32", x.data_ptr(), ldx, rows, Cc, out.data_ptr(), Cc, _stream())
    return out


def argmax_labels(logp: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """logp [..., C] -> uint8 labels [...] = logp.argmax(-1) (pcdseg.py:75), the first maximum winning (pn_argmax_labels_u8)."""
    Cc = logp.shape[-1]
    x, rows, _, ldx = _rows(logp.reshape(-1, Cc), "logp")
    if out is None:
        out = torch.empty(logp.shape[:-1], dtype=torch.uint8, device=x.device)
    elif out.dtype != torch.uint8 or out.numel() != rows or not out.is_contiguous() or not out.is_cuda:
        raise ValueError("out must be a contiguous uint8 CUDA tensor with one element per row")
    with _on_device(x):
        nv.call("pn_argmax_labels_u8", x.data_ptr(), ldx, rows, Cc, out.data_ptr(), _stream())
    return out


# ------------------------------------------------------------------------------------------------
# Fused shared-MLP chains on the tensor cores (tcgen05 + TMEM): pn_*_bf16x3 entry points.
# "bf16x3" computes every product as a_hi*w_hi + a_hi*w_lo + a_lo*w_hi with fp32 accumulation: fp32 parity
# (relative error ~1e-5) at tensor-core speed.  "fp32" keeps the exact-fp32 CUDA-core path (pn_linear_f32).
OUT_ROWS, OUT_MAX32, OUT_LOG_SOFTMAX = 0, 1, 2
if os.environ.get("PN12_MLP", "bf16x3") in ("bf16x3", "bf16", "fp32"):
    _DEFAULTS["precision"] = os.environ.get("PN12_MLP", "bf16x3")


def set_mlp_mode(mode: str) -> str:
    """'bf16x3' (tensor cores, 3-pass split bf16 = fp32 parity, default), 'bf16' (the same kernels issuing only the
    hi x hi product: plain bf16 inputs, fp32 accumulation, a third of the tensor-core work) or 'fp32' (CUDA cores, exact
    fp32 accumulation).  Sets the process default (and drops the calling thread's override); returns the old mode.
    For one thread or one block of code use `with ops.options(precision=...)`."""
    if mode not in ("bf16x3", "bf16", "fp32"):
        raise ValueError("mode must be 'bf16x3', 'bf16' or 'fp32'")
    old = _opt("precision")
    _DEFAULTS["precision"] = mode
    if hasattr(_tls, "precision"):
        del _tls.precision
    return old


def mlp_mode() -> str:
    """The engine the modules use: 'bf16x3' (tensor-core chains, in either precision) or 'fp32'."""
    return "fp32" if _opt("precision") == "fp32" else "bf16x3"


def mlp_precision() -> str:
    return _opt("precision")


_ENGINES = {"auto": 0, "stream": 1, "resident": 2, "auto-rowwise": 4, "resident-rowwise": 6, "auto-noslice": 8,
            "stream-noslice": 9, "auto-narrow": 16, "stream-narrow": 17}


def set_mlp_engine(engine: str = "auto") -> None:
    """Tuning hook (process default of pn_launch_opts.mlp_engine): 'auto' (resident-weight kernel when the packed chain fits
    in shared memory, streaming ring otherwise), 'stream' or 'resident'; '*-rowwise' keeps the row-per-thread producers (no
    coalesced quad producer) for A/B comparisons."""
    _DEFAULTS["mlp_engine"] = _ENGINES[engine]


def set_reserved_sms(sms: int = 0) -> None:
    """SMs the resident-weight chain launches of the CALLING THREAD leave to kernels of other streams."""
    _tls.reserved_sms = int(sms)


FOLD_FIRST_FP_LAYER = os.environ.get("PN12_FP_FOLD", "1") != "0"
# Levels with fewer 128-row tiles than this run layer by layer: a single-layer chain is N-sliced over gridDim.y, so
# every launch fills the GPU, whereas the fused chain occupies only `tiles` SMs for the whole level.  Measured on
# B200 at C2 size the fused chains still win (every sliced launch repeats the row producer, which is the latency-
# bound part: sa4 73 vs 40 us, fp2 84 vs 41 us), so the default is 0 = never; kept for larger per-level row counts.
LAYERWISE_MAX_TILES = int(os.environ.get("PN12_LAYERWISE_TILES", "0"))


class PackedChain:
    """A conv+BN(+ReLU) chain folded and packed for the tensor-core kernels (device blob + descriptor)."""

    def __init__(self, layers: Sequence[Tuple[torch.Tensor, Optional[torch.Tensor], bool]], transposed: bool = False):
        """layers = [(w [cout, cin], bias or None, relu)].  transposed: every w is given as the TRANSPOSE of the layer's
        weight, a row-major [cin, cout] matrix (the input-gradient GEMM of the training step packs W^T this way)."""
        self.desc = nv.MlpDesc()
        self.desc.nlayers = len(layers)
        for i, (w, _, relu) in enumerate(layers):
            co, ci = (int(w.shape[1]), int(w.shape[0])) if transposed else (int(w.shape[0]), int(w.shape[1]))
            self.desc.cout[i], self.desc.cin[i] = co, ci
            self.desc.relu[i] = int(bool(relu))
        self.cin, self.cout = int(self.desc.cin[0]), int(self.desc.cout[len(layers) - 1])
        nbytes = nv.lib().pn_mlp_blob_bytes(C.byref(self.desc))
        if nbytes == 0:
            raise RuntimeError("chain not supported by the tensor-core path: "
                               + nv.lib().pn_last_error_string().decode("utf-8", "replace"))
        dev = layers[0][0].device
        self.blob = torch.empty(nbytes, dtype=torch.uint8, device=dev)      # the pack kernels write every byte (padding = 0)
        ws = [_f32(w, "w").contiguous() for w, _, _ in layers]
        bs = [None if b is None else _f32(b, "bias").contiguous() for _, b, _ in layers]
        n = len(layers)
        wp = (C.c_void_p * n)(*[w.data_ptr() for w in ws])
        bp = (C.c_void_p * n)(*[None if b is None else b.data_ptr() for b in bs])
        with _on_device(self.blob):
            if transposed:
                nv.call("pn_mlp_pack_t_bf16x3", C.byref(self.desc), wp, bp, (C.c_int * n)(*([1] * n)), self.blob.data_ptr(), _stream())
            else:
                nv.call("pn_mlp_pack_bf16x3", C.byref(self.desc), wp, bp, self.blob.data_ptr(), _stream())
        self._keep = (ws, bs)     # the pack kernels read them asynchronously

    @property
    def resident(self) -> bool:
        """True when the chain's weights stay resident in shared memory (pn_mlp_resident_groups): one weight load per CTA
        instead of one per row tile."""
        return nv.lib().pn_mlp_resident_groups(C.byref(self.desc)) > 0

    def bias_view(self, layer: int = 0) -> torch.Tensor:
        """The fp32 bias of one layer inside the packed blob ([cout] view): a caller whose bias depends on the input (the
        per-cloud bias of PointNetSeg's first head layer) writes it there before the launch instead of re-packing the chain."""
        off, boff = 0, 0
        n = int(self.desc.nlayers)
        pad = lambda v: (v + 31) // 32 * 32      # noqa: E731
        for l in range(n):
            k_pad = pad(int(self.desc.cin[l])) if l == 0 else pad(int(self.desc.cout[l - 1]))
            off += pad(int(self.desc.cout[l])) * k_pad * 4
        for l in range(layer):
            boff += pad(int(self.desc.cout[l]))
        start = off + 4 * boff
        return self.blob[start:start + 4 * int(self.desc.cout[layer])].view(torch.float32)

    @staticmethod
    def supported(dims: Sequence[Tuple[int, int]]) -> bool:
        """dims = [(cin, cout), ...]"""
        if not 1 <= len(dims) <= nv.MLP_MAX_LAYERS:
            return False
        d = nv.MlpDesc()
        d.nlayers = len(dims)
        for i, (ci, co) in enumerate(dims):
            d.cin[i], d.cout[i], d.relu[i] = int(ci), int(co), 1
        return nv.lib().pn_mlp_blob_bytes(C.byref(d)) > 0


def mlp_rows_tc(chain: PackedChain, x: torch.Tensor, out_mode: int = OUT_ROWS,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """chain(x) for x [rows, cin]; OUT_MAX32 pools every 32 consecutive rows, OUT_LOG_SOFTMAX ends in log_softmax.
    out: optional [out_rows, cout] view with unit channel stride to write into."""
    x, rows, cin, ldx = _rows(x, "x")
    if cin != chain.cin:
        raise ValueError(f"chain expects {chain.cin} input channels, got {cin}")
    out_rows = rows // 32 if out_mode == OUT_MAX32 else rows
    if out is None:
        out = torch.empty((out_rows, chain.cout), dtype=torch.float32, device=x.device)
    elif out.shape != (out_rows, chain.cout) or out.stride(1) != 1 or out.dtype != torch.float32:
        raise ValueError("out must be a float32 [out_rows, cout] view with unit channel stride")
    ldy = out.stride(0) if out_rows > 1 else max(out.stride(0), chain.cout)
    with _on_device(x):
        nv.call("pn_mlp_rows_bf16x3", C.byref(chain.desc), chain.blob.data_ptr(), x.data_ptr(), ldx, rows, out_mode,
                out.data_ptr(), ldy, C.byref(_launch_opts(True)), _stream())
    return out


def sa_mlp_max_tc(chain: PackedChain, xyz: torch.Tensor, feat: Optional[torch.Tensor], new_xyz: torch.Tensor,
                  idx: torch.Tensor, msg_order: bool, out: Optional[torch.Tensor] = None,
                  out_mode: int = 1) -> torch.Tensor:
    """Grouping + shared MLP + max over nsample in one kernel -> [B, S, cout] (or into the strided view `out`).
    out_mode=OUT_ROWS keeps the grouped rows instead: [B*S*K, cout] (layer-by-layer execution of small levels)."""
    xyz, new_xyz = _cloud(xyz, "xyz", 3), _cloud(new_xyz, "new_xyz", 3)
    idx = _i64(idx, "idx")
    B, N, _ = xyz.shape
    _, S, K = idx.shape
    if feat is not None:
        feat = _cloud(feat, "points")
        D, fs = feat.shape[2], feat.stride()
    else:
        D, fs = 0, (0, 0, 0)
    if out_mode != OUT_ROWS and K != 16 and K % 32:
        raise ValueError(f"the fused set-abstraction kernel pools groups of 16 or 32 m samples, got nsample={K}")
    if out_mode != OUT_ROWS and K > 32:
        # the kernel pools runs of 32 rows; the K / 32 partial maxima of a group are reduced by pn_group_max_f32
        part = torch.empty((B * S * (K // 32), chain.cout), dtype=torch.float32, device=xyz.device)
        with _on_device(xyz):
            nv.call("pn_sa_mlp_bf16x3", C.byref(chain.desc), chain.blob.data_ptr(), xyz.data_ptr(), *xyz.stride(), _p(feat),
                    *fs, D, new_xyz.data_ptr(), *new_xyz.stride(), idx.data_ptr(), B, N, S, K, int(msg_order), int(out_mode),
                    part.data_ptr(), chain.cout, C.byref(_launch_opts(True)), _stream())
        pooled = group_max(part, K // 32, out=out)
        return pooled.view(B, S, chain.cout) if out is None else out
    if out_mode == OUT_ROWS:
        if out is not None:
            raise ValueError("out= is only supported with the max-pooled output")
        out = torch.empty((B * S * K, chain.cout), dtype=torch.float32, device=xyz.device)
        ldo = chain.cout
    elif out is None:
        out = torch.empty((B, S, chain.cout), dtype=torch.float32, device=xyz.device)
        ldo = chain.cout
    else:
        if out.shape != (B * S, chain.cout) or out.stride(1) != 1:
            raise ValueError("out must be a [B*S, cout] view with unit channel stride")
        ldo = out.stride(0)
    with _on_device(xyz):
        nv.call("pn_sa_mlp_bf16x3", C.byref(chain.desc), chain.blob.data_ptr(), xyz.data_ptr(), *xyz.stride(), _p(feat),
                *fs, D, new_xyz.data_ptr(), *new_xyz.stride(), idx.data_ptr(), B, N, S, K, int(msg_order), int(out_mode),
                out.data_ptr(), ldo, C.byref(_launch_opts(True)), _stream())
    return out


def fp_mlp_tc(chain: PackedChain, points1: Optional[torch.Tensor], points2: torch.Tensor, idx: torch.Tensor,
              weight: torch.Tensor, out_mode: int = OUT_ROWS, relu_in: bool = False,
              order: Optional[BallGrid] = None, out: Optional[torch.Tensor] = None,
              clouds: Optional[Tuple[int, int]] = None, residual: Optional[torch.Tensor] = None) -> torch.Tensor:
    """3-NN interpolation + skip concat + shared MLP (+ head + log_softmax) in one kernel -> [B, N, cout].
    relu_in: ReLU on the interpolated channels first (the level's first layer was folded into the coarse level).
    order: a BallGrid of the fine cloud -- tiles then walk the points in bucket order (same result, L1-friendly).
    out: a contiguous [B, N, cout] float32 buffer to write into; clouds = (b0, b1): only that slice of the batch is
    computed (into out[b0:b1]) -- a caller can then start moving the first clouds while the rest are computed.
    residual: [B, N, C] rows (C = first layer's width rounded up to 32) added to the first layer's pre-activation: the
    skip half of that layer, computed by the caller beforehand (then points1 is None and the chain holds only W_b)."""
    points2 = _cloud(points2, "points2")
    idx = _i64(idx, "idx")
    weight = _f32(weight, "weight").contiguous()
    B, S, D2 = points2.shape
    N = idx.shape[1]
    if points1 is not None:
        points1 = _cloud(points1, "points1")
        D1, s1 = points1.shape[2], points1.stride()
    else:
        D1, s1 = 0, (0, 0, 0)
    if out is None:
        out = torch.empty((B, N, chain.cout), dtype=torch.float32, device=points2.device)
    elif out.shape != (B, N, chain.cout) or not out.is_contiguous() or out.dtype != torch.float32 or not out.is_cuda:
        raise ValueError("out must be a contiguous float32 CUDA tensor of shape [B, N, cout]")
    optr, oes, obs = (None, 0, 0)
    if order is not None:
        if (order.B, order.N) != (B, N):
            raise ValueError("order grid was built for another cloud shape")
        optr, oes, obs = order.order()
    rptr, ldr = None, 0
    if residual is not None:
        if clouds is not None or points1 is not None:
            raise ValueError("residual= cannot be combined with points1 or clouds")
        if residual.shape[:2] != (B, N) or not residual.is_contiguous() or residual.dtype != torch.float32:
            raise ValueError("residual must be a contiguous float32 [B, N, C] tensor")
        rptr, ldr = residual.data_ptr(), residual.shape[2]
    full_out = out
    if clouds is not None:
        b0, b1 = clouds
        if not 0 <= b0 < b1 <= B:
            raise ValueError(f"clouds={clouds} is not a slice of the batch of {B}")
        points1 = points1[b0:b1] if points1 is not None else None
        points2, idx, weight, out = points2[b0:b1], idx[b0:b1], weight[b0:b1], out[b0:b1]
        if optr is not None:
            optr += 4 * obs * b0
        B = b1 - b0
    with _on_device(points2):
        nv.call("pn_fp_mlp_bf16x3", C.byref(chain.desc), chain.blob.data_ptr(), _p(points1), *s1, D1, points2.data_ptr(),
                *points2.stride(), D2, S, idx.data_ptr(), weight.data_ptr(), int(bool(relu_in)), optr, oes, obs, rptr, ldr,
                B, N, out_mode, out.data_ptr(), chain.cout, C.byref(_launch_opts(True)), _stream())
    return full_out


# ------------------------------------------------------------------------------------------------
# Training-step and evaluation-metric kernels (csrc/train.cu).  Row matrices are 2-D float32 views with unit
# channel stride (a leading dimension is taken from stride(0)); statistics accumulators are float64.
def _ld(t: torch.Tensor) -> int:
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t.shape[1])


def _rowmat(t: torch.Tensor, name: str) -> torch.Tensor:
    _need_cuda(t, name)
    if t.dtype != torch.float32 or t.dim() != 2 or (t.stride(1) != 1 and t.shape[1] != 1):
        raise ValueError(f"{name} must be a float32 [rows, C] matrix with unit channel stride")
    return t


class BatchStats:
    """Statistics one BatchNorm layer normalises with: scale/shift for the forward, mean/invstd for the backward.
    running=False: the batch's own (training mode); running=True: the module's running statistics (running_stats)."""

    __slots__ = ("scale", "shift", "mean", "invstd", "rows", "running")

    def __init__(self):
        self.running = False


def uses_running_stats(bn) -> bool:
    """nn.BatchNorm's rule: batch statistics in training mode or when the module keeps no running statistics."""
    return not bn.training and bn.running_mean is not None and bn.running_var is not None


def running_stats(bn) -> BatchStats:
    """BatchStats from bn's running statistics, the expressions of fold_conv_bn: scale = gamma/sqrt(var+eps), shift =
    beta - mean*scale, invstd = 1/sqrt(var+eps).  Nothing of bn is written.  Cached on the module until a parameter or buffer
    changes (storage or version) -- a write that bypasses the version counter (through .data) is not seen, as with the folded
    weights of the eval path; under CUDA-graph capture they are computed inside the graph instead, so that a replay
    follows the parameters an optimizer has updated in place since."""
    capturing = bn.running_mean.is_cuda and torch.cuda.is_current_stream_capturing()
    tensors = (bn.weight, bn.bias, bn.running_mean, bn.running_var)
    key = (float(bn.eps),) + tuple((t.data_ptr(), t._version) if t is not None else None for t in tensors)
    cached = bn.__dict__.get("_pn_running_stats")
    if cached is not None and cached[0] == key and not capturing:
        return cached[1]
    with torch.no_grad():
        mean = bn.running_mean.detach().float()
        root = torch.sqrt(bn.running_var.detach().float() + bn.eps)
        invstd = 1.0 / root
        scale = bn.weight.detach().float() / root if bn.weight is not None else invstd
        shift = (bn.bias.detach().float() if bn.bias is not None else torch.zeros_like(mean)) - mean * scale
        st = BatchStats()
        st.scale, st.shift, st.mean, st.invstd = scale.contiguous(), shift.contiguous(), mean.contiguous(), invstd.contiguous()
    st.rows, st.running = None, True
    if not capturing:
        bn.__dict__["_pn_running_stats"] = (key, st)
    return st


def bn_batch_stats(y: torch.Tensor, bn, momentum_update: bool = True) -> BatchStats:
    """pn_bn_stats_f32 + pn_bn_finalize_f32 over the rows of y; updates bn.running_* / num_batches_tracked like
    nn.BatchNorm in train mode (momentum = bn.momentum)."""
    y = _rowmat(y, "y")
    rows, Cc = y.shape
    acc = torch.zeros((2, Cc), dtype=torch.float64, device=y.device)
    st = BatchStats()
    buf = torch.empty((4, Cc), dtype=torch.float32, device=y.device)
    st.scale, st.shift, st.mean, st.invstd = buf[0], buf[1], buf[2], buf[3]
    st.rows = rows
    track = momentum_update and bn.track_running_stats and bn.running_mean is not None
    with _on_device(y):
        nv.call("pn_bn_stats_f32", y.data_ptr(), _ld(y), rows, Cc, acc[0].data_ptr(), acc[1].data_ptr(), _stream())
        nv.call("pn_bn_finalize_f32", acc[0].data_ptr(), acc[1].data_ptr(), rows, Cc, _p(bn.weight), _p(bn.bias),
                float(bn.eps), float(bn.momentum if bn.momentum is not None else 0.1),
                bn.running_mean.data_ptr() if track else None, bn.running_var.data_ptr() if track else None,
                bn.num_batches_tracked.data_ptr() if track and bn.num_batches_tracked is not None else None,
                st.scale.data_ptr(), st.shift.data_ptr(), st.mean.data_ptr(), st.invstd.data_ptr(), _stream())
    if track:      # written through raw pointers: tell torch (the eval path refolds BatchNorm when a version changes)
        torch.autograd.graph.increment_version([b for b in (bn.running_mean, bn.running_var, bn.num_batches_tracked) if b is not None])
    return st


def bn_finalize(acc: torch.Tensor, rows: int, bn) -> BatchStats:
    """pn_bn_finalize_f32 on column sums acc float64 [2, C] (sum, sum of squares) accumulated over `rows` rows -- by
    pn_bn_stats_f32 or by the epilogue of pn_train_gemm_bf16x3; updates bn.running_* like nn.BatchNorm in train mode."""
    Cc = acc.shape[1]
    st = BatchStats()
    buf = torch.empty((4, Cc), dtype=torch.float32, device=acc.device)
    st.scale, st.shift, st.mean, st.invstd = buf[0], buf[1], buf[2], buf[3]
    st.rows = rows
    track = bn.track_running_stats and bn.running_mean is not None
    with _on_device(acc):
        nv.call("pn_bn_finalize_f32", acc[0].data_ptr(), acc[1].data_ptr(), rows, Cc, _p(bn.weight), _p(bn.bias),
                float(bn.eps), float(bn.momentum if bn.momentum is not None else 0.1),
                bn.running_mean.data_ptr() if track else None, bn.running_var.data_ptr() if track else None,
                bn.num_batches_tracked.data_ptr() if track and bn.num_batches_tracked is not None else None,
                st.scale.data_ptr(), st.shift.data_ptr(), st.mean.data_ptr(), st.invstd.data_ptr(), _stream())
    if track:
        torch.autograd.graph.increment_version([b for b in (bn.running_mean, bn.running_var, bn.num_batches_tracked) if b is not None])
    return st


def train_gemm_supported(cin: int, cout: int) -> bool:
    return bool(nv.lib().pn_train_gemm_supported(int(cin), int(cout)))


def train_gemm(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], in_stats: Optional[BatchStats] = None,
               in_relu: bool = True, stats_acc: Optional[torch.Tensor] = None, transposed: bool = False,
               packed: Optional[torch.Tensor] = None) -> torch.Tensor:
    """pn_train_gemm_bf16x3: y = f(x) @ W^T + bias with f = the normalise(+ReLU) of the layer that produced x (in_stats:
    its BatchStats; None = identity), column sums of y / y*y added to stats_acc (float64 [2, cout], zeroed by the caller).
    W = w [cout, cin], or w^T for w [cin, cout] when transposed."""
    x = _rowmat(x, "x")
    rows, cin = x.shape
    w = _f32(w, "w").contiguous()
    cout = w.shape[1] if transposed else w.shape[0]
    if (w.shape[0] if transposed else w.shape[1]) != cin:
        raise ValueError(f"weight shape {tuple(w.shape)} does not match {cin} input channels")
    y = torch.empty((rows, cout), dtype=torch.float32, device=x.device)
    # packed: the weight image already converted by pn_train_pack_many (train.PackedWeights); else converted by this call
    scratch = packed if packed is not None else torch.empty((int(nv.lib().pn_train_gemm_scratch_bytes(cin, cout)),),
                                                            dtype=torch.uint8, device=x.device)
    with _on_device(x):
        nv.call("pn_train_gemm_bf16x3", x.data_ptr(), _ld(x), rows, cin, _p(in_stats.scale) if in_stats is not None else None,
                _p(in_stats.shift) if in_stats is not None else None, int(in_relu), None if packed is not None else w.data_ptr(),
                int(transposed), _p(bias), cout,
                y.data_ptr(), cout, _p(stats_acc[0]) if stats_acc is not None else None,
                _p(stats_acc[1]) if stats_acc is not None else None, scratch.data_ptr(), _stream(), tag=(rows, cin, cout))
    return y


def train_gemm_bnbwd(dy: torch.Tensor, w: torch.Tensor, prev_y: torch.Tensor, prev_st: BatchStats, acc: torch.Tensor,
                     transposed: bool = True, packed: Optional[torch.Tensor] = None) -> torch.Tensor:
    """pn_train_gemm_bnbwd_bf16x3: dz = dy @ W (w [cout_layer, cin_layer] given as stored, transposed=True) plus, in the
    epilogue, the two reductions of the BatchNorm backward of the layer BELOW (pre-normalisation output prev_y, statistics
    prev_st) into acc (float64 [2, C], zeroed): bn_act_backward(..., acc=acc, acc_ready=True) then skips its own pass."""
    dy = _rowmat(dy, "dy")
    rows, cin = dy.shape
    w = _f32(w, "w").contiguous()
    cout = w.shape[1] if transposed else w.shape[0]
    prev_y = _rowmat(prev_y, "prev_y")
    if prev_y.shape != (rows, cout):
        raise ValueError("prev_y must be [rows, cout]")
    dz = torch.empty((rows, cout), dtype=torch.float32, device=dy.device)
    scratch = packed if packed is not None else torch.empty((int(nv.lib().pn_train_gemm_scratch_bytes(cin, cout)),),
                                                            dtype=torch.uint8, device=dy.device)
    with _on_device(dy):
        nv.call("pn_train_gemm_bnbwd_bf16x3", dy.data_ptr(), _ld(dy), rows, cin, None if packed is not None else w.data_ptr(),
                int(transposed), cout, dz.data_ptr(),
                cout, prev_y.data_ptr(), _ld(prev_y), prev_st.scale.data_ptr(), prev_st.shift.data_ptr(), prev_st.mean.data_ptr(),
                prev_st.invstd.data_ptr(), acc[0].data_ptr(), acc[1].data_ptr(), scratch.data_ptr(), _stream())
    return dz


def train_gemm_bneval(dy: torch.Tensor, w: torch.Tensor, prev_y: torch.Tensor, prev_st: BatchStats, acc: torch.Tensor,
                      dgamma: Optional[torch.Tensor] = None, dbeta: Optional[torch.Tensor] = None, transposed: bool = True,
                      packed: Optional[torch.Tensor] = None) -> torch.Tensor:
    """pn_train_gemm_bneval_bf16x3: the input-gradient GEMM dy @ W of a layer whose input came from a BatchNorm with FIXED
    statistics prev_st (running_stats) applied to prev_y, with that BatchNorm's backward in the epilogue: returns the layer
    below's dy = scale * g (what bn_eval_backward would return for dz = dy @ W), adds its affine gradients to dgamma / dbeta.
    acc: float64 [2, C] scratch, ZEROED."""
    dy = _rowmat(dy, "dy")
    rows, cin = dy.shape
    w = _f32(w, "w").contiguous()
    cout = w.shape[1] if transposed else w.shape[0]
    prev_y = _rowmat(prev_y, "prev_y")
    if prev_y.shape != (rows, cout):
        raise ValueError("prev_y must be [rows, cout]")
    out = torch.empty((rows, cout), dtype=torch.float32, device=dy.device)
    scratch = packed if packed is not None else torch.empty((int(nv.lib().pn_train_gemm_scratch_bytes(cin, cout)),),
                                                            dtype=torch.uint8, device=dy.device)
    with _on_device(dy):
        nv.call("pn_train_gemm_bneval_bf16x3", dy.data_ptr(), _ld(dy), rows, cin, None if packed is not None else w.data_ptr(),
                int(transposed), cout, out.data_ptr(), cout, prev_y.data_ptr(), _ld(prev_y), prev_st.scale.data_ptr(),
                prev_st.shift.data_ptr(), prev_st.mean.data_ptr(), prev_st.invstd.data_ptr(), acc[0].data_ptr(), acc[1].data_ptr(),
                _p(dgamma), _p(dbeta), scratch.data_ptr(), _stream())
    return out


def bn_act(y: torch.Tensor, st: BatchStats, relu: bool = True, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    y = _rowmat(y, "y")
    rows, Cc = y.shape
    if out is None:
        out = torch.empty((rows, Cc), dtype=torch.float32, device=y.device)
    with _on_device(y):
        nv.call("pn_bn_act_f32", y.data_ptr(), _ld(y), rows, Cc, st.scale.data_ptr(), st.shift.data_ptr(), int(relu),
                out.data_ptr(), _ld(out), _stream())
    return out


def bn_act_max(y: torch.Tensor, st: BatchStats, K: int, relu: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
    """-> (pooled [rows/K, C], argmax int32 [rows/K, C])."""
    y = _rowmat(y, "y")
    rows, Cc = y.shape
    G = rows // K
    out = torch.empty((G, Cc), dtype=torch.float32, device=y.device)
    am = torch.empty((G, Cc), dtype=torch.int32, device=y.device)
    with _on_device(y):
        nv.call("pn_bn_act_max_f32", y.data_ptr(), _ld(y), G, int(K), Cc, st.scale.data_ptr(), st.shift.data_ptr(),
                int(relu), out.data_ptr(), Cc, am.data_ptr(), _stream())
    return out, am


def bn_act_backward(y: torch.Tensor, st: BatchStats, dz: torch.Tensor, relu: bool = True,
                    argmax: Optional[torch.Tensor] = None, K: int = 1, dgamma: Optional[torch.Tensor] = None,
                    dbeta: Optional[torch.Tensor] = None, acc: Optional[torch.Tensor] = None, acc_ready: bool = False):
    """Backward of act(bn(y)) with batch statistics.  dgamma / dbeta given ([C] float32 buffers): the affine gradients
    are ADDED to them and dy [rows, C] is returned; otherwise -> (dy, dgamma, dbeta) with fresh buffers.
    argmax/K: dz is the pooled gradient [rows/K, C] of bn_act_max."""
    y, dz = _rowmat(y, "y"), _rowmat(dz, "dz")
    rows, Cc = y.shape
    if acc is None:          # float64 [2, C] scratch for the two reductions, ZEROED (a caller may pass a slice of a larger buffer)
        acc = torch.zeros((2, Cc), dtype=torch.float64, device=y.device)
    dy = torch.empty((rows, Cc), dtype=torch.float32, device=y.device)
    fresh = dgamma is None
    if fresh:
        dgb = torch.zeros((2, Cc), dtype=torch.float32, device=y.device)
        dgamma, dbeta = dgb[0], dgb[1]
    common = (y.data_ptr(), _ld(y), rows, Cc, dz.data_ptr(), _ld(dz), _p(argmax), int(K), st.scale.data_ptr(),
              st.shift.data_ptr(), st.mean.data_ptr(), st.invstd.data_ptr(), int(relu), acc[0].data_ptr(), acc[1].data_ptr())
    with _on_device(y):
        if not acc_ready:        # (acc_ready: the reductions were accumulated by the epilogue of train_gemm_bnbwd)
            nv.call("pn_bn_bwd_stats_f32", *common, _stream())
        nv.call("pn_bn_bwd_apply_f32", *common, dy.data_ptr(), Cc, dgamma.data_ptr(), dbeta.data_ptr(), _stream())
    return (dy, dgamma, dbeta) if fresh else dy


def bn_eval_backward(y: torch.Tensor, st: BatchStats, dz: torch.Tensor, relu: bool = True,
                     argmax: Optional[torch.Tensor] = None, K: int = 1, dgamma: Optional[torch.Tensor] = None,
                     dbeta: Optional[torch.Tensor] = None, acc: Optional[torch.Tensor] = None):
    """pn_bn_eval_bwd_f32: backward of act(bn(y)) with fixed statistics (running_stats), one pass: dy = scale * g.
    dgamma / dbeta and argmax / K as in bn_act_backward; acc: float64 [2, C] scratch, ZEROED."""
    y, dz = _rowmat(y, "y"), _rowmat(dz, "dz")
    rows, Cc = y.shape
    if acc is None:
        acc = torch.zeros((2, Cc), dtype=torch.float64, device=y.device)
    dy = torch.empty((rows, Cc), dtype=torch.float32, device=y.device)
    fresh = dgamma is None
    if fresh:
        dgb = torch.zeros((2, Cc), dtype=torch.float32, device=y.device)
        dgamma, dbeta = dgb[0], dgb[1]
    with _on_device(y):
        nv.call("pn_bn_eval_bwd_f32", y.data_ptr(), _ld(y), rows, Cc, dz.data_ptr(), _ld(dz), _p(argmax), int(K),
                st.scale.data_ptr(), st.shift.data_ptr(), st.mean.data_ptr(), st.invstd.data_ptr(), int(relu),
                acc[0].data_ptr(), acc[1].data_ptr(), dy.data_ptr(), Cc, dgamma.data_ptr(), dbeta.data_ptr(), _stream())
    return (dy, dgamma, dbeta) if fresh else dy


GRAD_TC_MIN_TILE = int(os.environ.get("PN12_GRAD_TC_MIN", "1024"))     # cout * cin from which the 128 x 128 tensor-core tile is worth its padding


def grad_weight(dy: torch.Tensor, x: torch.Tensor, dw: torch.Tensor, db: Optional[torch.Tensor],
                engine: str = "auto", x_stats: Optional[BatchStats] = None, x_relu: bool = True) -> None:
    """dw [cout, cin] += dy^T x, db [cout] += column sums of dy (in place; the buffers hold zeros or a gradient).
    engine: "tc" (pn_grad_weight_bf16x3, tensor cores, 3-pass split bf16), "fp32" (pn_grad_weight_f32, CUDA cores) or
    "auto" (tensor cores unless the MLP mode is 'fp32' or the layer is tiny)."""
    dy, x = _rowmat(dy, "dy"), _rowmat(x, "x")
    rows, cout = dy.shape
    cin = x.shape[1]
    if x.shape[0] != rows or dw.shape != (cout, cin) or not dw.is_contiguous() or dw.dtype != torch.float32:
        raise ValueError("grad_weight: shape mismatch")
    if engine == "auto":
        engine = "tc" if (mlp_mode() == "bf16x3" and cout * cin >= GRAD_TC_MIN_TILE) else "fp32"
    if x_stats is not None:
        # x is the PRE-normalisation output of the previous layer: its normalise + ReLU is applied on load (tensor cores only)
        with _on_device(dy):
            nv.call("pn_grad_weight_bn_bf16x3", dy.data_ptr(), _ld(dy), x.data_ptr(), _ld(x), x_stats.scale.data_ptr(),
                    x_stats.shift.data_ptr(), int(x_relu), rows, cout, cin, dw.data_ptr(), cin, _p(db), _stream())
        return
    name = {"tc": "pn_grad_weight_bf16x3", "fp32": "pn_grad_weight_f32"}[engine]
    with _on_device(dy):
        nv.call(name, dy.data_ptr(), _ld(dy), x.data_ptr(), _ld(x), rows, cout, cin, dw.data_ptr(), cin, _p(db), _stream())


def transpose(w: torch.Tensor) -> torch.Tensor:
    w = _f32(w, "w").contiguous()
    r, c = w.shape
    out = torch.empty((c, r), dtype=torch.float32, device=w.device)
    with _on_device(w):
        nv.call("pn_transpose_f32", w.data_ptr(), r, c, out.data_ptr(), _stream())
    return out


def group_backward(dgrouped: torch.Tensor, col0: int, D: int, idx: torch.Tensor, N: int) -> torch.Tensor:
    """dgrouped [B*S*K, >= col0+D] -> dfeat [B, N, D] (scatter-add through the ball-query indices)."""
    dgrouped = _rowmat(dgrouped, "dgrouped")
    idx = _i64(idx, "idx")
    B, S, K = idx.shape
    dfeat = torch.zeros((B, N, D), dtype=torch.float32, device=dgrouped.device)
    with _on_device(dgrouped):
        nv.call("pn_group_bwd_f32", dgrouped.data_ptr(), _ld(dgrouped), int(col0), int(D), idx.data_ptr(), B, N, S, K,
                dfeat.data_ptr(), _stream())
    return dfeat


def three_interpolate_backward(dx: torch.Tensor, D1: int, D2: int, idx: torch.Tensor, weight: torch.Tensor, S: int):
    """dx [B*N, D1+D2] -> (dpoints1 [B,N,D1] or None, dpoints2 [B,S,D2])."""
    dx = _rowmat(dx, "dx")
    idx = _i64(idx, "idx")
    weight = _f32(weight, "weight").contiguous()
    B, N, _ = idx.shape
    dp1 = torch.empty((B, N, D1), dtype=torch.float32, device=dx.device) if D1 else None
    dp2 = torch.zeros((B, S, D2), dtype=torch.float32, device=dx.device)
    with _on_device(dx):
        nv.call("pn_three_interpolate_bwd_f32", dx.data_ptr(), _ld(dx), int(D1), int(D2), idx.data_ptr(), weight.data_ptr(),
                B, N, int(S), _p(dp1), dp2.data_ptr(), _stream())
    return dp1, dp2


def group_backward_xyz(dgrouped: torch.Tensor, col0: int, idx: torch.Tensor, N: int, recentred: bool = True):
    """Coordinate gradient of the grouping: dgrouped [B*S*K, >= col0+3] with the xyz_rel columns at col0 -> (dxyz [B,N,3],
    dnew_xyz [B,S,3] = -sum over each group, or None when the group was not recentred (group-all))."""
    dgrouped = _rowmat(dgrouped, "dgrouped")
    idx = _i64(idx, "idx")
    B, S, K = idx.shape
    dxyz = torch.zeros((B, N, 3), dtype=torch.float32, device=dgrouped.device)
    dnew = torch.empty((B, S, 3), dtype=torch.float32, device=dgrouped.device) if recentred else None
    with _on_device(dgrouped):
        nv.call("pn_group_bwd_xyz_f32", dgrouped.data_ptr(), _ld(dgrouped), int(col0), idx.data_ptr(), B, int(N), S, K,
                dxyz.data_ptr(), _p(dnew), _stream())
    return dxyz, dnew


def three_interpolate_backward_xyz(dx: torch.Tensor, D1: int, D2: int, idx: torch.Tensor, weight: torch.Tensor,
                                   points2: torch.Tensor, xyz1: torch.Tensor, xyz2: torch.Tensor):
    """three_interpolate_backward plus the gradient through the 3-NN weights: points2 [B,S,D2], xyz1 [B,N,3], xyz2 [B,S,3]
    (the forward's inputs, any strides) -> (dpoints1 [B,N,D1] or None, dpoints2 [B,S,D2], dxyz1 [B,N,3], dxyz2 [B,S,3]).
    Needs S >= 3."""
    dx = _rowmat(dx, "dx")
    idx = _i64(idx, "idx")
    weight = _f32(weight, "weight").contiguous()
    points2 = _cloud(points2, "points2")
    xyz1, xyz2 = _cloud(xyz1, "xyz1", 3), _cloud(xyz2, "xyz2", 3)
    B, N, _ = idx.shape
    S = points2.shape[1]
    dp1 = torch.empty((B, N, D1), dtype=torch.float32, device=dx.device) if D1 else None
    dp2 = torch.zeros((B, S, D2), dtype=torch.float32, device=dx.device)
    dxyz1 = torch.empty((B, N, 3), dtype=torch.float32, device=dx.device)
    dxyz2 = torch.zeros((B, S, 3), dtype=torch.float32, device=dx.device)
    with _on_device(dx):
        nv.call("pn_three_interpolate_bwd_xyz_f32", dx.data_ptr(), _ld(dx), int(D1), int(D2), idx.data_ptr(), weight.data_ptr(),
                points2.data_ptr(), *points2.stride(), xyz1.data_ptr(), *xyz1.stride(), xyz2.data_ptr(), *xyz2.stride(), B, N, S,
                _p(dp1), dp2.data_ptr(), dxyz1.data_ptr(), dxyz2.data_ptr(), _stream())
    return dp1, dp2, dxyz1, dxyz2


def dropout(x: torch.Tensor, p: float, seed_offset: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None,
            want_mask: bool = True):
    """-> (y, mask uint8 [rows, C]).  mask given: applied as is (also the backward pass); else drawn from the Philox
    stream named by seed_offset (uint64/int64 [2] on the device: seed, offset)."""
    x = _rowmat(x, "x")
    rows, Cc = x.shape
    y = torch.empty((rows, Cc), dtype=torch.float32, device=x.device)
    out_mask = None
    if mask is None:
        if seed_offset is None:
            raise ValueError("dropout needs a mask or a seed")
        out_mask = torch.empty((rows, Cc), dtype=torch.uint8, device=x.device) if want_mask else None
    elif mask.dtype != torch.uint8 or mask.numel() != rows * Cc or not mask.is_contiguous():
        raise ValueError("mask must be a contiguous uint8 [rows, C] tensor")
    with _on_device(x):
        nv.call("pn_dropout_f32", x.data_ptr(), _ld(x), rows, Cc, float(p), _p(seed_offset), _p(mask), _p(out_mask),
                y.data_ptr(), Cc, _stream())
    return y, (mask if mask is not None else out_mask)


def cross_entropy(x: torch.Tensor, target: torch.Tensor, want_grad: bool = True, grad_scale: float = 1.0):
    """nn.CrossEntropyLoss() over rows x [rows, C], target [rows] -> (loss 0-d tensor, dx or None).  Label -100 is
    ignored (its default ignore_index): left out of the mean, zero gradient."""
    x = _rowmat(x, "x")
    target = _i64(target.reshape(-1), "target")
    rows, Cc = x.shape
    if target.numel() != rows:
        raise ValueError("target must hold one label per row")
    scratch = torch.empty((2,), dtype=torch.float64, device=x.device)
    loss = torch.empty((), dtype=torch.float32, device=x.device)
    dx = torch.empty((rows, Cc), dtype=torch.float32, device=x.device) if want_grad else None
    with _on_device(x):
        nv.call("pn_cross_entropy_f32", x.data_ptr(), _ld(x), target.data_ptr(), rows, Cc, scratch.data_ptr(),
                loss.data_ptr(), _p(dx), Cc, float(grad_scale), _stream())
    return loss, dx


def log_softmax_backward(dy: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    dy, y = _rowmat(dy, "dy"), _rowmat(y, "y")
    rows, Cc = y.shape
    dx = torch.empty((rows, Cc), dtype=torch.float32, device=y.device)
    with _on_device(y):
        nv.call("pn_log_softmax_bwd_f32", dy.data_ptr(), _ld(dy), y.data_ptr(), _ld(y), rows, Cc, dx.data_ptr(), Cc, _stream())
    return dx


def adam_step(param: torch.Tensor, grad: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, step: int,
              lr: float, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0, grad_scale: float = 1.0) -> None:
    """One torch.optim.Adam update of a flat float32 buffer, in place."""
    for t, name in ((param, "param"), (grad, "grad"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
        _need_cuda(t, name)
        if t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != param.numel():
            raise ValueError(f"{name} must be a contiguous float32 buffer of the parameter's size")
    with _on_device(param):
        nv.call("pn_adam_f32", param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), param.numel(),
                float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay), int(step), float(grad_scale),
                _stream())


def adam_step_dev(param: torch.Tensor, grad: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor,
                  lr: torch.Tensor, step: torch.Tensor, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0,
                  grad_scale: float = 1.0) -> None:
    """adam_step with the learning rate (float32 [1]) and the step counter (int64 [1], incremented by the call) on the
    device: capturable in a CUDA graph."""
    with _on_device(param):
        nv.call("pn_adam_dev_f32", param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), param.numel(),
                lr.data_ptr(), step.data_ptr(), float(betas[0]), float(betas[1]), float(eps), float(weight_decay),
                float(grad_scale), _stream())


def seg_metrics(logp: torch.Tensor, target: torch.Tensor, want_pred: bool = False):
    """logp [..., C] log-probabilities, target [...] -> counts int64 [3C+1] (intersection | predicted | target per class,
    then correct points) and optionally the arg-max labels."""
    Cc = logp.shape[-1]
    x = _rowmat(_f32(logp, "logp").reshape(-1, Cc), "logp")
    target = _i64(target.reshape(-1), "target")
    rows = x.shape[0]
    if target.numel() != rows:
        raise ValueError("target must hold one label per point")
    counts = torch.empty((3 * Cc + 1,), dtype=torch.int64, device=x.device)
    pred = torch.empty((rows,), dtype=torch.int64, device=x.device) if want_pred else None
    with _on_device(x):
        nv.call("pn_seg_metrics_f32", x.data_ptr(), _ld(x), target.data_ptr(), rows, Cc, _p(pred), counts.data_ptr(), _stream())
    return (counts, pred.view(logp.shape[:-1])) if want_pred else counts

