"""CUDA-graph replay of a network forward, with several batches in flight.

A PointNet2SemSeg forward is ~40 kernel launches spread over six streams; captured once per input shape it replays as
a single graph launch, with the fork/join between the streams preserved as graph dependencies.  Only device memory,
streams and graphs come from PyTorch; every node of the graph is one of our kernels.

    runner = GraphedSemSeg(net)            # net: PointNet2SemSeg or the load_pointnet wrapper, in eval mode
    logp = runner(points)                  # points [B, 4, N] on the device or in (pinned) host memory

Batches in flight (`depth` > 1).  One forward is a long serial phase on a third of the SMs (level-1 farthest-point sampling:
1024 dependent iterations per cloud) followed by tensor-core chains that want the whole GPU; consecutive batches are
independent (the reference's loop `for points, target in loader: pred = model(points)`, pcdseg.py:58-97), so the runner keeps
`depth` static buffer sets with one captured graph each and replays them on their own streams: the sampling of batch k+1 runs
beside the chains of batch k.  The resident-weight chain kernels then hand out their row tiles dynamically (ops.TileCounters),
because a persistent CTA may get its SM only when a sampling cluster of the other batch has left it.

    t1 = runner.submit(batch1)             # asynchronous: copies the input, replays set (k % depth)
    t2 = runner.submit(batch2)
    logp1 = runner.result(t1)              # orders the current stream (device output) or the host (to_host) after batch 1
    ...                                    # a result stays valid until `depth` further submits

The FPS start indices are drawn on the CPU generator for every batch, exactly like the reference (pointnet_util.py:75),
and reach the graph's static buffer through a small ring of pinned staging buffers.
"""
from __future__ import annotations

import operator
import os
import time
from collections import deque
from typing import Dict, List, Optional, Tuple

import torch

from . import ops

_VERSION_OF = operator.attrgetter("_version")


class Ticket:
    """Handle of a submitted batch (GraphedSemSeg.submit)."""

    __slots__ = ("set", "seq", "done", "to_host")

    def __init__(self, st, seq, done, to_host):
        self.set, self.seq, self.done, self.to_host = st, seq, done, to_host


class Pacer:
    """Spacing of the submits of a host-output loop (GraphedSemSeg.pace).

    The host waits for batch k before it submits batch k + depth; left alone, the batches in flight fall into step: they finish
    in a burst, the host resubmits in a burst, all of them sample at once and then all of them run their chains.  Submits are
    therefore spaced at least `factor` x the running time per batch apart.  That time is estimated over windows of `window`
    completions: if the host had to wait for any of them the GPU set the rate (followed upwards by 5 % per window at most, so that a
    hiccup does not throttle what comes after it); if it never waited, the spacing itself set the rate and is shortened by 7 %.
    Pure host logic (clock and sleep are injectable: tests/test_host_cpu.py)."""

    def __init__(self, factor: float, window: int = 8, clock=time.perf_counter):
        self.factor, self.clock = float(factor), clock
        self.done_at = deque(maxlen=window)
        self.blocked = 0
        self.per_batch = None          # running seconds per batch
        self.in_flight = 0
        self.last_submit = 0.0

    def next_submit_time(self) -> float:
        """Earliest time of the next submit (0.0: at once)."""
        if self.in_flight <= 0:        # the pipeline ran empty: completion times before the pause say nothing
            self.done_at.clear()
            self.blocked = 0
        return self.last_submit + self.factor * self.per_batch if self.per_batch is not None else 0.0

    def submitted(self) -> None:
        self.last_submit = self.clock()
        self.in_flight += 1

    def completed(self, waited: float) -> None:
        """A result was handed out; `waited`: seconds the host spent blocked on it."""
        self.in_flight = max(0, self.in_flight - 1)
        self.blocked += waited > 20e-6
        self.done_at.append(self.clock())
        if len(self.done_at) == self.done_at.maxlen:
            seen = (self.done_at[-1] - self.done_at[0]) / (len(self.done_at) - 1)
            if self.per_batch is None:
                self.per_batch = seen
            elif self.blocked:
                self.per_batch = min(max(seen, 0.93 * self.per_batch), 1.05 * self.per_batch)
            else:
                self.per_batch *= 0.93
            self.done_at.clear()
            self.blocked = 0


class GraphedSemSeg:
    """Shape-keyed CUDA-graph cache around PointNet2SemSeg.forward with `depth` batches in flight."""

    RING = 4
    FPS1_PIPELINED = (3, 256, 2)          # depth 2..7: 3 CTAs x 8 warps per cloud
    FPS1_DEEP = (2, 256, 2)               # depth >= 8: 2 CTAs x 8 warps, 48 points per thread

    def __init__(self, net, warmup: int = 2, depth: int = 1):
        self.net = net.module if hasattr(net, "module") else net
        self.warmup = warmup
        self.depth = max(1, int(depth))
        self.timing = False                       # True: tickets carry timing-enabled completion events (benchmarks)
        self._graphs: Dict[Tuple, dict] = {}
        self._tensors = list(self.net.parameters()) + list(self.net.buffers())
        self._sig, self._vsum, self._checks, self._last_check = None, 0, 0, 0.0
        # host-output modes: submits are spaced >= pace x the running time per batch apart (class Pacer; state per shape and mode)
        self.pace = float(os.environ.get("PN12_PIPE_PACE", "0.92")) if self.depth > 1 else 0.0

    # ---- the captured graphs bake in the device pointers of the folded / packed weights: any change of a parameter or
    # BatchNorm buffer (optimizer step, load_state_dict, .to()) must rebuild them (and must not replay freed blobs)
    def _signature(self):
        return tuple((t.data_ptr(), t._version) for t in self._tensors)

    def _versions(self) -> int:
        return sum(map(_VERSION_OF, self._tensors))

    def _check_weights(self, dev):
        # The full signature (pointer and version of 156 tensors for PointNet2SemSeg) costs ~50 us of host time, half of a submit.
        # One batch at a time it is taken on every call.  With batches in flight a submit that follows the previous one within
        # 2 ms only sums the version counters (~20 us: every in-place update -- optimizer step, load_state_dict, copy_ -- bumps
        # one); the pointers (.to(), .data reassignment) are compared after any pause and on every 64th submit.
        now = time.perf_counter()
        self._checks += 1
        full = self.depth == 1 or self._sig is None or now - self._last_check > 2e-3 or (self._checks & 63) == 0
        self._last_check = now
        if full:
            sig = self._signature()
            changed = sig != self._sig
        else:
            changed = self._versions() != self._vsum
            sig = self._signature() if changed else self._sig
        if changed:
            if self._graphs:
                torch.cuda.synchronize(dev)       # replays in flight still read the old blobs
                self._graphs.clear()
            self._sig, self._vsum = sig, self._versions()

    def _capture_options(self, st) -> dict:
        """Launch options of a captured forward.  With several batches in flight what counts is the SM time a batch occupies,
        not the latency of one forward: level-1 sampling runs on 3 or (deep pipelines) 2 CTAs of 8 warps per cloud instead of
        the latency-optimal 8 CTAs x 4 warps (0.73 / 1.00 ms instead of 0.48 ms, on 24 / 16 SMs instead of 64 at C2), and the
        level-1 ball query runs after it on the whole GPU instead of polling beside it on SMs the other batches' chains can
        use (measured at C2, B200: profiles/r02_summary.md sections 1 and 6)."""
        if self.depth == 1:
            return {"tile_counters": None}
        # (the last level is NOT cut into batch slices for the host output: the copy of batch k overlaps batch k+1 anyway, and
        # eight one-cloud launches of fp1 + head quantise badly: 188 tiles on 148 SMs each)
        return {"tile_counters": st["counters"], "fps1_config": self.fps1_shape(st["x"].shape[2]), "stream_ball": False,
                "host_out_slices": int(os.environ.get("PN12_PIPE_HOST_SLICES", "1"))}

    def fps1_shape(self, N: int) -> Optional[Tuple[int, int, int]]:
        """Launch shape (cluster, threads, exchange) of the level-1 sampling with batches in flight: the fewest CTAs of 8 warps
        whose threads can hold the cloud in registers (48 points each), from 2 (depth >= 8) or 3 upwards; None (the automatic,
        latency-optimal shape) for one batch at a time and for clouds beyond 8 x 256 x 48 points."""
        if self.depth == 1:
            return None
        first = self.FPS1_DEEP if self.depth >= 8 else self.FPS1_PIPELINED
        for cluster in (2, 3, 4, 8):
            if cluster >= first[0] and N <= cluster * 256 * 48:
                return (cluster, 256, 2)
        return None

    def _build_set(self, points: torch.Tensor, to_host: bool) -> dict:
        net, dev = self.net, points.device
        B, C, N = points.shape
        sizes = [N] + [m.npoint for m in (net.sa1, net.sa2, net.sa3)]
        st = {
            "x": torch.empty((B, C, N), dtype=torch.float32, device=dev),
            "starts": torch.zeros((len(sizes), B), dtype=torch.int64, device=dev),
            "sizes": sizes,
            "pinned": [torch.zeros((len(sizes), B), dtype=torch.int64).pin_memory() for _ in range(self.RING)],
            "events": [None] * self.RING,
            "ready": torch.cuda.Event(),
            "slot": 0,
            "stream": torch.cuda.Stream(dev),
            "counters": ops.TileCounters(dev, 128) if self.depth > 1 else None,
            "seq": -1,
        }
        st["x"].copy_(points)
        classes = net.conv2.out_channels
        labels = to_host == "labels"
        st["host_out"] = torch.empty((B, N, classes), dtype=torch.float32).pin_memory() if (to_host and not labels) else None
        st["host_labels"] = torch.empty((B, N), dtype=torch.uint8).pin_memory() if labels else None
        stream = st["stream"]
        stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(stream), torch.no_grad():
            for _ in range(self.warmup):             # folds BatchNorm, packs weights, sizes the allocator pools
                with ops.options(**{k: v for k, v in self._capture_options(st).items() if k != "tile_counters"}):
                    net(st["x"], fps_starts=list(st["starts"].unbind(0)), host_out=st["host_out"])
        torch.cuda.current_stream(dev).wait_stream(stream)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        with ops.options(**self._capture_options(st)):
            with torch.cuda.graph(graph, stream=stream), torch.no_grad():
                st["out"] = net(st["x"], fps_starts=list(st["starts"].unbind(0)), host_out=st["host_out"])
                if labels:      # what the reference's evaluation loop keeps of the output: pred.argmax(-1) (pcdseg.py:75)
                    st["labels"] = ops.argmax_labels(st["out"])
                    st["host_labels"].copy_(st["labels"], non_blocking=True)
        st["graph"] = graph
        return st

    def _sets(self, points: torch.Tensor, dev, to_host) -> dict:
        self._check_weights(dev)
        mode = "labels" if to_host == "labels" else bool(to_host)
        key = (tuple(points.shape), dev, mode)
        entry = self._graphs.get(key)
        if entry is None:
            on_dev = points.to(dev)
            entry = self._graphs[key] = {"sets": [self._build_set(on_dev, mode) for _ in range(self.depth)], "n": 0,
                                           "pace": Pacer(self.pace)}
            for st in entry["sets"]:
                st["pace"] = entry["pace"]
            self._sig, self._vsum = self._signature(), self._versions()   # (the warm-up folded the weights; nothing changed)
        return entry

    @torch.no_grad()
    def submit(self, points: torch.Tensor, to_host=False) -> Ticket:
        """Starts the forward of one batch on the next buffer set and returns at once.  `points`: device tensor (ordered
        after the work already queued on the current stream) or pinned host tensor (copied by the set's own stream).
        to_host: False (device log-probabilities), True (log-probabilities [B, N, classes] into the set's pinned host buffer)
        or "labels" (only pred.argmax(-1) as uint8 [B, N] travels to the host: what the reference's evaluation loop uses,
        pcdseg.py:75 -- 1 byte per point instead of 76)."""
        dev = points.device if points.is_cuda else torch.device("cuda", torch.cuda.current_device())
        entry = self._sets(points, dev, to_host)
        if to_host and self.pace > 0.0:
            until = entry["pace"].next_submit_time()
            while True:                               # sleep (the interpreter lock is free for other threads), spin the last 0.1 ms
                rem = until - time.perf_counter()
                if rem <= 0.0:
                    break
                if rem > 150e-6:
                    time.sleep(rem - 100e-6)
            entry["pace"].submitted()
        seq = entry["n"]
        entry["n"] = seq + 1
        st = entry["sets"][seq % self.depth]
        st["seq"] = seq
        B = points.shape[0]
        slot = st["slot"] = (st["slot"] + 1) % self.RING
        ev = st["events"][slot]
        if ev is not None:
            ev.synchronize()                          # the copy that last used this staging buffer has run
        else:
            ev = st["events"][slot] = torch.cuda.Event()
        pinned = st["pinned"][slot]
        for i, n in enumerate(st["sizes"]):           # the reference's draws, same generator, same order, straight into pinned memory
            torch.randint(0, n, (B,), dtype=torch.long, out=pinned[i])
        stream = st["stream"]
        # ordered after the caller's stream: a device input exists from here on, and whatever the caller queued to consume
        # the result this set held before (`depth` submits ago) has been issued ahead of this point
        ready = st["ready"]                           # (events are reused: the host side of a submit is ~100 us, all of it on the
        ready.record()                                #  critical path of a short run's pipeline fill)
        stream.wait_event(ready)
        if points.is_cuda:
            points.record_stream(stream)
        with torch.cuda.stream(stream):
            st["starts"].copy_(pinned, non_blocking=True)
            ev.record()
            st["x"].copy_(points, non_blocking=True)
            st["graph"].replay()
            done = torch.cuda.Event(enable_timing=self.timing)
            done.record()
        return Ticket(st, seq, done, "labels" if to_host == "labels" else bool(to_host))

    def result(self, ticket: Ticket) -> torch.Tensor:
        """The log-probabilities [B, N, classes] of a submitted batch.  Device output: the set's static buffer, ordered before
        whatever the caller queues next on the current stream.  to_host: the set's static PINNED HOST buffer, complete on
        return (the host waits for that batch only).  Valid until `depth` further submits reuse the set."""
        if ticket.set["seq"] != ticket.seq:
            raise RuntimeError(f"the result of batch {ticket.seq} was overwritten: at most depth={self.depth} batches are in flight")
        if ticket.to_host:
            t0 = time.perf_counter()
            ticket.done.synchronize()
            if self.pace > 0.0:
                ticket.set["pace"].completed(time.perf_counter() - t0)
            return ticket.set["host_labels"] if ticket.to_host == "labels" else ticket.set["host_out"]
        torch.cuda.current_stream(ticket.set["out"].device).wait_event(ticket.done)
        return ticket.set["out"]

    @torch.no_grad()
    def __call__(self, points: torch.Tensor, out: torch.Tensor = None, to_host: bool = False) -> torch.Tensor:
        """One batch, start to finish: submit + result.  Returns the static output buffer (valid until `depth` further
        calls) or, when `out` is given (device or pinned host), copies the log-probabilities there asynchronously.
        to_host=True: the device-to-host copies are nodes of the graph (the last level runs in batch slices and the first
        clouds travel while the last are computed); returns the runner's static PINNED HOST buffer."""
        res = self.result(self.submit(points, to_host=to_host))
        if to_host:
            return res
        if out is not None:
            out.copy_(res, non_blocking=True)
            return out
        return res

    def run_pipelined(self, batches, to_host=False, consume=None) -> Optional[List[torch.Tensor]]:
        """The reference's evaluation loop (pcdseg.py:58-97) with `depth` batches in flight: submits batch k + depth - 1
        before it hands batch k's result to `consume(k, logp)` (default: collect clones)."""
        pending, results = [], []
        for k, pts in enumerate(batches):
            pending.append((k, self.submit(pts, to_host=to_host)))
            if len(pending) >= self.depth:
                j, t = pending.pop(0)
                r = self.result(t)
                results.append(consume(j, r) if consume is not None else r.clone())
        for j, t in pending:
            r = self.result(t)
            results.append(consume(j, r) if consume is not None else r.clone())
        return results


class PinnedRing:
    """Pinned int64 host buffers that stage values for a graph's static device buffer, used in turn: `next()` returns the
    next buffer once the copy that last read it has run; `send(dst)` copies it to `dst` with one asynchronous copy on the
    current stream."""

    def __init__(self, shape, depth: int):
        self.bufs = [torch.zeros(shape, dtype=torch.int64).pin_memory() for _ in range(depth)]
        self.events = [None] * depth
        self.slot = 0

    def next(self) -> torch.Tensor:
        self.slot = (self.slot + 1) % len(self.bufs)
        if self.events[self.slot] is not None:
            self.events[self.slot].synchronize()
        return self.bufs[self.slot]

    def send(self, dst: torch.Tensor) -> None:
        dst.copy_(self.bufs[self.slot], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self.events[self.slot] = ev


class GraphedModule:
    """CUDA-graph replay of any eval-mode network of this package, one batch at a time.  PointNetSeg / PointNetCls /
    PointNetDenseCls (model/pointnet.py) draw nothing on the host; the PointNet++ classification / part-segmentation nets
    (model/pointnet2.py) draw one FPS start index per sampling level and cloud: the runner draws them for every call on the CPU
    generator, in the reference's order (pointnet_util.py:75), and feeds the graph's static buffer (`fps_level_sizes`).
    Config C1 (PointNetSeg, one cloud of 24000 points) is ~25 launches of a few microseconds each plus per-call host glue, config
    C4 (PointNet2ClsMsg, 32 clouds of 1024 points) ~70; captured once per input shape each is one graph launch.  Returns the
    graph's static output tensors (valid until the next call); rebuilt when a parameter or BatchNorm buffer changes."""

    RING = 4

    def __init__(self, net, warmup: int = 2):
        self.net = net.module if hasattr(net, "module") else net
        self.warmup = warmup
        self._graphs: Dict[Tuple, dict] = {}
        self._tensors = list(self.net.parameters()) + list(self.net.buffers())
        self._sig = None

    def _signature(self):
        return tuple((t.data_ptr(), t._version) for t in self._tensors)

    def _forward(self, st):
        if st["starts"] is not None:
            return self.net(*st["in"], fps_starts=list(st["starts"].unbind(0)))
        return self.net(*st["in"])

    @torch.no_grad()
    def __call__(self, *inputs: torch.Tensor):
        dev = next((t.device for t in inputs if t.is_cuda), torch.device("cuda", torch.cuda.current_device()))
        sig = self._signature()
        if sig != self._sig:
            if self._graphs:
                torch.cuda.synchronize(dev)
                self._graphs.clear()
            self._sig = sig
        key = tuple((tuple(t.shape), t.dtype) for t in inputs) + (dev,)
        st = self._graphs.get(key)
        B = inputs[0].shape[0]
        if st is None:
            st = {"in": [torch.empty(t.shape, dtype=t.dtype, device=dev) for t in inputs], "starts": None}
            sizes = self.net.fps_level_sizes(inputs[0].shape[2]) if hasattr(self.net, "fps_level_sizes") else []
            if sizes:
                st["sizes"] = sizes
                st["starts"] = torch.zeros((len(sizes), B), dtype=torch.int64, device=dev)
                st["ring"] = PinnedRing((len(sizes), B), self.RING)
            for s, t in zip(st["in"], inputs):
                s.copy_(t)
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(self.warmup):
                    self._forward(st)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                st["out"] = self._forward(st)
            st["graph"] = graph
            self._graphs[key] = st
            self._sig = self._signature()
        if st["starts"] is not None:
            pinned = st["ring"].next()
            for i, n in enumerate(st["sizes"]):           # the reference's draws, same generator, same order
                pinned[i] = torch.randint(0, n, (B,), dtype=torch.long)
            st["ring"].send(st["starts"])
        for s, t in zip(st["in"], inputs):
            s.copy_(t, non_blocking=True)
        st["graph"].replay()
        return st["out"]
