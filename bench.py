"""bench.py -- PointNet++ SSG semantic-segmentation forward, points/sec (BASELINE.json metric, config C2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--depth D] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One step = one eval forward of PointNet2SemSeg (the reference's shipped pointnet2-inview checkpoint) over a
batch of 8 synthetic KITTI-shaped clouds of 24 000 points (xyz + reflectance) per GPU.  Clouds are
independent, so ranks shard the work with no data-path collective (weak scaling: 8 clouds per GPU).

Our arm prints one JSON line with
  value          whole-job points/sec, inputs resident in HBM, `depth` batches in flight (runtime.GraphedSemSeg), the K steps
                 timed as one region with CUDA events, max over ranks; inputs rotate over 48 different batches (> L2)
  sequential     the same one batch at a time with per-step events and an L2 flush between steps (round-1 protocol)
  e2e            the same loop from pinned HOST batches to pinned HOST [B,N,19] log-probabilities (H2D and D2H in the region)
  e2e_labels     ... moving only pred.argmax(-1) (uint8) to the host: what the reference's evaluation loop consumes
  roofline       the dominant kernel (level-1 farthest-point sampling at N=24000): algorithmic bytes B*npoint*N*16 per
                 launch / launch duration (CUDA events, stand-alone, cold L2) against the measured HBM copy bandwidth
  roofline_all   every kernel group of the forward timed alone, against its roofline (tools/kernel_rooflines.py)
  cpu_baseline   the UNMODIFIED reference (baseline/_ref: model/utils.py load_pointnet + eval forward) on the host CPUs,
                 CUDA hidden, in a child process; cpu_baseline_port = the C/OpenMP oracle port (oracle/)
  train, dp_check  config C5 (training iteration with the NCCL gradient all-reduce) and the data-parallel equivalence check
`--impl reference` runs that unmodified reference as the reference arm (rank 0 only under torchrun), same metric and `config`.
`--dump-outputs DIR` (our arm, c2) writes what the last step of each timed region returned to its caller, as float32 .npy files
(rank 0's): log_probs [B, N, 19] (inputs in HBM), e2e_log_probs [B, N, 19] (pinned host) and e2e_labels [B, N] (argmax), 30 MB
in all.  The inputs and the FPS start draws of the timed steps are seeded, so two runs with the same arguments, on two builds,
can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CKPT = os.path.join(ROOT, "tests", "golden", "pointnet2-inview-0.55884-0001.pth")
BATCH, NPOINTS, CLASSES = 8, 24000, 19
BASE_BATCHES, NB_INPUTS = 12, 48     # 96 synthetic clouds, combined into 48 different batches (147 MB > L2)
LEVEL_N = (24000, 1024, 256, 64)
METRIC = "pointnet2_semseg_forward_points_per_sec"
FPS_DRAM_BYTES_PER_LAUNCH = 2337024   # ncu: 2.34 MB read + 0 written per level-1 launch (the cloud lives in registers)
FPS_ENTRY_POINTS = ["pn_fps_f32", "pn_fps_progress_f32"]   # the same kernel with / without the progress feed
WORKLOAD = "C2: PointNet2SemSeg(19, feature_dims=1) eval forward, pointnet2-inview checkpoint, 8 synthetic KITTI-shaped clouds x 24000 points per GPU"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU legs (our arm only)")
    ap.add_argument("--depth", type=int, default=int(os.environ.get("PN12_DEPTH", "10")), help="batches in flight (GraphedSemSeg depth)")
    ap.add_argument("--ref-clouds", type=int, default=0, help="reference arm: clouds per step (0 = the full batch of 8, reduced "
                                                              "automatically if the run would exceed a few minutes)")
    ap.add_argument("--no-train", action="store_true", help="skip the config-C5 `train` / `dp_check` sub-records")
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "bf16", "fp32"],
                    help="bf16x3 (default, fp32 parity), bf16 (single-pass, stated tolerance) or fp32 (CUDA cores)")
    ap.add_argument("--workload", default="c2", choices=["c2", "train", "preprocess"],
                    help="c2 (default): the headline eval forward; train: config C5, one training iteration per step "
                         "(tools/bench_train.py; same JSON contract); preprocess: raw scans -> network input (tools/bench_preprocess.py)")
    ap.add_argument("--mode", default="graph", choices=["graph", "eager"],
                    help="graph: one CUDA-graph replay per step (default); eager: ~40 launches per step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step of each region as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c2"):
        ap.error("--dump-outputs covers the c2 workload of --impl ours")
    return args


def dump_outputs(path, arrays):
    """--dump-outputs: one float32 DIR/<name>.npy per array."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


_NVML_POLLER = r"""
import sys, time, threading
import pynvml as n
n.nvmlInit()
h = n.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
ev = lambda a, b, d: getattr(n, a, getattr(n, b, d))
bits = [ev("nvmlClocksEventReasonHwSlowdown", "nvmlClocksThrottleReasonHwSlowdown", 0x8),
        ev("nvmlClocksEventReasonHwThermalSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
        ev("nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
        ev("nvmlClocksEventReasonSwPowerCap", "nvmlClocksThrottleReasonSwPowerCap", 0x4)]
reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
stop = threading.Event()
threading.Thread(target=lambda: (sys.stdin.readline(), stop.set()), daemon=True).start()
rows = []
def sample():
    m = reasons(h)
    rows.append("%.6f,%d,%d,%s" % (time.time(), n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM), mx,
                                   ",".join("Active" if m & b else "Not Active" for b in bits)))
sample()
print("ready", flush=True)
while not stop.is_set() and len(rows) < 200000:
    sample()
    time.sleep(float(sys.argv[2]))
print("\n".join(rows), flush=True)
"""


class ClockSampler:
    """Samples SM clocks / throttle reasons of one GPU while the timed region runs.

    The timed region is ~20 ms, shorter than one `nvidia-smi -lms` period (and than nvidia-smi's start-up on an 8-GPU
    box), so the samples come from NVML directly -- the library nvidia-smi itself reads -- every 2 ms in a thread:
    clocks.sm, clocks.max.sm and the clocks_event_reasons bits hw_slowdown / hw_thermal_slowdown / sw_thermal_slowdown /
    sw_power_cap of the recipe's clocks line.  nvidia-smi is the fallback when NVML cannot be loaded."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.nvml, self.stop = index, [], None, None, threading.Event()
        self.source = None

    def __enter__(self):
        # the sampling thread shares the interpreter lock with a main thread that is busy submitting batches: with the default
        # 5 ms switch interval it got 1-10 samples per run; 0.5 ms lets it sample every ~2 ms as intended
        self._switch = sys.getswitchinterval()
        sys.setswitchinterval(5e-4)
        # first choice: a helper PROCESS that polls NVML every 2 ms and time-stamps its rows (the in-process thread below
        # shares the interpreter lock and the driver's per-process locks with the thread that launches the work, and got
        # anything between 1 and 11 samples per run); rows outside [enter, exit] are dropped
        self.t_enter, self.helper = time.time(), None
        try:
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[self.index]) if visible and visible.split(",")[self.index].isdigit() else self.index
            period = float(os.environ.get("PN12_CLOCK_PERIOD_MS", "2")) * 1e-3
            self.helper = subprocess.Popen([sys.executable, "-c", _NVML_POLLER, str(phys), str(period)], stdin=subprocess.PIPE,
                                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            if self.helper.stdout.readline().strip() != "ready":      # NVML initialised, first sample taken
                raise OSError("poller did not start")
            self.t_enter, self.source = time.time(), f"nvml (helper process, {period * 1e3:g} ms period)"
            return self
        except Exception:
            if self.helper is not None:
                self.helper.kill()
            self.helper = None
        try:
            import pynvml

            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[self.index]) if visible and visible.split(",")[self.index].isdigit() else self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml, self.source = pynvml, "nvml"
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return self
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.source = "nvidia-smi"
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _poll_nvml(self):
        n = self.nvml
        bits = [("hw_slowdown", n.nvmlClocksEventReasonHwSlowdown if hasattr(n, "nvmlClocksEventReasonHwSlowdown")
                 else n.nvmlClocksThrottleReasonHwSlowdown),
                ("hw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonHwThermalSlowdown",
                                                getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40))),
                ("sw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonSwThermalSlowdown",
                                                getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20))),
                ("sw_power_cap", getattr(n, "nvmlClocksEventReasonSwPowerCap",
                                         getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)))]
        reasons_fn = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        while True:                      # (at least one sample, taken at once: a region can be shorter than one NVML call)
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                mask = reasons_fn(self.handle)
                self.rows.append([str(sm), str(mx)] + ["Active" if mask & b else "Not Active" for _, b in bits])
            except Exception:
                pass
            if self.stop.is_set():
                break
            time.sleep(0.002)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        sys.setswitchinterval(self._switch)
        if self.helper is not None:
            t_exit = time.time()
            try:
                out, _ = self.helper.communicate(input="stop\n", timeout=5)
            except Exception:
                self.helper.kill()
                out = ""
            for line in out.splitlines():
                c = [x.strip() for x in line.split(",")]
                if len(c) == 7 and self.t_enter <= float(c[0]) <= t_exit:
                    self.rows.append(c[1:])
            return
        if self.nvml is not None:
            self.stop.set()
            self.thread.join(timeout=2)
            try:
                self.nvml.nvmlShutdown()
            except Exception:
                pass
        elif self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": self.source}


def fps_starts(torch, batch):
    """The four FPS start-index draws of one forward, exactly as the modules draw them (pointnet_util.py:75)."""
    return [torch.randint(0, n, (batch,), dtype=torch.long) for n in LEVEL_N]


def shared_config(depth):
    """`config` of BOTH arms (identical keys and values, so that the driver can compare them)."""
    return {
        "workload": WORKLOAD, "batch_per_gpu": BATCH, "points_per_cloud": NPOINTS,
        "launch": (f"B200 arm: one CUDA-graph replay per batch (6 internal streams forked/joined inside the graph), {depth} batches "
                   f"in flight on {depth} static buffer sets (GraphedSemSeg.submit / result: the level-1 sampling of batch k+1 runs "
                   "beside the tensor-core chains of batch k; chain tiles handed out dynamically); reference arm: the unmodified "
                   "model/utils.py load_pointnet + eval forward on the host CPU, all cores"),
        "l2": (f"inputs larger than L2: the timed steps rotate over {NB_INPUTS} different input batches "
               f"({NB_INPUTS * BATCH * 4 * NPOINTS * 4 / 1e6:.0f} MB resident in HBM / pinned host memory > 126 MB L2); "
               "the `sequential` sub-record writes 512 MiB between steps instead"),
        "fps_start": "torch.randint on the CPU generator per level and batch, as the reference draws it",
    }


# ------------------------------------------------------------------------------------------------ CPU legs
def oracle_forward_timer(batch):
    import torch

    from oracle import oracle as orc
    from pointnet12_b200 import synthetic as syn

    # torchrun exports OMP_NUM_THREADS=1 to every rank: the CPU arm uses all host cores explicitly
    orc.set_num_threads(os.cpu_count() or 1)
    sd = orc.numpy_state_dict(torch.load(CKPT, map_location="cpu"))
    pts = syn.kitti_batch(batch, NPOINTS, config=2)
    torch.manual_seed(0)
    starts = [s.numpy() for s in fps_starts(torch, batch)]

    def step():
        t = time.perf_counter()
        orc.pointnet2_semseg(sd, pts, starts)
        return time.perf_counter() - t

    return step, orc.num_threads()


def import_reference():
    """The UNMODIFIED reference package from baseline/_ref (tools/install_reference.py copies /root/reference/model/*.py there,
    byte for byte, with a sha256 manifest) as `_pn12_ref`; returns its model.utils module or None when it is absent / altered."""
    import importlib.util
    import types

    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import install_reference as inst

    if not inst.verify():
        return None
    base = os.path.join(inst.DST, "model")
    pkg = types.ModuleType("_pn12_ref")
    pkg.__path__ = [base]
    sys.modules["_pn12_ref"] = pkg
    mods = {}
    for name in ("pointnet_util", "pointnet", "pointnet2", "utils"):
        spec = importlib.util.spec_from_file_location(f"_pn12_ref.{name}", os.path.join(base, name + ".py"))
        m = importlib.util.module_from_spec(spec)
        sys.modules[spec.name] = m
        spec.loader.exec_module(m)
        mods[name] = m
    return mods["utils"], os.path.join(inst.DST, "checkpoints", os.path.basename(CKPT))


def run_reference(args):
    """Reference arm: the reference's OWN PyTorch-CPU path (model/utils.py:15-34 load_pointnet -> DataParallel(PointNet2SemSeg)
    .eval(), pointnet2.py:159-176) from baseline/_ref, on all host cores, same config / metric / unit.  CUDA is hidden from this
    process, so load_pointnet takes its `cuda not available` branch.  Falls back to the C/OpenMP oracle port (kind "port") only
    when baseline/_ref is missing."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):          # torchrun pins every rank to one thread
        os.environ.pop(k, None)
    import contextlib
    import io

    import torch

    from pointnet12_b200 import synthetic as syn

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = import_reference()
    clouds = BATCH if args.ref_clouds <= 0 else args.ref_clouds
    if ref is not None:
        utils, ckpt = ref
        with contextlib.redirect_stdout(io.StringIO()):       # load_pointnet prints '=> cuda not available'
            net = utils.load_pointnet("pointnet2", CLASSES, ckpt)
        kind, what = "reference", "unmodified reference (baseline/_ref: model/utils.py load_pointnet, torch %s CPU)" % torch.__version__
        pts = torch.from_numpy(syn.kitti_batch(BATCH, NPOINTS, config=2))

        def step(n):
            t = time.perf_counter()
            torch.manual_seed(0)                              # fixes the four FPS start draws (pointnet_util.py:75)
            with torch.no_grad():
                net(pts[:n])
            return time.perf_counter() - t
    else:
        stepper, cores = oracle_forward_timer(BATCH)
        kind, what = "port", "C/OpenMP oracle port (oracle/pn_oracle.c): baseline/_ref is absent"
        clouds = BATCH

        def step(n):
            return stepper()
    first = step(clouds)                                      # warm-up; also sizes the sample
    if args.ref_clouds <= 0 and kind == "reference" and first * (args.steps + 1) > 240.0:
        clouds = max(1, min(BATCH, int(BATCH * 240.0 / (first * (args.steps + 1)))))     # keep the run within a few minutes
    for _ in range(max(0, min(args.warmup, 2) - 1)):
        step(clouds)
    times = [step(clouds) for _ in range(args.steps)]
    total = sum(times)
    value = clouds * NPOINTS * args.steps / total
    sample = (f"{'full step' if clouds == BATCH else 'bounded sample'}: {clouds} clouds x {NPOINTS} points per step, {args.steps} steps after "
              f"{max(1, min(args.warmup, 2))} warm-up, {what}, {cores} threads on {os.cpu_count()} host CPUs")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(args.depth),
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def reference_leg_subprocess(depth):
    """The reference arm in a child process with CUDA hidden (1 warm-up + 1 timed full batch): the `cpu_baseline` of our line."""
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "OMP_NUM_THREADS", "MKL_NUM_THREADS")}
    env["CUDA_VISIBLE_DEVICES"] = ""
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1",
                              "--ref-clouds", str(BATCH), "--depth", str(depth)], env=env, capture_output=True, text=True, timeout=600)
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        return line["cpu_baseline"]
    except Exception as e:   # noqa: BLE001
        return {"value": None, "unit": "points/s", "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {e!r}"[:300]}


# ------------------------------------------------------------------------------------------------ our arm
def make_inputs(torch, rank):
    """NB_INPUTS different batches: every batch is a different combination of 8 of 96 synthetic clouds (a pinned host tensor
    [NB, 8, 4, N]); together they exceed the L2, so a timed step never finds its input cached."""
    import numpy as np

    from pointnet12_b200 import synthetic as syn

    base = np.concatenate([syn.kitti_batch(BATCH, NPOINTS, config=2, first=(rank * BASE_BATCHES + i) * BATCH) for i in range(BASE_BATCHES)])
    rng = np.random.default_rng(100 + rank)
    need = NB_INPUTS * BATCH
    order = np.concatenate([rng.permutation(len(base)) for _ in range((need + len(base) - 1) // len(base))])[:need]
    return torch.from_numpy(base[order].reshape(NB_INPUTS, BATCH, 4, NPOINTS)).pin_memory()


def run_ours(args):
    import torch
    import torch.distributed as dist

    from pointnet12_b200 import _native as nv
    from pointnet12_b200 import ops
    from pointnet12_b200.model.utils import load_pointnet
    from pointnet12_b200.runtime import GraphedSemSeg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from pointnet12_b200.dist import bind_to_gpu_numa

    numa = bind_to_gpu_numa(local) if world > 1 else {"gpu": local, "numa_node": None, "bound": False}

    # CPU legs first (rank 0 of a single-GPU run only): nothing else competes for the host cores yet
    cpu_legs = {}
    if world == 1 and not args.no_cpu_baseline:
        cpu_legs["cpu_baseline"] = reference_leg_subprocess(args.depth)
        step, threads = oracle_forward_timer(BATCH)
        step()
        times = [step() for _ in range(5)]
        cpu_legs["cpu_baseline_port"] = {"value": BATCH * NPOINTS * len(times) / sum(times), "unit": "points/s", "cores": threads,
                                         "kind": "port", "sample": f"5 forwards of the same {BATCH} x {NPOINTS} batch after 1 warm-up, "
                                                                   f"C/OpenMP oracle (oracle/pn_oracle.c) on {os.cpu_count()} host CPUs"}
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    ops.set_mlp_mode(args.precision)
    net = load_pointnet("pointnet2", CLASSES, CKPT, device=dev)
    host_batches = make_inputs(torch, rank)
    dev_batches = host_batches.to(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    depth = 1 if args.mode == "eager" else args.depth
    runner = GraphedSemSeg(net, depth=depth) if args.mode == "graph" else None
    seq_runner = GraphedSemSeg(net, depth=1) if args.mode == "graph" else None

    def region(batches, steps, to_host):
        """K steps with `depth` batches in flight, timed as ONE region on the device; returns (ms, per-step completion times,
        the output of the last step: a static buffer, valid until the next step)."""
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dones, pending, out = [], [], None
        start.record()
        for i in range(steps):
            if runner is None:
                with torch.no_grad():
                    x = batches[i % NB_INPUTS]
                    if to_host:
                        net(x.to(dev, non_blocking=True), host_out=eager_host_out)
                        out = eager_host_out
                    else:
                        out = net(x)
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                dones.append(ev)
                continue
            pending.append(runner.submit(batches[i % NB_INPUTS], to_host=to_host))
            if len(pending) >= depth:
                t = pending.pop(0)
                out = runner.result(t)        # device output: orders this stream after batch k; host output: waits for it
                dones.append(t.done)
        for t in pending:
            out = runner.result(t)
            dones.append(t.done)
        end.record()
        torch.cuda.synchronize()
        marks = sorted(start.elapsed_time(d) for d in dones)     # (batches run on their own streams and may finish out of order)
        return start.elapsed_time(end), [b - a for a, b in zip([0.0] + marks[:-1], marks)], out

    outputs = {}

    def keep(name, out):
        """--dump-outputs: a float32 host copy of a region's last output, taken before the next region reuses the buffer."""
        if args.dump_outputs and rank == 0:
            outputs[name] = out.to("cpu", torch.float32, copy=True).numpy()

    eager_host_out = torch.empty((BATCH, NPOINTS, CLASSES), dtype=torch.float32).pin_memory() if runner is None else None
    if runner is not None:
        runner.timing = True
    torch.manual_seed(1234 + rank)
    W = max(args.warmup, 3)
    # (with batches in flight the warm-up also fills the pipeline a few times over: the runner spaces its submits by the
    # running time per batch it has observed, runtime.GraphedSemSeg.pace)
    Wp = W + 10 * depth if runner is not None else W
    region(dev_batches, Wp, False)
    region(host_batches, Wp, True)
    if runner is not None:
        region(host_batches, Wp, "labels")
    barrier()
    # the FPS start draws of the timed steps then depend on the seed and --steps only, not on how many draws the warm-up made
    torch.manual_seed(1234 + rank)

    # ---- timed regions (the clock sampler spans all of them: one region is only ~10 ms long)
    with ClockSampler(local) as clocks:
        # 1: inputs resident in HBM, `depth` batches in flight
        ms, per_step, out = region(dev_batches, args.steps, False)
        keep("log_probs", out)
        barrier()
        # 2: end to end from pinned host memory and back (full log-probabilities)
        ms_e2e, _, out = region(host_batches, args.steps, True)
        keep("e2e_log_probs", out)
        barrier()
        # 3: the same with what the reference's evaluation loop keeps of the output: pred.argmax(-1) (pcdseg.py:75) as uint8
        ms_lab = 0.0
        if runner is not None:
            ms_lab, _, out = region(host_batches, args.steps, "labels")
            keep("e2e_labels", out)
            barrier()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)

    # ---- one batch at a time (round-1 protocol: per-step CUDA events, 512 MiB written between steps) for comparison
    seq = None
    if seq_runner is not None:
        evs = []
        for i in range(W + args.steps):
            flush.fill_(i & 0xFF)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            seq_runner(dev_batches[i % NB_INPUTS])
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        seq_ms = [a.elapsed_time(b) for a, b in evs[W:]]
        seq = sum(seq_ms) / len(seq_ms)
    barrier()

    # launches per forward (= kernel nodes a replay runs), counted on an eager forward
    l0 = nv.launch_count
    with torch.no_grad():
        net(dev_batches[0])
    per_forward = nv.launch_count - l0
    torch.cuda.synchronize()

    t = torch.tensor([ms, ms_e2e, seq if seq is not None else 0.0, ms_lab], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e, seq, ms_lab = float(t[0]), float(t[1]), float(t[2]), float(t[3])
    points = world * BATCH * NPOINTS * args.steps

    line = None
    if rank == 0:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import kernel_rooflines

        torch.manual_seed(0)
        st = [s.to(dev) for s in fps_starts(torch, BATCH)]
        fps1_shape = runner.fps1_shape(NPOINTS) if runner is not None else None
        per_kernel = kernel_rooflines.measure(net, dev_batches[0], st, fps1_config=fps1_shape)
        fps1 = next(k for k in per_kernel["kernels"] if k["name"] == "fps level 1")
        spread = sorted(per_step)
        precision = ops.mlp_precision()
        cfg = shared_config(depth)
        cfg["precision"] = {"bf16x3": "bf16x3: tcgen05 tensor cores, 3-pass split bf16 with fp32 accumulation (fp32 parity, ~1e-5 relative)",
                            "bf16": "bf16: tcgen05 tensor cores, single pass (max |delta log-prob| 0.38, 99.6 % equal labels at this config)",
                            "fp32": "fp32 FMA on CUDA cores"}[precision] if args.precision != "bf16x3" else None
        if cfg["precision"] is None:
            del cfg["precision"]                 # (default mode: both arms then carry identical `config` objects)
        line = {
            "metric": METRIC, "value": points / (ms * 1e-3), "unit": "points/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "warmup_steps_run": Wp, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": {"bf16x3": "f32 (MLP products as split bf16 hi/lo on tensor cores)", "bf16": "bf16 (fp32 accumulation)",
                      "fp32": "f32"}[precision],
            "data": "synthetic", "config": cfg,
            "e2e": {"value": points / (ms_e2e * 1e-3), "unit": "points/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": BATCH * 4 * NPOINTS * 4 + 4 * BATCH * 8,
                    "d2h_bytes_per_step": BATCH * NPOINTS * CLASSES * 4,
                    "host_link_gbs_all_gpus": world * (BATCH * 4 * NPOINTS * 4 + BATCH * NPOINTS * CLASSES * 4) / (ms_e2e / args.steps * 1e-3) / 1e9,
                    "note": "the [B, N, 19] fp32 log-probabilities are 14.6 MB per batch and GPU; a plain pinned copy of that size runs at "
                            "~54 GB/s on one GPU of this pool's (virtualised) hosts, but all eight GPUs together saturate the host link at "
                            "~100 GB/s, which bounds this figure at N = 8 whatever the GPUs do (see e2e_labels for the evaluation loop's "
                            "real consumer); the fill and drain of the pipeline are inside the timed region (K steps, " + f"{depth} batches in flight)"},
            "e2e_labels": None if not ms_lab else {
                "value": points / (ms_lab * 1e-3), "unit": "points/s", "ms_per_step": ms_lab / args.steps,
                "h2d_bytes_per_step": BATCH * 4 * NPOINTS * 4 + 4 * BATCH * 8, "d2h_bytes_per_step": BATCH * NPOINTS,
                "what": "the same end-to-end path moving only pred.argmax(-1) to the host (uint8 [B, N]), which is all the reference's "
                        "evaluation loop uses of the output (pcdseg.py:75); the headline e2e above moves the full log-probabilities"},
            "host": {"numa": numa, "cpus": os.cpu_count()},
            "gpu_launches": per_forward * args.steps,
            "step_ms": {"min": spread[0], "median": spread[len(spread) // 2], "max": spread[-1],
                        "what": "intervals between the completions of consecutive batches inside the timed region"},
            "sequential": None if not seq else {"ms_per_step": seq, "value": world * BATCH * NPOINTS / (seq * 1e-3), "unit": "points/s",
                                                "what": "one batch at a time (depth 1), per-step CUDA events, 512 MiB written between steps: "
                                                        "the round-1 protocol"},
            "roofline": {"kernel": "fps_async_kernel (pn_fps_f32 / pn_fps_progress_f32, level 1: N=24000 -> 1024 centroids)",
                         "bound": "hbm", "achieved": fps1["achieved"], "peak": fps1["peak"], "unit": "GB/s", "frac": fps1["frac"],
                         "traffic": fps1["traffic"] if fps1["traffic"] is not None else FPS_DRAM_BYTES_PER_LAUNCH,
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture (profiles/)",
                         "peak_source": per_kernel["peak_source"], "algorithmic_bytes_per_launch": fps1["algorithmic_bytes"],
                         "launch_ms": fps1["launch_ms"], "share_of_step": fps1["launch_ms"] / (ms / args.steps),
                         "sm_time_share_of_step": (fps1.get("sms_occupied") or 0) / 148.0 * fps1["launch_ms"] / (ms / args.steps),
                         # launches of consecutive batches overlap: one sampling launch completes per step
                         "achieved_per_step": fps1["algorithmic_bytes"] / (ms / args.steps * 1e-3) / 1e9,
                         "frac_per_step": fps1["algorithmic_bytes"] / (ms / args.steps * 1e-3) / 1e9 / fps1["peak"],
                         "launch_shape": fps1.get("launch_shape"), "sms_occupied": fps1.get("sms_occupied"),
                         "fp32_pipe_frac_on_its_sms": fps1.get("fp32_pipe_frac_on_its_sms"),
                         "timing": "CUDA events around the stand-alone launch (cold L2) right after the timed regions, in the launch "
                                   "shape the timed step uses; inside the step the kernel runs beside the other batches' kernels, so "
                                   "share_of_step (latency / step) exceeds 1 and sm_time_share_of_step (x its share of the 148 SMs) is "
                                   "the comparable figure; the serialised ncu list (profiles/r02_final_launches_summary.txt) shows 56 %",
                         "note": "coordinates and running distances are register-resident, so DRAM traffic is ~0 and the figure is an "
                                 "effective bandwidth on SURVEY 8(d)'s algorithmic bytes.  With batches in flight the runner trades "
                                 "latency for SM time: 2 CTAs per cloud (16 of 148 SMs, 1.0 ms) instead of the latency-optimal 8 (64 "
                                 "SMs, 0.46 ms, frac 1.04: second fps row of roofline_all), so this fraction HALVES while the step gets "
                                 "faster; what bounds the kernel is the FP32 pipe of the SMs it occupies (fp32_pipe_frac_on_its_sms: "
                                 "12 lane operations per point and iteration, none fusable under the reference's rounding)"},
            "roofline_all": per_kernel,
            "clocks": clocks.summary(),
        }
        line.update(cpu_legs)
        if "cpu_baseline" in cpu_legs:
            line["cpu_baseline_torch"] = cpu_legs["cpu_baseline"]
    return line, (world, rank, dev)


def cpu_train_oracle(B=2, N=2048):
    """The float64 numpy oracle of one training iteration (oracle/train_oracle.py) on a bounded sample: points/s."""
    import numpy as np
    import torch

    from oracle import oracle as orc
    from oracle import train_oracle as tor
    from pointnet12_b200 import synthetic as syn
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg

    torch.manual_seed(1234)
    sd = orc.numpy_state_dict(PointNet2SemSeg(19, feature_dims=1).state_dict())
    pts = syn.kitti_batch(B, N, config=5)
    rng = np.random.default_rng(0)
    target = rng.integers(0, 19, (B, N))
    starts = [rng.integers(0, n, B) for n in (N, 1024, 256, 64)]
    keep = rng.integers(0, 2, (B * N, 128))
    t0 = time.perf_counter()
    tor.semseg_train_step(sd, pts, target, starts, keep)
    dt = time.perf_counter() - t0
    return {"value": B * N / dt, "unit": "points/s", "cores": orc.num_threads(), "kind": "port",
            "sample": f"one training iteration (forward, loss, backward) of {B} clouds x {N} points, numpy float64 oracle "
                      f"(BLAS threads) + C/OpenMP geometry, {dt:.2f} s"}


def cpu_preprocess_oracle(scan, npoints, scans):
    """CPU leg of --workload preprocess: the numpy restatement of the reference's loader path on ONE raw scan."""
    import numpy as np

    from oracle import preprocess_oracle as por
    from pointnet12_b200 import synthetic as syn

    t0 = time.perf_counter()
    k, _ = por.scan_filter(*scan, syn.SEMANTIC_KITTI_LEARNING_MAP)
    rng = np.random.default_rng(0)
    por.scan_sample(*scan, syn.SEMANTIC_KITTI_LEARNING_MAP, npoints, rng.integers(0, len(k), npoints),
                    noise=np.zeros((len(k), 4), np.float32))
    ms = (time.perf_counter() - t0) * 1e3
    return {"value": scan[0].shape[0] / (ms * 1e-3), "unit": "points/s", "cores": 1, "kind": "port",
            "sample": f"one raw scan of {scan[0].shape[0]} points through oracle/preprocess_oracle.py (numpy), {ms:.1f} ms; "
                      f"a batch of {scans} scans = {ms * scans:.0f} ms"}


def main():
    args = parse()
    if args.workload in ("train", "preprocess") and args.impl == "ours":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        if args.workload == "preprocess":
            import bench_preprocess

            bench_preprocess.main(["--steps", str(args.steps), "--warmup", str(args.warmup)],
                                  cpu_baseline=None if args.no_cpu_baseline else cpu_preprocess_oracle)
            return
        import bench_train

        bench_train.main(["--steps", str(args.steps), "--warmup", str(args.warmup)] + (["--eager"] if args.mode == "eager" else [])
                         + (["--no-cpu-baseline"] if args.no_cpu_baseline else []),
                         cpu_baseline=None if args.no_cpu_baseline else cpu_train_oracle)
        return
    if args.impl == "reference":
        run_reference(args)
        return
    line, (world, rank, dev) = run_ours(args)
    if not args.no_train and args.mode == "graph":
        # config C5 in front of the driver: the training iteration with its NCCL gradient all-reduce, and the data-parallel
        # equivalence check, on the same ranks (tools/bench_train.py)
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_train

        train = bench_train.main(["--steps", str(args.steps), "--warmup", str(max(3, args.warmup)), "--no-cpu-baseline"],
                                 init_pg=False, emit=False)
        check = bench_train.dp_check(world, rank, dev)
        if line is not None:
            line["train"] = None if train is None else {
                k: train[k] for k in ("metric", "value", "unit", "steps", "ms_per_step", "step_ms", "e2e", "allreduce_us", "allreduce_bytes",
                                      "gpu_launches", "final_loss")}
            if train is not None:
                line["train"]["config"] = train["config"]
                line["train"]["roofline"] = train["roofline"]
            line["dp_check"] = check
    if line is not None:
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
