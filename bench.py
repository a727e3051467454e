#!/usr/bin/env python
"""bench.py -- agent-steps/sec of the DecentralPlannerNet hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one addGSO + forward of one batch of synthetic rollout-like input at the configuration
BASELINE.json quotes the metric on (configs[1], "C2"): DCP K=3, 10 agents, 20x20 map, batch 64
inference per GPU (640 agent-steps per step per GPU, weak scaling, no collective on the data path).

How every number is timed: untimed warm-up steps (at least W and at least half a second, so that clocks, the
library's lanes and the host loop are in steady state), then exactly K back-to-back timed steps, after a barrier +
torch.cuda.synchronize() on both sides.  CUDA events on the launching stream (wall clock for the host calls) split the
K steps into up to 10 consecutive windows; a rank's figure is K times the MEDIAN per-step time of its windows (robust to
host scheduler hiccups, which a single window of a host-bound loop is not), the reported figure the MAX over ranks.  The
default K = 5000 makes the headline window about 110 ms on a B200 (22.4 us per step measured at a 1000 W power limit);
much shorter windows measure host submission jitter more than the GPU.  The legs time their own step counts derived
from K (below).  Inputs rotate through a device pool larger than L2.

--dump-outputs DIR   after the timed steps, writes the logits [10 agents, 64 episodes, 5 actions] (float32) that the
        last timed step of `value` returned to DIR/logits.npy (rank 0).  The inputs depend only on the arguments, so two
        builds run with the same arguments can be compared output for output.

value   C2 device-resident (inputs already in HBM), 6 independent episode batches in flight over the library's compute
        lanes (DecentralPlannerNet.infer_async / join); `single_stream` = the same steps one after the other on one stream.
e2e     C2 through the public host-buffer call: every step's x / S cross PCIe from pinned host memory and
        its logits come back, inside the timed region.  `value` = 6 independent episode batches in flight (`value_3_in_flight`: 3)
        (DecentralPlannerNet.infer_host_async / wait), `sync_value` = one blocking call per step.
legs    the other BASELINE.json configs, same timing rules: C1 (K=2, batch 1, float64 GSO: rollout-step
        latency), C4 (40 agents, 50x50 map, batch 256), train_C3 (K=3, 10 agents, batch 64: forward + fused
        loss + backward + Adam), train_C5_shard (20 agents, 28x28 map, 64 episodes per GPU -- C5 is 512
        episodes over 8 GPUs; with N > 1 ranks the flat-gradient NCCL all-reduce runs INSIDE the timed step).
roofline / roofline_graph_filter / roofline_graph_filter_saturated
        algorithmic flops / bytes per launch (SURVEY.md 8d) over the kernel's mean duration from CUDA events
        recorded around each kernel on the launching stream; `traffic` = DRAM bytes per launch from the committed
        ncu captures (profiles/), scaled to this launch's size.
cpu_baseline   the oracle port (oracle/planner_oracle.py: the reference's own PyTorch-CPU op sequence) on this
        box's host cores, bounded sample of the SAME workload (rank 0, N=1 only).
--impl reference   times that same CPU path as the reference arm (the reference is pure Python/PyTorch and
        /root/reference does not travel to the GPU box).
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "agent-steps/sec (DCP K=3, 10 agents, 20x20 map)"
UNIT = "agent-steps/s"
K_TAPS, N_AGENTS, MAP_W, BATCH = 3, 10, 20, 64
WORKLOAD = "DCP K=3, 10 agents, 20x20 map, batch=64 inference per GPU (BASELINE.json configs[1])"

# SURVEY.md section 8d algorithmic figures
FE_FLOPS_PER_AGENT_STEP = 2476224 + 32768          # 5 conv layers + compress MLP
# DRAM traffic per unit from the committed ncu captures (dram__bytes_read.sum + dram__bytes_write.sum):
#   profiles/r02_ncu_feature_mma_c2.csv: feature_mma_kernel per C2 launch (640 agent-steps)
#   profiles/r02_ncu_gf_small_c2.txt: gf_small_mma_kernel 0.593 MB per C2 launch
#   profiles/r02_ncu_pair_v16_summary.txt: gf_fwd_pair_kernel 664.54 MB for 65,536 episodes x 10 agents
NCU_FE_BYTES_PER_AGENT_STEP = 1.752576e6 / 640        # feature_mma_kernel: 0.93 MB of inputs + 0.63 MB of filter images + constants
NCU_GF_BYTES_PER_AGENT_STEP = 0.593408e6 / 640
NCU_PAIR_BYTES_PER_AGENT_STEP = 664.54e6 / 655360


def gf_bytes_per_agent_step(n):
    return 4 * (128 * n + n * n + 128 * n) // n


def gf_flops_per_agent_step(n, k):
    return (2 * 128 * n * n * (k - 1) + 2 * n * k * 128 * 128) // n


def config_dict(world):
    """The SAME dict in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "K": K_TAPS, "num_agents": N_AGENTS, "map_w": MAP_W, "batch_per_gpu": BATCH,
            "global_batch": BATCH * world,
            "parallelism": "episode-sharded replicas x%d, no collective on the inference data path" % world,
            "timing": "K timed steps after >= W warm-up steps and >= 0.5 s, in up to 10 windows (CUDA events), median window, "
                      "max over ranks",
            "l2_policy": "device-resident inputs rotate through a pool > 126 MB L2"}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "measured"
    except Exception:
        return 6650.0, 1400.0, "fallback"       # B200_PROFILING.md fallback figures


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while timed regions run."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.01)

    def __enter__(self):
        if self.nv is not None:
            self._stop.clear()
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        if self._thr is not None:
            self._stop.set()
            self._thr.join()
            self._thr = None

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def make_state_dict(K=K_TAPS, seed=1337):
    from oracle import planner_oracle as po      # parameter construction only (not timed, not compute)
    sd = po.init_state_dict(K, seed=seed)
    po.randomize_bn_stats(sd)
    return sd


def make_inputs(unique, seed, batch=BATCH, n=N_AGENTS, map_w=MAP_W, gso_dtype=np.float32):
    from gnn_pathplanning_b200 import synthetic
    xs, Ss = [], []
    for i in range(unique):
        x, S = synthetic.make_batch(batch, n, map_w, seed=seed + i, gso_dtype=gso_dtype)
        xs.append(torch.from_numpy(x))
        Ss.append(torch.from_numpy(S))
    return xs, Ss


def cpu_forward_factory(sd, xs, Ss):
    from oracle import planner_oracle as po

    def step(i):
        with torch.no_grad():
            return po.planner_forward(sd, Ss[i % len(Ss)], xs[i % len(xs)])
    return step


def cpu_infer_arm(n, k, batch, map_w, steps):
    """CPU port (oracle) on one of the other BASELINE configs: agent-steps/s of `steps` inference steps after one warm-up."""
    from oracle import planner_oracle as po
    sd = make_state_dict(k, seed=1000 + n)
    xs, Ss = make_inputs(1, 9200 + n, batch, n, map_w)
    with torch.no_grad():
        po.planner_forward(sd, Ss[0], xs[0])
        t0 = time.perf_counter()
        for _ in range(steps):
            po.planner_forward(sd, Ss[0], xs[0])
    return steps * batch * n / (time.perf_counter() - t0)


def cpu_train_arm(sd, n, batch, map_w, steps):
    """CPU port (oracle) train step -- forward + loss + backward, no optimizer -- agent-steps/s."""
    from oracle import planner_oracle as po
    from gnn_pathplanning_b200 import synthetic
    x, S = synthetic.make_batch(batch, n, map_w, seed=9000 + n)
    tg = torch.from_numpy(synthetic.random_targets(batch, n, seed=9100 + n))
    leaf = {k2: (v.clone().requires_grad_(True) if (v.is_floating_point() and "running" not in k2) else v)
            for k2, v in sd.items()}
    bn = {k2: v.clone() for k2, v in sd.items() if "running" in k2 or "tracked" in k2}
    t0 = time.perf_counter()
    for _ in range(steps):
        po.planner_loss(po.planner_forward(leaf, torch.from_numpy(S), torch.from_numpy(x), True, bn), tg).backward()
    return steps * batch * n / (time.perf_counter() - t0)


def usable_cpus():
    """CPUs this process may really use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def pick_cpu_threads(step, budget_s=6.0):
    """The reference's PyTorch-CPU path is N sequential tiny convolutions; on a many-core host it gets SLOWER
    with more intra-op threads (measured: 19 s/step at 128 threads vs ~20 ms at 8).  The CPU arm is given its
    best case: the thread count with the highest measured throughput among {all usable, 64, 32, ..., 1}."""
    cap = usable_cpus()
    cands = sorted({c for c in (cap, 64, 32, 16, 8, 4, 2, 1) if c <= cap}, reverse=True)
    best, best_t = 1, float("inf")
    t_start = time.perf_counter()
    for c in reversed(cands):                       # small counts first: they are cheap to probe
        torch.set_num_threads(c)
        step(0)
        t0 = time.perf_counter()
        step(1)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
        if time.perf_counter() - t_start > budget_s or dt > 4 * best_t:
            break
    torch.set_num_threads(best)
    return best, cap


def time_cpu(step, budget_s, min_steps=5, warmup=3):
    for i in range(warmup):
        step(i)
    t0 = time.perf_counter()
    n = 0
    while True:
        step(n)
        n += 1
        el = time.perf_counter() - t0
        if n >= min_steps and el >= budget_s:
            break
    return n, el


# ----------------------------------------------------------------------------------------------------------
# timing helper: K steps in up to WINDOWS consecutive windows
# ----------------------------------------------------------------------------------------------------------
class Timer:
    WINDOWS = 10
    SETTLE_S = 0.5

    def __init__(self, dist, dev):
        self.dist, self.dev = dist, dev

    def _bounds(self, K):
        n = min(K, self.WINDOWS)
        return [round(j * K / n) for j in range(n + 1)]

    def _warm_up(self, step, warmup, drain, period):
        """Untimed steps 0 .. n-1: `warmup` of them, then more in rounds of `warmup` until every rank has spent at least
        SETTLE_S seconds, then up to n = warmup modulo `period` so that the timed steps n, n+1, ... see the same inputs
        however long the warm-up took.  Whether to run another round is decided over all ranks, so every rank runs the
        same n steps: a step may contain a collective (the training legs' gradient all-reduce).  Returns n."""
        self.barrier()
        t0, n, rnd = time.perf_counter(), 0, max(1, warmup)
        while True:
            for _ in range(rnd):
                step(n)
                n += 1
            (more,) = self.max_over_ranks(float(time.perf_counter() - t0 < self.SETTLE_S))
            if not more:
                break
        while (n - warmup) % period:
            step(n)
            n += 1
        drain()
        self.barrier()
        return n

    @staticmethod
    def _median_ms(K, bounds, ms):
        """K x the median per-step ms of the windows; ms[w] is window w's duration."""
        return K * float(np.median([ms[w] / (bounds[w + 1] - bounds[w]) for w in range(len(ms))]))

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def device_window(self, step, K, warmup, drain=None, period=1):
        """step(i) enqueues one step on the current stream (or on the library's lanes, whose steps the current stream
        joins as it goes: then drain() makes it wait for everything outstanding before the last window's closing event).
        After the warm-up (_warm_up) the next K steps are timed.  Returns K x the median per-step ms of the windows on
        this rank."""
        drain = drain or (lambda: None)
        n = self._warm_up(step, warmup, drain, period)
        bounds = self._bounds(K)
        evs = [torch.cuda.Event(enable_timing=True) for _ in bounds]
        evs[0].record()
        for w in range(len(bounds) - 1):
            for i in range(bounds[w], bounds[w + 1]):
                step(n + i)
            if w == len(bounds) - 2:
                drain()
            evs[w + 1].record()
        torch.cuda.synchronize()
        self.barrier()
        return self._median_ms(K, bounds, [evs[w].elapsed_time(evs[w + 1]) for w in range(len(bounds) - 1)])

    def host_window(self, step, K, warmup, drain):
        """step(i) is a host call (may leave work in flight; drain() completes it before the last window closes).
        Wall-clock windows, warm-up and result as in device_window."""
        n = self._warm_up(step, warmup, drain, 1)
        bounds = self._bounds(K)
        ts = [time.perf_counter()]
        for w in range(len(bounds) - 1):
            for i in range(bounds[w], bounds[w + 1]):
                step(n + i)
            if w == len(bounds) - 2:
                drain()
                torch.cuda.synchronize()
            ts.append(time.perf_counter())
        self.barrier()
        return self._median_ms(K, bounds, [(ts[w + 1] - ts[w]) * 1e3 for w in range(len(bounds) - 1)])

    def max_over_ranks(self, *vals):
        if self.dist is None:
            return vals
        t = torch.tensor(list(vals), device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return tuple(float(v) for v in t)


def device_pool(xs_h, Ss_h, dev, pool_mb, rank):
    bytes_per_batch = xs_h[0].numel() * xs_h[0].element_size() + Ss_h[0].numel() * Ss_h[0].element_size()
    pool_n = max(len(xs_h), int(pool_mb * 1e6 / bytes_per_batch) + 1)
    g = torch.Generator().manual_seed(rank)
    B = xs_h[0].shape[0]
    pool_x = torch.empty((pool_n,) + tuple(xs_h[0].shape), device=dev, dtype=xs_h[0].dtype)
    pool_S = torch.empty((pool_n,) + tuple(Ss_h[0].shape), device=dev, dtype=Ss_h[0].dtype)
    for i in range(pool_n):
        perm = torch.randperm(B, generator=g)
        pool_x[i].copy_(xs_h[i % len(xs_h)][perm])
        pool_S[i].copy_(Ss_h[i % len(Ss_h)][perm])
    return pool_x, pool_S, pool_n, bytes_per_batch


def build_model(gp, sd, n, k, dev, gf_mode="auto", fe_mode="auto"):
    class Cfg:
        num_agents, nGraphFilterTaps, device = n, k, dev
    model = gp.DecentralPlannerNet(Cfg())
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    model.set_graph_filter_mode(gf_mode)
    model.set_feature_mode(fe_mode)
    return model


def saturated_filter_roofline(gp, dev, batch, hbm_peak, peak_src):
    """The fused graph filter alone (node-major in/out, + ReLU) on a batch large enough to fill the machine: the
    headline configuration moves only 0.68 MB per launch and is launch-latency bound, so this is where the kernel's
    bandwidth fraction is visible.  Inputs (batch x 10 x 128 floats and the GSOs) exceed L2 many times over; CUDA
    events around back-to-back calls of the public op; the tap re-layout launches (|w| maximum + fp16 split images,
    ~8 us) that precede every standalone call are inside the timed region."""
    g = torch.Generator().manual_seed(0)
    w = ((torch.rand(128, 1, K_TAPS, 128, generator=g) - 0.5) * 0.2).to(dev)
    b = (torch.rand(128, 1, generator=g) - 0.5).to(dev)
    x = torch.randn(batch, N_AGENTS, 128, device=dev)
    # rollout-like GSOs: normalised adjacency of random agent positions on the 20x20 map, radius 6
    pos = torch.randint(0, MAP_W, (batch, N_AGENTS, 2), device=dev).float()
    A = ((pos[:, :, None, :] - pos[:, None, :, :]).norm(dim=-1) < 6.0).float() * (1.0 - torch.eye(N_AGENTS, device=dev))
    dinv = A.sum(-1).clamp(min=1.0).rsqrt() * (A.sum(-1) > 0)
    S = (dinv[:, :, None] * A * dinv[:, None, :]).contiguous()
    for _ in range(3):
        gp.graph_filter(x, S, w, b, True, gp.NODE_MAJOR, gp.NODE_MAJOR)
    torch.cuda.synchronize()
    iters = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        gp.graph_filter(x, S, w, b, True, gp.NODE_MAJOR, gp.NODE_MAJOR)
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) * 1e-3 / iters
    nbytes = gf_bytes_per_agent_step(N_AGENTS) * batch * N_AGENTS
    gbs = nbytes / sec / 1e9
    return {"kernel": "gf_fwd_pair_kernel (tcgen05 cta_group::2, fp16 2-way split, resident taps, TMA tensor stores) via "
                      "gpp_graph_filter_forward",
            "bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
            "traffic": NCU_PAIR_BYTES_PER_AGENT_STEP * batch * N_AGENTS,
            "traffic_source": "profiles/r02_ncu_pair_v16_summary.txt (dram read + write at 65,536 episodes, scaled by size)",
            "peak_source": peak_src, "mean_launch_us": sec * 1e6,
            "workload": "K=3, 10 agents, %d episodes (%.0f MB of node signals + GSOs in, %.0f MB out)"
                        % (batch, (batch * N_AGENTS * (128 + N_AGENTS) * 4) / 1e6, batch * N_AGENTS * 128 * 4 / 1e6),
            "agent_steps_per_s": batch * N_AGENTS / sec, "algorithmic_bytes_per_launch": nbytes}


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU implementation of the path = its PyTorch-CPU op sequence, restated in
    oracle/planner_oracle.py (the Python reference cannot travel to the GPU box).  All host threads, same
    config/metric/unit as the CUDA arm."""
    if rank != 0:
        return
    sd = make_state_dict()
    xs, Ss = make_inputs(4, 1337)
    step = cpu_forward_factory(sd, xs, Ss)
    threads, cap = pick_cpu_threads(step)
    # bounded sample: if K full-batch steps would not end within ~4 minutes on this host, each step processes the
    # first `sub` episodes of the batch instead (same per-episode work)
    t0 = time.perf_counter()
    step(0)
    t_step = time.perf_counter() - t0
    sub = BATCH
    if t_step * (args.steps + args.warmup) > 240.0:
        sub = max(1, int(BATCH * 240.0 / (t_step * (args.steps + args.warmup))))
        xs, Ss = [x[:sub].contiguous() for x in xs], [s[:sub].contiguous() for s in Ss]
        step = cpu_forward_factory(sd, xs, Ss)
    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
    el = time.perf_counter() - t0
    val = sub * N_AGENTS * args.steps / el
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config_dict(args.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "usable_cpus": cap,
                         "sample": "%d steps of %d episodes x 10 agents of the same workload on rank 0; thread count "
                                   "auto-picked for best CPU throughput" % (args.steps, sub)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------
# legs
# ----------------------------------------------------------------------------------------------------------
def leg_inference(gp, timer, dev, rank, world, n, k, batch, map_w, gso_dtype, K, warmup, pool_mb, label, global_batch=None,
                  cpu=False):
    """`global_batch`: strong scaling -- the batch is the global one split evenly over the ranks (remainder dropped) and the
    throughput is that of the whole job; otherwise `batch` episodes per GPU (weak)."""
    if global_batch is not None:
        batch = max(1, global_batch // world)
    sd = make_state_dict(k, seed=1000 + n)
    model = build_model(gp, sd, n, k, dev)
    xs_h, Ss_h = make_inputs(4, 4242 + 100 * rank + n, batch, n, map_w, gso_dtype)
    pool_x, pool_S, pool_n, _ = device_pool(xs_h, Ss_h, dev, pool_mb, rank)

    def step(i):
        model.addGSO(pool_S[i % pool_n])
        return model(pool_x[i % pool_n])
    with torch.no_grad():
        ms = timer.device_window(step, K, warmup)
    (ms,) = timer.max_over_ranks(ms)
    out = {"workload": label, "ms_per_step": ms / K, "us_per_step": 1e3 * ms / K,
           "agent_steps_per_s": world * batch * n * K / (ms * 1e-3), "steps": K, "gso_dtype": str(np.dtype(gso_dtype))}
    if global_batch is not None:
        out["scaling"] = "strong"
        out["global_batch"] = batch * world
        out["batch_per_gpu"] = batch
    if cpu:
        # SURVEY 8d: the reference pins a rollout to one core (main.py:25-27) -- 1-thread and all-thread latency of the port
        step_cpu = cpu_forward_factory(sd, xs_h, Ss_h)
        for nthreads, key in ((1, "cpu_us_per_step_1_thread"), (usable_cpus(), "cpu_us_per_step_all_threads")):
            torch.set_num_threads(nthreads)
            n_cpu, el = time_cpu(step_cpu, 1.0)
            out[key] = 1e6 * el / n_cpu
        out["cpu_threads_all"] = usable_cpus()
    if batch == 1 and global_batch is None:
        # the rollout step as the reference's agent runs it: host tensors in, logits out, one blocking call
        hx, hS = [t.pin_memory() for t in xs_h], [t.pin_memory() for t in Ss_h]
        hout = torch.empty(n, batch, 5).pin_memory()
        hms = timer.host_window(lambda i: model.infer_host(hx[i % 4], hS[i % 4], hout), K, warmup, lambda: None)
        (hms,) = timer.max_over_ranks(hms)
        out["host_call_us_per_step"] = 1e3 * hms / K
        out["host_call_api"] = "DecentralPlannerNet.infer_host (pinned host x / float64 S in, logits out, blocking)"
    del model, pool_x, pool_S
    torch.cuda.empty_cache()
    return out


def leg_rollout(gp, timer, dev, rank, world, n, k, episodes, map_w, K, warmup, label, cpu):
    """Rows f1/f2: one lock-step rollout step of `episodes` device-resident episodes = gpp_rollout_build_inputs (FOV tensors
    + float64 GSOs from the positions) -> planner forward -> gpp_rollout_move; nothing crosses PCIe.  The CPU figure next to
    it is the oracle's restatement of the reference simulator's per-step work around the model (getCurrentState + getGSO +
    move, one episode at a time, oracle/sim_oracle.py)."""
    from gnn_pathplanning_b200 import synthetic
    rng = np.random.default_rng(77 + rank)
    cases = [synthetic.random_episode(rng, n, map_w, 0.1) for _ in range(min(episodes, 64))]
    rep = (episodes + len(cases) - 1) // len(cases)
    maps = np.stack([c[0] for c in cases] * rep)[:episodes]
    starts = np.stack([c[1] for c in cases] * rep)[:episodes]
    goals = np.stack([c[2] for c in cases] * rep)[:episodes]
    sd = make_state_dict(k, seed=1000 + n)
    sd["actionsMLP.0.weight"] = sd["actionsMLP.0.weight"] * 40.0
    model = build_model(gp, sd, n, k, dev)
    ro = gp.BatchedRollout(n, 6.0, dev).setup(starts, goals, maps, 1 << 30)

    def step(i):
        x, S = ro.build_inputs(i + 1)
        model.addGSO(S)
        ro.move(model.forward_logits(x), i + 2)
    with torch.no_grad():
        from gnn_pathplanning_b200 import _lib
        step(0)                                  # the first forward also runs the weight-preparation kernels
        l0 = _lib.launch_count()
        step(1)
        launches = _lib.launch_count() - l0
        ms = timer.device_window(step, K, warmup)
    (ms,) = timer.max_over_ranks(ms)
    out = {"workload": label, "us_per_step": 1e3 * ms / K, "episode_steps_per_s": world * episodes * K / (ms * 1e-3),
           "agent_steps_per_s": world * episodes * n * K / (ms * 1e-3), "steps": K, "launches_per_step": int(launches),
           "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    if cpu:
        from oracle import sim_oracle
        sim = sim_oracle.SimOracle(n, 6.0).setup(starts[0], goals[0], maps[0], 1 << 30)
        lg = np.random.default_rng(5).standard_normal((200, n, 5)).astype(np.float32)
        sim.inputs(0)
        t0, cnt = time.perf_counter(), 0
        while time.perf_counter() - t0 < 2.0:
            sim.inputs(cnt + 1)
            sim.move(lg[cnt % 200], cnt + 2)
            cnt += 1
        out["cpu_sim_us_per_episode_step"] = 1e6 * (time.perf_counter() - t0) / cnt
        out["cpu_sim_note"] = "oracle/sim_oracle.py, one episode, 1 thread, simulator work only (no model), %d steps" % cnt
    del model, ro
    torch.cuda.empty_cache()
    return out


def leg_training(gp, timer, dist, dev, rank, world, n, batch, map_w, K, warmup, label):
    """forward (train-mode, per-agent BatchNorm) + fused cross-entropy + backward + [flat gradient all-reduce] + Adam."""
    from gnn_pathplanning_b200 import sharding, synthetic, _lib
    sd = make_state_dict(K_TAPS, seed=77)

    class Cfg:
        num_agents, nGraphFilterTaps, device = n, K_TAPS, dev
    model = gp.DecentralPlannerNet(Cfg())
    model.load_state_dict(sd)
    model = model.to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-5)      # agents/decentralplannerlocal.py:59
    bucket = sharding.GradientBucket(model)
    unique = 8
    xs, Ss, ts = [], [], []
    for i in range(unique):
        x, S = synthetic.make_batch(batch, n, map_w, seed=9000 + 50 * rank + i)
        xs.append(torch.from_numpy(x).to(dev))
        Ss.append(torch.from_numpy(S).to(dev))
        ts.append(torch.from_numpy(synthetic.random_targets(batch, n, seed=9100 + 50 * rank + i)).to(dev))
    gbatch = batch * world

    def step(i):
        j = i % unique
        return sharding.train_step(model, opt, bucket, xs[j], Ss[j], ts[j], gbatch)
    _lib.reset_launch_count()
    step(0)
    torch.cuda.synchronize()
    launches = _lib.launch_count()
    ms = timer.device_window(step, K, warmup)
    (ms,) = timer.max_over_ranks(ms)
    out = {"workload": label, "ms_per_step": ms / K, "agent_steps_per_s": world * batch * n * K / (ms * 1e-3), "steps": K,
           "library_launches_per_step": int(launches),
           "step": "train-mode forward + fused loss (gpp_planner_ce_loss) + backward + %sAdam"
                   % ("one flat 826 KB gradient all-reduce (NCCL, inside the timed step) + " if world > 1 else "")}
    if world > 1:
        # the collective alone, same buffer, on the same stream (it runs after backward(), not overlapped with it)
        for _ in range(5):
            dist.all_reduce(bucket.flat)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(50):
            dist.all_reduce(bucket.flat)
        e1.record()
        torch.cuda.synchronize()
        (ar,) = timer.max_over_ranks(e0.elapsed_time(e1) / 50)
        out["allreduce_us"] = 1e3 * ar
        out["allreduce_bytes"] = int(bucket.flat.numel() * 4)
        out["allreduce_overlapped"] = False
        out["allreduce_share_of_step"] = ar / (ms / K)
    del model, opt, bucket
    torch.cuda.empty_cache()
    return out


def sharded_parity(gp, dist, dev, rank, world):
    """Before timing, with N > 1 ranks: (1) episode-sharded inference == the unsharded forward of the same global
    batch; (2) the weighted flat all-reduce == sum_r (b_r / B) g_r of the per-rank gradients."""
    from gnn_pathplanning_b200 import sharding, synthetic
    n, per = 10, 6
    Bg = per * world + 1                               # ragged on purpose
    sd = make_state_dict(K_TAPS, seed=5)
    x, S = synthetic.make_batch(Bg, n, MAP_W, seed=321)              # same on every rank
    tgt = synthetic.random_targets(Bg, n, seed=322)
    xt, St, tt = torch.from_numpy(x).to(dev), torch.from_numpy(S).to(dev), torch.from_numpy(tgt).to(dev)
    model = build_model(gp, sd, n, K_TAPS, dev)
    lo, hi = sharding.shard_range(Bg, rank, world)
    with torch.no_grad():
        model.addGSO(St)
        full = torch.stack(model(xt))
        model.addGSO(St[lo:hi])
        local = torch.stack(model(xt[lo:hi]))
    gathered = sharding.gather_logits(local, Bg)
    e_inf = float((gathered - full).abs().max() / full.abs().max())
    model.train()
    bucket = sharding.GradientBucket(model)
    bucket.zero()
    model.addGSO(St[lo:hi])
    gp.planner_loss(model.forward_logits(xt[lo:hi]), tt[lo:hi]).backward()
    mine = bucket.flat.clone()
    parts = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(parts, mine)
    want = sum(p.double() * ((sharding.shard_range(Bg, r, world)[1] - sharding.shard_range(Bg, r, world)[0]) / Bg)
               for r, p in enumerate(parts))
    bucket.all_reduce(hi - lo, Bg)
    e_grad = float((bucket.flat.double() - want).abs().max() / want.abs().max())
    t = torch.tensor([e_inf, e_grad], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    assert float(t[0]) <= 1e-5 and float(t[1]) <= 1e-5, "sharded parity failed: %s" % t.tolist()
    return {"inference_logits_vs_unsharded": float(t[0]), "allreduced_gradient_vs_weighted_sum": float(t[1]),
            "global_batch": Bg, "ranks": world}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--pool-mb", type=float, default=160.0, help="device input pool size (> L2)")
    ap.add_argument("--gf-mode", default="auto", choices=["auto", "cuda", "tc", "pair"])
    ap.add_argument("--fe-mode", default="auto", choices=["auto", "cuda", "tc"])
    ap.add_argument("--sat-batch", type=int, default=131072,
                    help="episodes in the saturated graph-filter roofline measurement (0 = skip)")
    ap.add_argument("--no-legs", action="store_true", help="headline configuration only")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's logits to DIR/logits.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        args.steps = args.steps if args.steps is not None else 200
        args.warmup = args.warmup if args.warmup is not None else 3
        run_reference(args, rank, world)
        return
    args.steps = args.steps if args.steps is not None else 5000
    args.warmup = max(3, args.warmup if args.warmup is not None else 20)
    K, W = args.steps, args.warmup

    import gnn_pathplanning_b200 as gp
    from gnn_pathplanning_b200 import _lib
    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    timer = Timer(dist, dev)
    parity = sharded_parity(gp, dist, dev, rank, world) if world > 1 else None

    sd = make_state_dict()
    model = build_model(gp, sd, N_AGENTS, K_TAPS, dev, args.gf_mode, args.fe_mode)
    unique = 8
    xs_h, Ss_h = make_inputs(unique, 1337 + 1000 * rank)
    pool_x, pool_S, pool_n, bytes_per_batch = device_pool(xs_h, Ss_h, dev, args.pool_mb, rank)

    def dev_step(i):
        model.addGSO(pool_S[i % pool_n])
        return model(pool_x[i % pool_n])

    sampler = ClockSampler(local_rank)
    with torch.no_grad(), sampler:
        # ---- value: device-resident ------------------------------------------------------
        _lib.reset_launch_count()
        for i in range(K):
            dev_step(i)
        torch.cuda.synchronize()
        launches_per_window = _lib.launch_count()      # library kernels in one K-step window
        single_ms = timer.device_window(dev_step, K, W)      # one stream, one batch after the other
        # the same steps as a driver of independent episode batches issues them: DEV_DEPTH batches in flight over the
        # library's compute lanes (DecentralPlannerNet.infer_async / join), device tensors in, device logits out; the
        # closing event of a window waits for every outstanding step
        DEV_DEPTH = 6
        dev_outs = [torch.empty(N_AGENTS, BATCH, 5, device=dev) for _ in range(DEV_DEPTH)]
        dev_inflight, dev_last = [], [0]

        def dev_async_step(i):
            tk, _ = model.infer_async(pool_x[i % pool_n], pool_S[i % pool_n], dev_outs[i % DEV_DEPTH])
            dev_last[0] = i % DEV_DEPTH
            dev_inflight.append(tk)
            if len(dev_inflight) >= DEV_DEPTH:
                model.join(dev_inflight.pop(0))

        def dev_drain():
            while dev_inflight:
                model.join(dev_inflight.pop(0))
        ms = timer.device_window(dev_async_step, K, W, dev_drain, period=pool_n)
        if args.dump_outputs and rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "logits.npy"), dev_outs[dev_last[0]].cpu().numpy())

        # ---- per-kernel durations (events recorded around each kernel; PDL is off in this pass) -------
        nat = model._native_for(dev)
        prof_steps = 1000
        _lib.check(nat.lib.gpp_planner_set_profiling(nat.handle, 1))
        for i in range(prof_steps):
            dev_step(i)
        fe_ms, gf_ms, nst = C.c_double(), C.c_double(), C.c_int()
        _lib.check(nat.lib.gpp_planner_get_profile(nat.handle, C.byref(fe_ms), C.byref(gf_ms), C.byref(nst)))
        _lib.check(nat.lib.gpp_planner_set_profiling(nat.handle, 0))
        timer.barrier()

        # ---- e2e: host buffers through the public host calls -------------------------------------------
        hx = [t.pin_memory() for t in xs_h]
        hS = [t.pin_memory() for t in Ss_h]
        hout = torch.empty(N_AGENTS, BATCH, 5).pin_memory()
        # (a) one blocking host call per step
        sync_ms = timer.host_window(lambda i: model.infer_host(hx[i % unique], hS[i % unique], hout), K, W,
                                    lambda: None)
        # (b) pipelined over independent episode batches: step i is enqueued before step i - (DEPTH - 1) is waited for, as
        # a rollout driver advancing DEPTH groups of episodes in turn would do; every step still reads its x / S from
        # pinned host memory and writes its logits back to it.  The library rotates the tickets over 4 compute lanes.
        def pipelined(depth):
            houts = [torch.empty(N_AGENTS, BATCH, 5).pin_memory() for _ in range(depth)]
            inflight, sink = [], [0.0]

            def async_step(i):
                inflight.append((model.infer_host_async(hx[i % unique], hS[i % unique], houts[i % depth]), i % depth))
                if len(inflight) >= depth:
                    tk, slot = inflight.pop(0)
                    model.wait(tk)
                    sink[0] += float(houts[slot][0, 0, 0])       # the step's result is read on the host

            def drain():
                while inflight:
                    tk, slot = inflight.pop(0)
                    model.wait(tk)
                    sink[0] += float(houts[slot][0, 0, 0])
            return timer.host_window(async_step, K, W, drain)
        DEPTH = 6
        e2e_ms = pipelined(DEPTH)
        e2e3_ms = pipelined(3)
    ms, e2e_ms, sync_ms, e2e3_ms, single_ms = timer.max_over_ranks(ms, e2e_ms, sync_ms, e2e3_ms, single_ms)
    clocks = sampler.summary()

    agent_steps = BATCH * N_AGENTS
    value = world * agent_steps * K / (ms * 1e-3)

    legs = {}
    if not args.no_legs:
        with torch.no_grad():
            legs["C1_latency"] = leg_inference(gp, timer, dev, rank, world, 10, 2, 1, 20, np.float64, K, W, 8.0,
                                               "DCP K=2, 10 agents, 20x20 map, batch=1 (configs[0]): rollout-step latency, float64 GSO",
                                               cpu=(rank == 0 and world == 1))
            legs["C4"] = leg_inference(gp, timer, dev, rank, world, 40, 3, 256, 50, np.float32, max(5, K // 4), W, args.pool_mb,
                                       "DCP K=3, 40 agents, 50x50 map, batch=256 inference per GPU (configs[3])")
            if world > 1:
                # SURVEY 8d asks for both scalings: the same global batch split over the ranks (the headline line is weak)
                legs["C2_strong"] = leg_inference(gp, timer, dev, rank, world, 10, 3, 0, 20, np.float32, K, W, args.pool_mb,
                                                  "configs[1] with its GLOBAL batch of 64 episodes split over %d GPUs" % world,
                                                  global_batch=64)
                legs["C4_strong"] = leg_inference(gp, timer, dev, rank, world, 40, 3, 0, 50, np.float32, max(5, K // 4), W,
                                                  args.pool_mb, "configs[3] with its GLOBAL batch of 256 episodes split over %d "
                                                  "GPUs" % world, global_batch=256)
            legs["rollout_C2"] = leg_rollout(gp, timer, dev, rank, world, 10, 3, 256, 20, max(5, K // 4), W,
                                             "256 device-resident episodes per GPU in lock-step (10 agents, 20x20 map, K=3): "
                                             "inputs builder + planner forward + move per step", rank == 0 and world == 1)
        tk = max(5, K // 10)
        if world == 1:
            legs["train_C3"] = leg_training(gp, timer, dist, dev, rank, world, 10, 64, 20, tk, 3,
                                            "DCP-OE K=3 training, 10 agents, 20x20 map, batch=64 (configs[2])")
        legs["train_C5_shard"] = leg_training(gp, timer, dist, dev, rank, world, 20, 64, 28, tk, 3,
                                              "DCP-OE K=3 training, 20 agents, 28x28 map, 64 episodes per GPU x %d GPUs "
                                              "(configs[4] = 512 episodes over 8)" % world)

    if rank == 0:
        hbm_peak, tf_peak, peak_src = load_peaks()
        n = max(1, nst.value)
        fe_s, gf_s = fe_ms.value * 1e-3 / n, gf_ms.value * 1e-3 / n
        fe_tflops = FE_FLOPS_PER_AGENT_STEP * agent_steps / fe_s / 1e12
        gf_gbs = gf_bytes_per_agent_step(N_AGENTS) * agent_steps / gf_s / 1e9
        sm_mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
        fp32_peak = 148 * 128 * 2 * float(sm_mhz) * 1e6 / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(world),
            "value_api": "DecentralPlannerNet.infer_async / join -> gpp_planner_forward_async: device tensors in, device logits "
                         "out, %d independent episode batches in flight over the library's 4 compute lanes" % DEV_DEPTH,
            "single_stream": {"value": world * agent_steps * K / (single_ms * 1e-3), "ms_per_step": single_ms / K,
                              "api": "model.addGSO(S); model(x) on one stream, one batch after the other (the latency "
                                     "of a step; kernels chained by programmatic dependent launch)"},
            "e2e": {"value": world * agent_steps * K / (e2e_ms * 1e-3), "unit": UNIT, "steps": K,
                    "h2d_bytes_per_step": bytes_per_batch, "d2h_bytes_per_step": N_AGENTS * BATCH * 5 * 4,
                    "api": "DecentralPlannerNet.infer_host_async/wait -> gpp_planner_forward_host_async (pinned host "
                           "buffers; inputs staged by the copy engine on a copy stream, forward on one of four compute "
                           "lanes so one batch's CNN runs next to other batches' kernels on the SMs a 640-agent launch leaves "
                           "idle, logits written straight to host), %d independent episode batches in flight" % DEPTH,
                    "batches_in_flight": DEPTH,
                    "value_3_in_flight": world * agent_steps * K / (e2e3_ms * 1e-3),
                    "sync_value": world * agent_steps * K / (sync_ms * 1e-3),
                    "sync_api": "DecentralPlannerNet.infer_host -> gpp_planner_forward_host, one blocking call per step"},
            "gpu_launches": int(launches_per_window), "gpu_launches_per_step": int(launches_per_window) / K,
            "clocks": clocks,
            "roofline": {"kernel": "feature_mma_kernel (per-agent CNN + compress MLP on tcgen05: fp16 2-way split operands, "
                                   "3 products per term, fp32 accumulation in TMEM -- the dominant kernel of the step by time)",
                         "bound": "tensor", "pipe": "tcgen05.mma kind::f16 (SASS UTCHMMA), M=128 tiles, 8 agents per CTA",
                         "achieved": fe_tflops, "peak": tf_peak, "unit": "TFLOP/s", "frac": fe_tflops / tf_peak,
                         "traffic": NCU_FE_BYTES_PER_AGENT_STEP * agent_steps,
                         "traffic_source": "profiles/r02_ncu_feature_mma_c2.csv (dram read + write per launch)",
                         "peak_source": peak_src + " bf16 dense (sustained)",
                         "mean_launch_us": fe_s * 1e6,
                         "algorithmic_flops_per_launch": FE_FLOPS_PER_AGENT_STEP * agent_steps,
                         "note": "640 agents = 80 tiles of 8 on 80 of 148 SMs, one tile per CTA: the launch is latency-bound "
                                 "(12 serialized MMA / epilogue phases per tile); the issued tensor work is 3x the algorithmic "
                                 "flops (split products) on M tiles that are 25-60 % padding"},
            "roofline_graph_filter": {"kernel": "gf_small_mma_kernel (K-tap filter + ReLU + action MLP on tcgen05, clusters "
                                                "of 2 CTAs per 6 episodes; the benchmark size is launch-latency bound: 0.68 MB "
                                                "per launch)", "bound": "hbm",
                                      "achieved": gf_gbs, "peak": hbm_peak, "unit": "GB/s",
                                      "frac": gf_gbs / hbm_peak, "traffic": NCU_GF_BYTES_PER_AGENT_STEP * agent_steps,
                                      "traffic_source": "profiles/r02_ncu_gf_small_c2.txt",
                                      "peak_source": peak_src, "mean_launch_us": gf_s * 1e6,
                                      "algorithmic_bytes_per_launch": gf_bytes_per_agent_step(N_AGENTS) * agent_steps,
                                      "algorithmic_flops_per_launch": gf_flops_per_agent_step(N_AGENTS, K_TAPS) * agent_steps},
        }
        if legs:
            line["legs"] = legs
        if parity is not None:
            line["sharded_parity"] = parity
        if args.sat_batch > 0:
            line["roofline_graph_filter_saturated"] = saturated_filter_roofline(gp, dev, args.sat_batch, hbm_peak, peak_src)
        if world == 1:
            step = cpu_forward_factory(sd, xs_h, Ss_h)
            threads, cap = pick_cpu_threads(step, budget_s=min(6.0, max(0.5, args.cpu_seconds)))
            n_cpu, el = time_cpu(step, args.cpu_seconds)
            line["cpu_baseline"] = {"value": agent_steps * n_cpu / el, "unit": UNIT,
                                    "cores": threads, "kind": "port", "usable_cpus": cap,
                                    "sample": "%d full steps (batch 64 x 10 agents) of the same workload, %.1f s"
                                              % (n_cpu, el)}
            # parity spot-check of the timed configuration (not timed)
            ref = torch.stack(step(0)).numpy()
            model.addGSO(Ss_h[0].to(dev))
            with torch.no_grad():
                got = torch.stack(model(xs_h[0].to(dev))).cpu().numpy()
            line["parity_max_rel"] = float(np.abs(got - ref).max() / np.abs(ref).max())
            # CPU arms of the other legs (SURVEY 8d: the port timed on every configuration), bounded samples, the thread
            # count chosen above; a failure here must not cost the line
            try:
                if legs and "train_C3" in legs:
                    legs["train_C3"]["cpu_baseline_agent_steps_per_s"] = cpu_train_arm(sd, 10, 64, 20, 3)
                if legs and "C4" in legs:
                    legs["C4"]["cpu_baseline_agent_steps_per_s"] = cpu_infer_arm(40, 3, 256, 50, 2)
                if legs and "train_C5_shard" in legs:
                    legs["train_C5_shard"]["cpu_baseline_agent_steps_per_s"] = cpu_train_arm(sd, 20, 64, 28, 2)
                if legs:
                    line["legs_cpu_arm"] = {"kind": "port", "cores": threads,
                                            "sample": "3 / 2 / 2 steps of train_C3 / C4 / train_C5_shard"}
            except Exception as e:       # noqa: BLE001
                line["cpu_arms_error"] = repr(e)[:200]
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
