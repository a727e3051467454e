"""Training-batch throughput of ExpertDataset on 21,000 synthetic expert schedules (N = 10 agents, 20 x 20 maps,
obstacle density 0.1, up to 31 rows per case; seeded), the size of the original project's 10-agent training set.

Measured on the device: `add` (host validation + upload + the threshold kernel, synchronised wall time) and the
threshold kernel alone (CUDA events); `batch` at B = 64 and B = 4,096 (CUDA events, warmed up, median of repeated
launches); one epoch of training steps (Adam, B = 64, K = 3) fed by `batches()` and the same number of steps fed one
fixed pre-built batch, so the difference is the builder's share of an epoch.  Measured on the host, for comparison:
the numpy oracle transformer (oracle/dataset_oracle.py) per case and one scipy.io.loadmat per sample of a written
.mat file, as the original project's train loader calls it.  Prints one JSON line with the device name and power limit
read in the same run.

    python profiles/dataset_throughput.py [--cases 21000] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import scipy.io
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import gnn_pathplanning_b200 as gp  # noqa: E402
from gnn_pathplanning_b200 import synthetic  # noqa: E402
from oracle import dataset_oracle, planner_oracle as po  # noqa: E402

N, W, DENSITY, K = 10, 20, 0.1, 3


class Cfg:
    num_agents, nGraphFilterTaps, device = N, K, torch.device("cuda")


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def event_ms(fn, reps):
    """Median over `reps` launches of fn's device time (CUDA events around each launch)."""
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def epoch_seconds(ds, steps_source, steps):
    m = gp.DecentralPlannerNet(Cfg())
    m.load_state_dict(po.init_state_dict(K, seed=1))
    m = m.cuda().train()
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)
    it = steps_source()
    for _ in range(20):                                             # warm-up (not timed)
        x, S, t = next(it)
        opt.zero_grad()
        m.addGSO(S)
        gp.planner_loss(m.forward_logits(x), t).backward()
        opt.step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n = 0
    for x, S, t in steps_source():
        opt.zero_grad()
        m.addGSO(S)
        gp.planner_loss(m.forward_logits(x), t).backward()
        opt.step()
        n += 1
        if n == steps:
            break
    torch.cuda.synchronize()
    return time.perf_counter() - t0, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", type=int, default=21000)
    ap.add_argument("--seed", type=int, default=2020)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    rng = np.random.default_rng(args.seed)
    pos, goals, maps = synthetic.random_schedules(rng, args.cases, N, W, DENSITY, max_len=31)
    res = {"device": torch.cuda.get_device_name(), "power_limit": power_limit(), "cases": args.cases,
           "agents": N, "map": W}

    gp.ExpertDataset(N).add(pos[:8], goals[:8], maps[:8])          # module load, allocator warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ds = gp.ExpertDataset(N).add(pos, goals, maps)
    torch.cuda.synchronize()
    res["samples"] = len(ds)
    res["add_s"] = time.perf_counter() - t0
    res["dataset_device_MB"] = sum(t.numel() * t.element_size() for t in
                                   (ds.pos, ds.row_case, ds.case_first_row, ds.goal, ds.map, ds.radius)) / 1e6
    lib = gp._lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    radius = torch.empty_like(ds.radius)
    res["prepare_kernel_ms"] = event_ms(lambda: gp._lib.check(lib.gpp_dataset_prepare(
        ds.pos.data_ptr(), ds.case_first_row.data_ptr(), 5.0, radius.data_ptr(), ds.num_cases, N, stream)), 5)
    assert torch.equal(radius, ds.radius)

    g = torch.Generator("cuda").manual_seed(args.seed)
    for B in (64, 4096):
        rows = torch.randperm(len(ds), device="cuda", generator=g)[:B]
        out = ds.batch(rows)
        for _ in range(10):
            ds.batch(rows, out=out)
        ms = event_ms(lambda: ds.batch(rows, out=out), 200)
        res["batch_B%d_us" % B] = ms * 1e3
        res["batch_B%d_samples_per_s" % B] = B / (ms * 1e-3)

    steps = -(-len(ds) // 64)
    fixed = ds.batch(torch.arange(64, device="cuda"))

    def fixed_source():
        return iter([fixed] * (steps + 20))
    t_build, n_build = epoch_seconds(ds, lambda: ds.batches(64, generator=g), steps)
    t_fixed, n_fixed = epoch_seconds(ds, fixed_source, steps)
    assert n_build == n_fixed == steps
    res.update(epoch_steps=steps, epoch_s_with_builder=t_build, epoch_s_fixed_batch=t_fixed,
               step_ms_with_builder=t_build / steps * 1e3, step_ms_fixed_batch=t_fixed / steps * 1e3,
               builder_share_of_epoch=(t_build - t_fixed) / t_build)

    # host, for comparison: the numpy transformer per case and scipy.io.loadmat per sample
    sample = range(20)
    t0 = time.perf_counter()
    files = [dataset_oracle.transform(maps[c], goals[c], pos[c]) for c in sample]
    res["host_oracle_transform_ms_per_case"] = (time.perf_counter() - t0) / len(sample) * 1e3
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "train_ID0_MP%d.mat" % pos[0].shape[0])
        f = files[0]
        scipy.io.savemat(p, {"map": maps[0].astype(np.float64), "goal": goals[0].astype(np.float64),
                             "inputState": pos[0].astype(np.float64), "inputTensor": f["inputTensor"],
                             "target": f["target"], "GSO": f["GSO"], "makespan": pos[0].shape[0]})
        reps = 200
        t0 = time.perf_counter()
        for _ in range(reps):
            m = scipy.io.loadmat(p)
            torch.from_numpy(m["inputTensor"][0]).float()
        res["host_loadmat_ms_per_sample"] = (time.perf_counter() - t0) / reps * 1e3
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
