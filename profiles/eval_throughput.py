"""Test-set evaluation throughput: BatchedRollout.setup_cases + evaluate over 4,500 synthetic cases (N = 10 agents,
20 x 20 maps, obstacle density 0.1, K = 3 filter taps, the CUDA planner with an amplified action head so that agents
move) in one batch on the device, run twice; the per-case records of the two runs must be identical.  Prints one JSON
line: cases/s, lock-step steps and us per step of each run, the device name and power limit read in the same run, and
the oracle's CPU time per case (oracle/eval_oracle.py evaluate_case, simulator and bookkeeping only, fed the planner's
logits) on a sample of cases.

    python profiles/eval_throughput.py [--cases 4500] [--out FILE]
"""
import argparse
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import gnn_pathplanning_b200 as gp  # noqa: E402
from gnn_pathplanning_b200 import synthetic  # noqa: E402
from oracle import eval_oracle, planner_oracle as po  # noqa: E402

N, W, DENSITY, K = 10, 20, 0.1, 3
UNIQUE = 500          # distinct cases, tiled to --cases (the expert's breadth-first search runs on the host)


class Cfg:
    num_agents, nGraphFilterTaps, device = N, K, torch.device("cuda")


class LogitsRecorder:
    def __init__(self, inner):
        self.inner, self.training, self.logits = inner, False, []

    def addGSO(self, S):
        self.inner.addGSO(S)

    def forward_logits(self, x):
        lg = self.inner.forward_logits(x)
        self.logits.append(lg.clone())
        return lg


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def timed_evaluate(model, inp, target, makespan, maps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ro = gp.BatchedRollout(N).setup_cases(inp, target, makespan, maps)
    rec = ro.evaluate(model)                  # ends with the records' device -> host copy
    dt = time.perf_counter() - t0
    return rec, ro.step, dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", type=int, default=4500)
    ap.add_argument("--sample", type=int, default=16, help="cases timed through the CPU oracle")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "eval_throughput.py measures the device: no CUDA device found"
    rng = np.random.default_rng(2024)
    maps, starts, goals, target, makespan = synthetic.random_eval_cases(rng, UNIQUE, N, W, DENSITY)
    rep = np.arange(args.cases) % UNIQUE
    maps, starts, goals, target, makespan = maps[rep], starts[rep], goals[rep], target[rep], makespan[rep]
    inp = np.stack([goals, starts], axis=1)
    sd = po.init_state_dict(K, seed=3)
    po.randomize_bn_stats(sd, seed=4)
    sd["actionsMLP.0.weight"] = sd["actionsMLP.0.weight"] * 40.0
    m = gp.DecentralPlannerNet(Cfg())
    m.load_state_dict(sd)
    m = m.cuda().eval()
    timed_evaluate(m, inp[:64], target[:64], makespan[:64], maps[:64])           # warm-up: weight staging, modules
    runs = [timed_evaluate(m, inp, target, makespan, maps) for _ in range(2)]
    a, b = (dataclasses.asdict(r[0]) for r in runs)
    identical = all(np.array_equal(a[k], b[k]) for k in a)
    # CPU oracle on a sample, fed the planner's logits of the same steps
    S = args.sample
    rec_model = LogitsRecorder(m)
    small = gp.BatchedRollout(N).setup_cases(inp[:S], target[:S], makespan[:S], maps[:S]).evaluate(rec_model)
    lg = torch.stack(rec_model.logits).cpu().numpy()
    t0 = time.perf_counter()
    orc = [eval_oracle.evaluate_case(lambda x, S_, step, c=c: lg[step, :, c], starts[c], goals[c], maps[c], target[c],
                                    makespan[c]) for c in range(S)]
    cpu_s = (time.perf_counter() - t0) / S
    sample_equal = all(orc[c][k] == getattr(small, k)[c] for c in range(S) for k in orc[c])
    summ = gp.summarize(runs[-1][0])
    out = {
        "workload": "evaluate %d cases (N=%d, %dx%d, density %.1f, K=%d; %d distinct cases tiled), one batch"
                    % (args.cases, N, W, W, DENSITY, K, UNIQUE),
        "device": torch.cuda.get_device_name(), "power_limit": power_limit(),
        "runs": [{"seconds": round(dt, 4), "cases_per_s": round(args.cases / dt, 1), "lockstep_steps": steps,
                  "us_per_step": round(1e6 * dt / steps, 2)} for _, steps, dt in runs],
        "records_identical": identical,
        "oracle_cpu_s_per_case": round(cpu_s, 5), "oracle_sample": S, "oracle_sample_equal": sample_equal,
        "rateReachGoal": summ["rateReachGoal"], "avg_rate_deltaMP": summ["avg_rate_deltaMP"],
        "avg_rate_deltaFT": summ["avg_rate_deltaFT"],
        "note": "host clock around setup_cases + evaluate (the records' copy to the host synchronises); "
                "oracle = oracle/eval_oracle.py, one case at a time, 1 thread, simulator + bookkeeping without the model",
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    assert identical and sample_equal


if __name__ == "__main__":
    main()
