"""Generates tests/golden/schedule_trace.npz: what the original project's online expert writes, from its own code,
unmodified.  Needs a checkout of the original project:
    python tests/golden/make_schedule_trace.py

* Schedules.  Synthetic solver-format input / solution YAMLs (one set per case) are written to a temporary directory and
  turned into training files by the reference's DataTransformer (onlineExpert/DataTransformer_local_onlineExpert.py,
  `pipeline` per case, as its worker processes call it).  Stored per case: exactly what the .mat file holds (map, goal,
  inputState, inputTensor as uint8, target as uint8, GSO float64, makespan), the threshold computeAdjacencyMatrix
  returned, and the two YAML texts.  Cases: N = 10 on one shared 20x20 map, N = 10 with `obstacles: None`, N = 20 on
  28x28, N = 5 on 50x50 (one whose threshold grows only at later steps), N = 64 on 32x32; random walks with waits and
  plans of different lengths (goal padding).  One more solution has a two-cell jump, on which the reference raises.
* Failure cases.  The reference online-expert agent's mutliAgent_ActionPolicy(..., mode='test_trainingSet') with
  switch_toOnlineExpert = True on the cases of tests/golden/eval_trace.npz, driven by oracle/goal_policy.py with the
  round-robin chooser (as make_eval_trace.py does).  Stored: the file names it wrote, their texts and each failed case's
  final cells.
Consumed by tests/test_dataset_oracle.py (CPU) and tests/test_gpu_dataset.py (GPU)."""
import contextlib
import importlib
import io
import logging
import os
import random
import sys
import tempfile
import warnings

import numpy as np
import scipy.io
import torch

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import goal_policy, ref_agent, sim_oracle  # noqa: E402

DELTA = sim_oracle.DELTA


def random_map(rng, W, density):
    m = (rng.random((W, W)) < density).astype(np.int64)
    return m


def random_walks(rng, m, N, lengths, p_wait=0.25):
    """One plan per agent: a walk over free cells from distinct starts, with waits; the last cell is the goal."""
    W = m.shape[0]
    free = np.argwhere(m == 0)
    starts = free[rng.choice(len(free), N, replace=False)]
    plans = []
    for i in range(N):
        p = [tuple(int(v) for v in starts[i])]
        for _ in range(lengths[i] - 1):
            x, y = p[-1]
            opts = [(x + dx, y + dy) for dx, dy in DELTA[:4] if 0 <= x + dx < W and 0 <= y + dy < W and m[x + dx, y + dy] == 0]
            p.append(p[-1] if (rng.random() < p_wait or not opts) else opts[rng.integers(len(opts))])
        plans.append(p)
    return plans


def diverging_plans():
    """Five agents four cells apart in a row (connected at 5); agent i walks 4i cells down and stays: the pairs end
    sqrt(32) apart, so the threshold grows only once the later steps are reached."""
    plans = []
    for i in range(5):
        p = [(25, 10 + 4 * i)]
        for _ in range(4 * i):
            p.append((p[-1][0] + 1, p[-1][1]))
        plans.append(p)
    return plans


def input_yaml(m, starts, goals, obstacles_none=False):
    lines = ["map:", "    dimensions: [%d, %d]" % m.shape, "    obstacles:"]
    if not obstacles_none:
        lines += ["    - [%d, %d]" % (x, y) for x, y in np.argwhere(m != 0).tolist()]
    lines.append("agents:")
    for i, (s, g) in enumerate(zip(starts, goals)):
        lines += ["  - name: agent%d" % i, "    start: [%d, %d]" % tuple(s), "    goal: [%d, %d]" % tuple(g)]
    return "\n".join(lines) + "\n"


def solution_yaml(plans):
    makespan = max(len(p) for p in plans) - 1
    lines = ["statistics:", "  cost: %d" % sum(len(p) - 1 for p in plans), "  makespan: %d" % makespan,
             "  runtime: 0.01", "  highLevelExpanded: 1", "  lowLevelExpanded: 1", "schedule:"]
    for i, p in enumerate(plans):
        lines.append("  agent%d:" % i)
        for t, (x, y) in enumerate(p):
            lines += ["    - x: %d" % x, "      y: %d" % y, "      t: %d" % t]
    return "\n".join(lines) + "\n"


def make_cases():
    """name -> (W, input yaml, solution yaml)."""
    rng = np.random.default_rng(2024)
    cases = {}
    shared = random_map(rng, 20, 0.1)
    for k in range(4):
        plans = random_walks(rng, shared, 10, rng.integers(3, 26, 10))
        cases["n10_shared%d" % k] = (shared, plans, False)
    m = np.zeros((20, 20), dtype=np.int64)
    cases["n10_none"] = (m, random_walks(rng, m, 10, rng.integers(5, 20, 10)), True)
    for k in range(2):
        m = random_map(rng, 28, 0.05)
        cases["n20_%d" % k] = (m, random_walks(rng, m, 20, rng.integers(4, 30, 20)), False)
    cases["n5_late"] = (np.zeros((50, 50), dtype=np.int64), diverging_plans(), False)
    m = random_map(rng, 50, 0.05)
    cases["n5_scattered"] = (m, random_walks(rng, m, 5, rng.integers(10, 30, 5)), False)
    m = random_map(rng, 32, 0.05)
    cases["n64"] = (m, random_walks(rng, m, 64, rng.integers(5, 25, 64)), False)
    out = {}
    for name, (m, plans, none) in cases.items():
        out[name] = (m.shape[0], input_yaml(m, [p[0] for p in plans], [p[-1] for p in plans], none), solution_yaml(plans))
    return out


def run_transformer(dtmod, N, W, inp, sol, epoch=1):
    """The reference's DataTransformer on one case; returns (the .mat file's name, its contents, the threshold)."""
    with tempfile.TemporaryDirectory() as d:
        root = d + "/"
        os.makedirs(os.path.join(root, "input"))
        os.makedirs(os.path.join(root, "output_ECBS"))
        with open(os.path.join(root, "input", "failureCases_ID00000.yaml"), "w") as f:
            f.write(inp)
        with open(os.path.join(root, "output_ECBS", "failureCases_solved_ID00000.yaml"), "w") as f:
            f.write(sol)
        cfg = ref_agent.EasyDict(num_agents=N, map_w=W, map_h=W, failCases_dir=root, exp_net="dcp")
        dt = dtmod.DataTransformer(cfg)
        dt.set_up(epoch)
        seen = []
        orig = dt.computeAdjacencyMatrix

        def spy(*a, **k):
            r = orig(*a, **k)
            seen.append(r[1])
            return r
        dt.computeAdjacencyMatrix = spy
        with contextlib.redirect_stdout(io.StringIO()):
            dt.pipeline(0)
        files = os.listdir(dt.path_save_solDATA)
        assert len(files) == 1, files
        mat = scipy.io.loadmat(os.path.join(dt.path_save_solDATA, files[0]))
        return files[0], mat, seen[0]


def failure_cases(onmod, eval_trace, set_name):
    """The online-expert agent's test loop on one eval-trace set; returns (ids, file names, texts, final cells)."""
    g = {k[len(set_name) + 1:]: eval_trace[k] for k in eval_trace.files if k.startswith(set_name + "_")}
    N = int(g["cfg"][0])
    cfg = ref_agent.make_config(N, 3, "cpu", 2)
    with tempfile.TemporaryDirectory() as d:
        cfg.failCases_dir = d + "/"
        ag = object.__new__(onmod.DecentralPlannerAgentLocalWithOnlineExpert)
        ag.config = cfg
        ag.logger = logging.getLogger("ref-agent")
        ag.model = goal_policy.GoalSeekingPolicy().eval()
        ag.switch_toOnlineExpert = True
        with contextlib.redirect_stdout(io.StringIO()):
            ag.robot = onmod.multiRobotSim(cfg)
            ag.robot.createfolder_failure_cases()
        saved = random.choice
        ids, cells = [], []
        try:
            with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
                for b in range(g["input"].shape[0]):
                    random.choice = sim_oracle.round_robin_chooser()
                    inp = torch.from_numpy(g["input"][b][None].astype(np.float32))
                    before = set(os.listdir(ag.robot.failureCases_input))
                    ag.mutliAgent_ActionPolicy(inp, torch.from_numpy(g["target"][b][None]),
                                               torch.tensor([float(g["makespan"][b])]),
                                               torch.from_numpy(g["map"][b][None].astype(np.float32)), b,
                                               "test_trainingSet")
                    if set(os.listdir(ag.robot.failureCases_input)) != before:
                        ids.append(b)
                        cells.append([[int(v) for v in ag.robot.status_MultiAgent["agent%d" % i]["nextState_predict"][0]]
                                      for i in range(N)])
        finally:
            random.choice = saved
        names = sorted(os.listdir(ag.robot.failureCases_input))
        texts = [open(os.path.join(ag.robot.failureCases_input, n)).read() for n in names]
    return np.array(ids, dtype=np.int64), names, texts, np.array(cells, dtype=np.int64).reshape(-1, N, 2)


def main():
    out = {}
    cases = make_cases()
    with ref_agent.reference_env(dropin=False):
        dtmod = importlib.import_module("onlineExpert.DataTransformer_local_onlineExpert")
        onmod = importlib.import_module("agents.decentralplannerlocal_OnlineExpert")
        for name, (W, inp, sol) in cases.items():
            N = inp.count("name: agent")
            fname, mat, thr = run_transformer(dtmod, N, W, inp, sol)
            for k in ("inputTensor", "target"):
                assert np.isin(mat[k], (0, 1)).all(), (name, k)
            assert mat["GSO"].dtype == np.float64
            out[name + "_file"] = np.array(fname)
            out[name + "_map"] = mat["map"].astype(np.uint8)
            out[name + "_goal"] = mat["goal"].astype(np.int64)
            out[name + "_inputState"] = mat["inputState"].astype(np.int64)
            out[name + "_inputTensor"] = mat["inputTensor"].astype(np.uint8)
            out[name + "_target"] = mat["target"].astype(np.uint8)
            out[name + "_GSO"] = mat["GSO"]
            out[name + "_makespan"] = np.int64(mat["makespan"].item())
            out[name + "_threshold"] = np.float64(thr)
            out[name + "_input_yaml"] = np.array(inp)
            out[name + "_solution_yaml"] = np.array(sol)
            print(name, "N=%d W=%d T=%d threshold=%r" % (N, W, mat["inputState"].shape[0], thr))
        # a solution whose agent 3 jumps two cells: delta.index raises ValueError in the reference
        W, inp, sol = cases["n10_shared0"]
        lines = sol.split("\n")
        k = lines.index("  agent3:") + 4                # agent 3's second cell, two rows from its first
        x = int(lines[k - 3].split(":")[1])
        lines[k] = "    - x: %d" % (x + 2 if x + 2 < W else x - 2)
        bad = "\n".join(lines)
        try:
            run_transformer(dtmod, 10, W, inp, bad)
            raise AssertionError("the reference accepted a two-cell jump")
        except ValueError:
            pass
        out["invalid_input_yaml"] = np.array(inp)
        out["invalid_solution_yaml"] = np.array(bad)
        eval_trace = np.load(os.path.join(HERE, "eval_trace.npz"))
        for s in ("a", "b"):
            ids, names, texts, cells = failure_cases(onmod, eval_trace, s)
            print("failure cases of set", s, ids.tolist())
            out["fail_%s_ids" % s] = ids
            out["fail_%s_names" % s] = np.array(names)
            out["fail_%s_texts" % s] = np.array(texts)
            out["fail_%s_cells" % s] = cells
    out["cases"] = np.array(sorted(cases))
    path = os.path.join(HERE, "schedule_trace.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path))


if __name__ == "__main__":
    main()
