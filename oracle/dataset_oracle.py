"""CPU ORACLE -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Restatement (numpy, one case at a time) of what the original project's online-expert DataTransformer writes into a
case's .mat file and of the failure-case file its simulator writes -- the checker for
gnn_pathplanning_b200/csrc/dataset.cu and gnn_pathplanning_b200/dataset.py (SURVEY.md section 8 row f3):

    obtainSchedule                     onlineExpert/DataTransformer_local_onlineExpert.py:154-196
    computeAdjacencyMatrix(states, 5)  :256-305 (one threshold grown across the whole schedule)
    AgentState.toSeqInputTensor        dataloader/statetransformer.py:133-187
    multiRobotSim.save_failure_cases   utils/multirobotsim_dcenlocal_onlineExpert.py:705-730

PARITY PINNING: tests/golden/make_schedule_trace.py runs the reference's own DataTransformer and online-expert agent
and stores what they wrote in tests/golden/schedule_trace.npz; tests/test_dataset_oracle.py checks this module
against it bit for bit.
"""
from __future__ import annotations

import numpy as np

from .sim_oracle import fov_tensor, is_connected

DELTA = [[-1, 0], [0, -1], [1, 0], [0, 1], [0, 0]]       # DataTransformer.delta: up, left, down, right, stop


def obtain_schedule(plans, goals, makespan):
    """plans: per agent a list of (x, y) cells (the solver's schedule); goals [N,2].  Returns (positions [T,N,2] int64,
    one-hot targets [T,N,5] float64) for T = makespan + 1 rows; raises ValueError where the reference's
    `delta.index` would."""
    T, N = int(makespan) + 1, len(plans)
    pos = np.zeros((T, N, 2), dtype=np.int64)
    tgt = np.zeros((T, N, 5), dtype=np.float64)
    for i, plan in enumerate(plans):
        for t in range(T):
            cur = list(plan[t]) if t < len(plan) else list(goals[i])
            nxt = list(plan[t + 1]) if t < len(plan) - 1 else list(goals[i])
            d = [int(nxt[0]) - int(cur[0]), int(nxt[1]) - int(cur[1])]
            if d not in DELTA:
                raise ValueError("agent %d step %d: move %s is not one of %s" % (i, t, d, DELTA))
            pos[t, i] = cur
            tgt[t, i, DELTA.index(d)] = 1.0
    return pos, tgt


def schedule_threshold(positions, r0=5.0):
    """The threshold computeAdjacencyMatrix ends with: one value grown by 10 % while a step is disconnected, walking
    the steps in order and never resetting it."""
    thr = r0
    for p in np.asarray(positions, dtype=np.float64):
        d = np.sqrt(((p[:, None, :] - p[None, :, :]) ** 2).sum(-1))
        while True:
            A = (d < thr).astype(np.float64)
            A -= np.diag(np.diag(A))
            if is_connected(A):
                break
            thr = thr * 1.1
    return thr


def schedule_gso(positions, thr):
    """Every step's D^-1/2 A D^-1/2 (float64) at the final threshold, with no zero-degree guard."""
    out = []
    for p in np.asarray(positions, dtype=np.float64):
        d = np.sqrt(((p[:, None, :] - p[None, :, :]) ** 2).sum(-1))
        A = (d < thr).astype(np.float64)
        A -= np.diag(np.diag(A))
        D = np.diag(np.sqrt(1.0 / A.sum(axis=1)))
        out.append(D @ A @ D)
    return np.stack(out)


def seq_input_tensor(map_hw, goals, positions):
    """toSeqInputTensor: the field of view of every step, float32 [T,N,3,11,11]."""
    return np.stack([fov_tensor(map_hw, goals, p) for p in positions])


def transform(map_hw, goals, positions, r0=5.0):
    """The fields of one case's training file: inputTensor, GSO (float64), target (one-hot float64) and the threshold."""
    positions = np.asarray(positions, dtype=np.int64)
    T = positions.shape[0]
    nxt = np.concatenate([positions[1:], np.asarray(goals, dtype=np.int64)[None]])
    d = nxt - positions
    key = {tuple(v): k for k, v in enumerate(DELTA)}
    tgt = np.zeros(positions.shape[:2] + (5,), dtype=np.float64)
    for t in range(T):
        for i in range(positions.shape[1]):
            tgt[t, i, key[tuple(int(v) for v in d[t, i])]] = 1.0
    thr = schedule_threshold(positions, r0)
    return {"inputTensor": seq_input_tensor(map_hw, goals, positions), "GSO": schedule_gso(positions, thr),
            "target": tgt, "threshold": thr}


def failure_case_text(map_hw, cells, goals):
    """save_failure_cases: the solver input for one case, agents starting from their final cells."""
    m = np.asarray(map_hw)
    lines = ["map:", "    dimensions: [%d, %d]" % m.shape, "    obstacles:"]
    lines += ["    - [%d, %d]" % (int(x), int(y)) for x, y in zip(*np.nonzero(m))]
    lines.append("agents:")
    for i, (c, g) in enumerate(zip(cells, goals)):
        lines += ["  - name: agent%d" % i, "    start: [%d, %d]" % (int(c[0]), int(c[1])),
                  "    goal: [%d, %d]" % (int(g[0]), int(g[1]))]
    return "\n".join(lines) + "\n"
