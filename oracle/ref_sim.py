"""TEST INFRASTRUCTURE ONLY -- drive the reference's own rollout simulator (utils/multirobotsim_dcenlocal.py, unmodified,
from its checkout, oracle/ref_agent.py) step by step with given logits; reference_rollout needs that checkout,
oracle_rollout (the same rollout through oracle/sim_oracle.py) does not.  `random.choice` (:490) is replaced by the
round-robin contract of oracle/sim_oracle.py for the duration of a rollout, so that the reference becomes deterministic."""
from __future__ import annotations

import random

import numpy as np
import torch

from oracle import ref_agent, sim_oracle


def heuristic_logits(rng, cur, goal, map_hw, beta=1.5, noise=1.0):
    """Goal-seeking policy with Gumbel noise: enough structure that agents converge and conflict, enough noise that the
    edge / obstacle / swap branches fire.  [N,5] float32."""
    N = len(cur)
    out = np.zeros((N, 5), dtype=np.float32)
    for i in range(N):
        for k, (dx, dy) in enumerate(sim_oracle.DELTA):
            nx, ny = cur[i][0] + dx, cur[i][1] + dy
            out[i, k] = -beta * (abs(goal[i][0] - nx) + abs(goal[i][1] - ny))
    return (out + noise * rng.gumbel(size=out.shape)).astype(np.float32)


def reference_rollout(agmod, case, T, seed, num_agents, rate_maxstep=2, noise=1.0):
    """case = (map [W,W], start [N,2], goal [N,2], makespan).  Returns the per-step trace as a dict of arrays."""
    m, start, goal, makespan = case
    N = num_agents
    cfg = ref_agent.make_config(N, 3, "cpu", rate_maxstep)
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        sim = agmod.multiRobotSim(cfg)
    inp = torch.from_numpy(np.stack([goal, start])[None].astype(np.float32))
    tgt = torch.zeros(1, N, int(makespan), 5)
    tgt[..., 4] = 1.0
    chooser = sim_oracle.round_robin_chooser()
    saved = random.choice
    random.choice = chooser
    try:
        sim.setup(inp, tgt, torch.tensor([float(makespan)]), torch.from_numpy(m[None].astype(np.float32)), 0)
        rng = np.random.default_rng(seed)
        tr = {k: [] for k in ("logits", "x", "S", "pos", "flags", "radius", "last_action", "reached")}
        for step in range(T):
            cur = [tuple(int(v) for v in sim.status_MultiAgent["agent%d" % i]["currentState"][0]) for i in range(N)]
            x = sim.getCurrentState()[0].numpy()
            S = sim.getGSO(step)[0].numpy()
            lg = heuristic_logits(rng, cur, [tuple(g) for g in goal], m, noise=noise)
            flags = sim.move([torch.from_numpy(lg[i:i + 1]) for i in range(N)], step + 1)
            pos = [[int(v) for v in sim.status_MultiAgent["agent%d" % i]["currentState"][0]] for i in range(N)]
            tr["logits"].append(lg); tr["x"].append(x.astype(np.uint8)); tr["S"].append(S); tr["pos"].append(pos)
            tr["flags"].append([int(bool(f)) for f in flags]); tr["radius"].append(float(sim.communicationRadius))
            tr["last_action"].append([int(sim.status_MultiAgent["agent%d" % i]["action_predict"][-1]) for i in range(N)])
            tr["reached"].append([int(v) for v in sim.count_reachgoal])
    finally:
        random.choice = saved
    out = {k: np.asarray(v) for k, v in tr.items()}
    out["maxstep"] = np.int64(sim.getMaxstep())
    out["start_step"] = np.array([-1 if sim.status_MultiAgent["agent%d" % i]["startStep_action_predict"] is None
                                  else int(sim.status_MultiAgent["agent%d" % i]["startStep_action_predict"]) for i in range(N)])
    out["end_step"] = np.array([-1 if sim.status_MultiAgent["agent%d" % i]["endStep_action_predict"] is None
                                else int(sim.status_MultiAgent["agent%d" % i]["endStep_action_predict"]) for i in range(N)])
    out["choices"] = np.int64(chooser.state["c"])
    return out


def oracle_rollout(case, T, seed, num_agents, rate_maxstep=2, noise=1.0):
    """The same rollout through oracle/sim_oracle.py (same logits stream)."""
    m, start, goal, makespan = case
    N = num_agents
    if N >= 20:
        rate_maxstep = 3                                                   # multirobotsim_dcenlocal.py:76-79
    sim = sim_oracle.SimOracle(N, 6.0).setup(start, goal, m, int(makespan * rate_maxstep))
    rng = np.random.default_rng(seed)
    tr = {k: [] for k in ("logits", "x", "S", "pos", "flags", "radius", "last_action", "reached")}
    for step in range(T):
        cur = list(sim.cur)
        x, S = sim.inputs(step)
        lg = heuristic_logits(rng, cur, sim.goal, m, noise=noise)
        flags = sim.move(lg, step + 1)
        tr["logits"].append(lg); tr["x"].append(x.astype(np.uint8)); tr["S"].append(S)
        tr["pos"].append([list(p) for p in sim.cur]); tr["flags"].append([int(bool(f)) for f in flags])
        tr["radius"].append(float(sim.radius)); tr["last_action"].append(sim.last_actions())
        tr["reached"].append([int(v) for v in sim.reached])
    out = {k: np.asarray(v) for k, v in tr.items()}
    out["maxstep"] = np.int64(sim.maxstep)
    out["start_step"] = np.array([-1 if v is None else v for v in sim.start_step])
    out["end_step"] = np.array([-1 if v is None else v for v in sim.end_step])
    out["choices"] = np.int64(sim.choose.state["c"])
    return out


def make_case(rng, N, W, density, makespan):
    from gnn_pathplanning_b200 import synthetic
    while True:
        m, start, goal = synthetic.random_episode(rng, N, W, density)
        # an agent that starts ON its goal never records a start step, and the reference's end-of-episode statistics
        # then subtract None (multirobotsim_dcenlocal.py:708 raises TypeError): keep such cases out
        if not (start == goal).all(axis=1).any():
            return m, start, goal, makespan
