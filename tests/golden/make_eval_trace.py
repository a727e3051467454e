"""Generates tests/golden/eval_trace.npz: whole test sets evaluated by the reference's own test loop
(agents/decentralplannerlocal.py mutliAgent_ActionPolicy + utils/metrics.py MonitoringMultiAgentPerformance.update /
summary(label="valid"), unmodified; `random.choice` = the round-robin contract, a fresh chooser per case) with the
deterministic goal-seeking policy of oracle/goal_policy.py.  Stores the cases in the test loader's format, every
per-case field of the recorder and the summary scalars.  Needs a checkout of the original project:
    python tests/golden/make_eval_trace.py
Consumed by tests/test_eval_oracle.py (CPU: oracle/eval_oracle.py) and tests/test_gpu_evaluate.py (GPU: evaluate.cu)."""
import contextlib
import io
import logging
import os
import random
import sys
import warnings

import numpy as np
import torch

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from gnn_pathplanning_b200 import synthetic  # noqa: E402
from oracle import eval_oracle, goal_policy, ref_agent, sim_oracle  # noqa: E402

SETS = {  # name: (N, W, density, random cases); N = 20 runs at maxstep = 3 x makespan (multirobotsim_dcenlocal.py:76-79)
    "a": (10, 20, 0.0, 20),
    "b": (20, 28, 0.05, 4),
}
FIELDS = ("list_reachGoal", "list_noReachGoalSH", "list_findOptimalSolution", "list_collisionFreeSol",
          "list_CollisionPredictedinLoop", "list_MP_predict", "list_MP_target", "list_FT_predict", "list_FT_target",
          "list_numAgentReachGoal", "list_rate_deltaMP", "list_rate_deltaFT")
SUMMARY = ("rateReachGoal", "rateFailedReachGoalSH", "ratefindOptimalSolution", "rateCollsionFreeSol",
           "rateCollisionPredictedinLoop", "avg_rate_deltaMP", "std_rate_deltaMP", "avg_rate_deltaFT", "std_rate_deltaFT")


def l_path(start, goal):
    """Straight-line expert actions (rows first, then columns): getPathTarget never looks at the map."""
    dx, dy = int(goal[0] - start[0]), int(goal[1] - start[1])
    return [2 if dx > 0 else 0] * abs(dx) + [3 if dy > 0 else 1] * abs(dy)


def with_actions(target, i, acts):
    T = max(target.shape[1], len(acts))
    out = np.zeros((target.shape[0], T, 5), dtype=np.float32)
    out[..., 4] = 1.0
    out[:, :target.shape[1]] = target
    out[i] = 0.0
    out[i, :, 4] = 1.0
    out[i, np.arange(len(acts)), 4] = 0.0
    out[i, np.arange(len(acts)), acts] = 1.0
    return out


def boxed_collision_case(m, start, goal, target):
    """Agents 0 and 1 share agent 0's start cell, walled in on all four sides: both stay there, so the collision
    check after shielding fails every step -- a timeout with a real collision (check_CollisionHappenedinLoop)."""
    m, start, target = m.copy(), start.copy(), target.copy()
    W = m.shape[0]
    c = start[0]
    nb = [(c[0] + dx, c[1] + dy) for dx, dy in sim_oracle.DELTA[:4]]
    taken = {tuple(p) for p in np.concatenate([start[1:], goal])}
    if any(p in taken for p in nb) or (goal[1] == c).all():
        return None
    for p in nb:
        if 0 <= p[0] < W and 0 <= p[1] < W:
            m[p] = 1
    start[1] = c
    for i in (0, 1):
        target = with_actions(target, i, l_path(start[i], goal[i]))
    return m, start, goal, target


def pad(targets):
    T = max(t.shape[1] for t in targets)
    out = np.zeros((len(targets), targets[0].shape[0], T, 5), dtype=np.float32)
    out[..., 4] = 1.0
    for b, t in enumerate(targets):
        out[b, :, :t.shape[1]] = t
    return out


def reference_test_loop(agmod, N, maps, starts, goals, target, makespan):
    cfg = ref_agent.make_config(N, 3, "cpu", 2)
    ag = object.__new__(agmod.DecentralPlannerAgentLocal)
    ag.config = cfg
    ag.logger = logging.getLogger("ref-agent")
    ag.model = goal_policy.GoalSeekingPolicy().eval()
    with contextlib.redirect_stdout(io.StringIO()):
        ag.robot = agmod.multiRobotSim(cfg)
    ag.recorder = agmod.MonitoringMultiAgentPerformance(cfg)
    ag.recorder.reset()
    saved = random.choice
    try:
        with torch.no_grad():
            for b in range(maps.shape[0]):
                random.choice = sim_oracle.round_robin_chooser()
                inp = torch.from_numpy(np.stack([goals[b], starts[b]])[None].astype(np.float32))
                res = ag.mutliAgent_ActionPolicy(inp, torch.from_numpy(target[b][None]),
                                                 torch.tensor([float(makespan[b])]),
                                                 torch.from_numpy(maps[b][None].astype(np.float32)), b)
                ag.recorder.update(ag.robot.getMaxstep(), res)
    finally:
        random.choice = saved
    r = ag.recorder
    r.summary("valid", ref_agent._Writer(), 0)
    out = {k: np.asarray([int(v) for v in getattr(r, k)]) for k in FIELDS[5:10] + ("list_reachGoal", "list_noReachGoalSH")}
    out["list_rate_deltaMP"] = np.asarray(r.list_rate_deltaMP, dtype=np.float64)
    out["list_rate_deltaFT"] = np.asarray(r.list_rate_deltaFT, dtype=np.float64)
    out["counts"] = np.array([r.count_reachGoal, r.count_noReachGoalSH, r.count_findOptimalSolution,
                              r.count_collisionFreeSol, r.count_CollisionPredictedinLoop, r.count_validset])
    out["summary"] = np.array([float(getattr(r, k)) for k in SUMMARY])
    out["hist"] = np.array([r.list_numAgentReachGoal.count(i) for i in range(N + 1)])       # test_summary :208-210
    return out


def main():
    policy = goal_policy.GoalSeekingPolicy().eval()
    npolicy = policy.numpy_policy()
    out = {"sets": np.array(sorted(SETS)), "summary_keys": np.array(SUMMARY)}
    kinds = set()
    with ref_agent.reference_env(dropin=False) as agmod:
        for name, (N, W, density, E) in SETS.items():
            rng = np.random.default_rng(ord(name) * 7)
            at_maxstep = None
            maps, starts, goals, target, makespan = synthetic.random_eval_cases(rng, E, N, W, density)
            maps, starts, goals = list(maps), list(starts), list(goals)
            targets, makespan = [t for t in target], list(makespan)
            recs = [eval_oracle.evaluate_case(npolicy, starts[b], goals[b], maps[b], targets[b], makespan[b]) for b in range(E)]
            if name == "a":
                # success exactly at maxstep: the same case with makespan = (step of the all-reached move) / 2; the
                # trajectory up to that move does not depend on maxstep
                for b in range(E):
                    r = recs[b]
                    if not r["list_reachGoal"]:
                        continue
                    sim_final = _final_step(npolicy, maps[b], starts[b], goals[b], targets[b], makespan[b])
                    if sim_final % 2 == 0:
                        maps.append(maps[b]); starts.append(starts[b]); goals.append(goals[b])
                        targets.append(targets[b]); makespan.append(sim_final // 2)
                        at_maxstep = len(maps) - 1
                        break
                for b in range(E):
                    c = boxed_collision_case(maps[b], starts[b], goals[b], targets[b])
                    if c is not None:
                        maps.append(c[0]); starts.append(c[1]); goals.append(c[2]); targets.append(c[3])
                        makespan.append(max(int(np.sum(c[3][i, :, 4] == 0)) for i in range(N)))
                        break
            maps, starts, goals = np.stack(maps), np.stack(starts), np.stack(goals)
            target, makespan = pad(targets), np.array(makespan, dtype=np.int64)
            ref = reference_test_loop(agmod, N, maps, starts, goals, target, makespan)
            orc = [eval_oracle.evaluate_case(npolicy, starts[b], goals[b], maps[b], target[b], makespan[b])
                   for b in range(maps.shape[0])]
            for k in ref:
                if k.startswith("list_"):
                    assert np.array_equal(ref[k], np.array([o[k] for o in orc])), (name, k)
            flags = {k: np.array([o[k] for o in orc]) for k in FIELDS[:5]}
            assert ref["counts"].tolist()[2:5] == [int(flags[k].sum()) for k in FIELDS[2:5]], name
            osum = eval_oracle.summarize(orc, N)
            assert [osum[k] for k in SUMMARY] == ref["summary"].tolist() and osum["hist_numAgentReachGoal"] == ref["hist"].tolist()
            reach, opt, sh, pred = (flags[k] for k in ("list_reachGoal", "list_findOptimalSolution",
                                                        "list_noReachGoalSH", "list_CollisionPredictedinLoop"))
            if at_maxstep is not None and reach[at_maxstep] and flags["list_collisionFreeSol"][at_maxstep] \
                    and not opt[at_maxstep]:
                kinds.add("success at maxstep")
            if (reach & opt).any():
                kinds.add("optimal success")
            if (reach & ~opt.astype(bool)).any():
                kinds.add("non-optimal success")
            if sh.any():
                kinds.add("timeout, shielded")
            if (~reach.astype(bool) & pred.astype(bool) & ~sh.astype(bool)).any():
                kinds.add("timeout, real collision")
            out[name + "_cfg"] = np.array([N, W, maps.shape[0]])
            out[name + "_map"] = maps.astype(np.uint8)
            out[name + "_input"] = np.stack([goals, starts], axis=1).astype(np.int64)     # [B,2,N,2] = (goal, start)
            out[name + "_target"] = target
            out[name + "_makespan"] = makespan
            for k in FIELDS:
                out[name + "_" + k] = ref[k] if k in ref else flags[k]
            out[name + "_summary"] = ref["summary"]
            out[name + "_hist"] = ref["hist"]
            print(name, "N=%d W=%d cases=%d: reach %d, optimal %d, shielded timeouts %d, predicted collisions %d" % (
                N, W, maps.shape[0], reach.sum(), opt.sum(), sh.sum(), pred.sum()))
    for k in ("optimal success", "non-optimal success", "timeout, shielded", "timeout, real collision",
              "success at maxstep"):
        assert k in kinds, "the set lacks a case of kind: " + k
    path = os.path.join(HERE, "eval_trace.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path))


def _final_step(policy, m, st, gl, tgt, mk):
    """Step of the move at which the oracle's loop ends."""
    N = len(st)
    maxstep = int(mk) * (3 if N >= 20 else 2)
    sim = sim_oracle.SimOracle(N, 6.0).setup(st, gl, m, maxstep)
    for step in range(maxstep):
        x, S = sim.inputs(step)
        all_reach, _, _ = sim.move(policy(x, S, step), step + 1)
        if all_reach or step + 1 >= maxstep:
            return step + 1
    return 0


if __name__ == "__main__":
    main()
