"""CPU ORACLE -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Restatement (plain Python, one case at a time) of the reference's test loop around the rollout simulator -- the checker
for gnn_pathplanning_b200/csrc/evaluate.cu and gnn_pathplanning_b200/evaluation.py:

    multiRobotSim.getPathTarget        utils/multirobotsim_dcenlocal.py:159-229
    multiRobotSim.move (statistics)    :693-715
    multiRobotSim.checkOptimality      :825-832
    mutliAgent_ActionPolicy            agents/decentralplannerlocal.py:535-648
    MonitoringMultiAgentPerformance    utils/metrics.py:104-210 (update, summary, test_summary's histogram)

The simulator itself is oracle/sim_oracle.py's SimOracle.  PARITY PINNING: tests/golden/make_eval_trace.py checks this
module against the reference's own test loop and records it into tests/golden/eval_trace.npz, which
tests/test_eval_oracle.py (CPU) and tests/test_gpu_evaluate.py (GPU) replay.
"""
from __future__ import annotations

import numpy as np

from oracle.sim_oracle import DELTA, STOP, SimOracle


class EvalSimOracle(SimOracle):
    """SimOracle plus the expert replay and the end-of-episode statistics the test loop reads."""
    def setup_targets(self, target):
        """getPathTarget (:159-229) for the expert's one-hot actions target [N,T,5]; call right after setup().  Sets
        target_start / target_end (None = never), makespanTarget, flowtimeTarget (0 unless every agent arrives)."""
        assert all(not a for a in self.act), "setup_targets() replays from the start cells: call it before move()"
        target = np.asarray(target)
        N, T = self.N, target.shape[1]
        keys = [[int(np.argmax(target[i, t])) for t in range(T)] for i in range(N)]      # torch.max(., 1)[1] (:112)
        self.target_start = [None] * N
        self.target_end = [None] * N
        reached = [False] * N
        self.makespanTarget = 0                                           # setup :89-90
        self.flowtimeTarget = 0
        all_reach = False
        for i in range(N):
            cur = nxt = self.cur[i]
            for step in range(T):                                         # :183-207
                key = keys[i][step]
                if key != STOP and self.target_start[i] is None:
                    self.target_start[i] = step
                else:
                    cur = nxt
                nxt = (cur[0] + DELTA[key][0], cur[1] + DELTA[key][1])
                if nxt == self.goal[i] and not reached[i]:
                    reached[i] = True
                    self.target_end[i] = step + 1
                all_reach = all(reached)
            if all_reach:                                                 # :209-228
                self.flowtimeTarget = sum(e - s for e, s in zip(self.target_end, self.target_start))
                self.makespanTarget = max(self.target_end) - min(self.target_start)
                break
        return self.makespanTarget, self.flowtimeTarget

    def predicted_metrics(self):
        """The end-of-episode statistics of move (:693-715): (makespanPredict, flowtimePredict)."""
        flowtime = sum(e - s for e, s in zip(self.end_step, self.start_step))
        return max(self.end_step) - min(self.start_step), flowtime


def evaluate_case(policy, start, goal, map_hw, target, makespan, rate_maxstep=2, comm_radius=6.0, chooser=None):
    """One test case as mutliAgent_ActionPolicy (agents/decentralplannerlocal.py:535-648) runs it and
    MonitoringMultiAgentPerformance.update (utils/metrics.py:104-152) records it.  policy(x [N,3,11,11] f32,
    S [N,N] f64, step) -> logits [N,5].  Returns the case's record as a dict named after the recorder's lists."""
    N = len(start)
    rate = 3 if N >= 20 else rate_maxstep                                 # multirobotsim_dcenlocal.py:76-81
    maxstep = int(np.int32(makespan)) * rate
    sim = EvalSimOracle(N, comm_radius, chooser).setup(start, goal, map_hw, maxstep)
    mp_target, ft_target = sim.setup_targets(target)
    mp_predict, ft_predict = maxstep, maxstep * N                         # setup :91-92
    compare_mp, compare_ft = [mp_predict, mp_target], [ft_predict, ft_target]       # getOptimalityMetrics (:555)
    all_reach = no_reach_sh = optimal = collision_free = happened = predicted = False
    current = 0
    for step in range(maxstep):                                           # :560-606
        current = step + 1
        x, S = sim.inputs(step)
        all_reach, move_coll, predict_coll = sim.move(policy(x, S, step), current)
        if all_reach or current >= maxstep:                               # move :693-715
            mp_predict, ft_predict = sim.predicted_metrics()
        happened = happened or bool(move_coll)
        predicted = predicted or bool(predict_coll)
        if all_reach or current >= maxstep:
            break

    def check_optimality(free):                                           # multirobotsim_dcenlocal.py:825-832
        return (mp_predict <= mp_target and ft_predict <= ft_target and free), [mp_predict, mp_target], \
            [ft_predict, ft_target]

    if all_reach and not happened:                                        # :611-614
        collision_free = True
        optimal, compare_mp, compare_ft = check_optimality(True)
    if current >= maxstep:                                                # :618-619
        optimal, compare_mp, compare_ft = check_optimality(False)
    if current >= maxstep and not all_reach and predicted and not happened:      # :621-624
        optimal, compare_mp, compare_ft = check_optimality(False)
        no_reach_sh = True
    return {"list_reachGoal": int(bool(all_reach)), "list_noReachGoalSH": int(no_reach_sh),
            "list_findOptimalSolution": int(bool(optimal)), "list_collisionFreeSol": int(collision_free),
            "list_CollisionPredictedinLoop": int(predicted),
            "list_MP_predict": compare_mp[0], "list_MP_target": compare_mp[1],
            "list_FT_predict": compare_ft[0], "list_FT_target": compare_ft[1],
            "list_numAgentReachGoal": sum(bool(r) for r in sim.reached),
            "list_rate_deltaMP": abs(compare_mp[0] - compare_mp[1]) / compare_mp[1],          # metrics.py:110-111
            "list_rate_deltaFT": abs(compare_ft[0] - compare_ft[1]) / compare_ft[1]}


def summarize(records, num_agents):
    """MonitoringMultiAgentPerformance.update's counters and summary (utils/metrics.py:130-177) over per-case record
    dicts in case order, plus test_summary's histogram (:208-210)."""
    n = len(records)
    count = lambda k: sum(1 for r in records if r[k])                     # noqa: E731
    mp = np.array([r["list_rate_deltaMP"] for r in records])
    ft = np.array([r["list_rate_deltaFT"] for r in records])
    reach = [r["list_numAgentReachGoal"] for r in records]
    return {"num_cases": n,
            "rateReachGoal": count("list_reachGoal") / n,
            "rateFailedReachGoalSH": count("list_noReachGoalSH") / n,
            "ratefindOptimalSolution": count("list_findOptimalSolution") / n,
            "rateCollsionFreeSol": count("list_collisionFreeSol") / n,
            "rateCollisionPredictedinLoop": count("list_CollisionPredictedinLoop") / n,
            "avg_rate_deltaMP": float(np.mean(mp)), "std_rate_deltaMP": float(np.std(mp, ddof=1)),
            "avg_rate_deltaFT": float(np.mean(ft)), "std_rate_deltaFT": float(np.std(ft, ddof=1)),
            "hist_numAgentReachGoal": [reach.count(i) for i in range(num_agents + 1)]}
