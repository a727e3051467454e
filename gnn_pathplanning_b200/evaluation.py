"""Per-case records and summary of a planner's evaluation on a test set (the reference's
MonitoringMultiAgentPerformance, utils/metrics.py:104-210).

`BatchedRollout.evaluate` returns one `CaseRecords` per batch of cases; `summarize(*records)` concatenates them in case
order and computes what `MonitoringMultiAgentPerformance.summary` (and, for the histogram, `test_summary`) computes.
Runs on the host in numpy, once per evaluation.
"""
from __future__ import annotations

import dataclasses

import numpy as np

# column order of the record gpp_rollout_evaluate_finish writes (include/gnnpp_b200.h)
_COLUMNS = ("list_reachGoal", "list_noReachGoalSH", "list_findOptimalSolution", "list_collisionFreeSol",
            "list_CollisionPredictedinLoop", "list_MP_predict", "list_MP_target", "list_FT_predict", "list_FT_target",
            "list_numAgentReachGoal")


@dataclasses.dataclass
class CaseRecords:
    """One entry per case, named after the recorder's lists (int64 flags / metrics, float64 rates)."""
    num_agents: int
    list_reachGoal: np.ndarray
    list_noReachGoalSH: np.ndarray
    list_findOptimalSolution: np.ndarray
    list_collisionFreeSol: np.ndarray
    list_CollisionPredictedinLoop: np.ndarray
    list_MP_predict: np.ndarray
    list_MP_target: np.ndarray
    list_FT_predict: np.ndarray
    list_FT_target: np.ndarray
    list_numAgentReachGoal: np.ndarray
    list_rate_deltaMP: np.ndarray
    list_rate_deltaFT: np.ndarray

    @classmethod
    def from_record(cls, record: np.ndarray, num_agents: int) -> "CaseRecords":
        """record: int [B,10] in the column order of gpp_rollout_evaluate_finish."""
        cols = {k: np.asarray(record[:, i], dtype=np.int64) for i, k in enumerate(_COLUMNS)}
        return cls(num_agents=int(num_agents), **cols, **_rates(cols))

    def __len__(self) -> int:
        return int(self.list_reachGoal.shape[0])


def _rates(cols):
    # metrics.py:110-111: abs(predict - target) / target, Python int / int -> IEEE double, as numpy's true division
    return {"list_rate_deltaMP": np.abs(cols["list_MP_predict"] - cols["list_MP_target"]) / cols["list_MP_target"],
            "list_rate_deltaFT": np.abs(cols["list_FT_predict"] - cols["list_FT_target"]) / cols["list_FT_target"]}


def concatenate(*records: CaseRecords) -> CaseRecords:
    """Chunks of one evaluation, in case order."""
    if not records:
        raise ValueError("concatenate: no records")
    n = {r.num_agents for r in records}
    if len(n) != 1:
        raise ValueError("concatenate: records of different agent counts %s" % sorted(n))
    fields = [f.name for f in dataclasses.fields(CaseRecords) if f.name != "num_agents"]
    return CaseRecords(num_agents=n.pop(), **{k: np.concatenate([getattr(r, k) for r in records]) for k in fields})


def summarize(*records: CaseRecords) -> dict:
    """MonitoringMultiAgentPerformance.summary (metrics.py:154-177) over all cases of `records`, plus test_summary's
    histogram of the number of agents that reached their goals (:208-210)."""
    r = concatenate(*records)
    n = len(r)
    return {
        "num_cases": n,
        "rateReachGoal": int(r.list_reachGoal.sum()) / n,
        "rateFailedReachGoalSH": int(r.list_noReachGoalSH.sum()) / n,
        "ratefindOptimalSolution": int(r.list_findOptimalSolution.sum()) / n,
        "rateCollsionFreeSol": int(r.list_collisionFreeSol.sum()) / n,
        "rateCollisionPredictedinLoop": int(r.list_CollisionPredictedinLoop.sum()) / n,
        "avg_rate_deltaMP": float(np.mean(r.list_rate_deltaMP)),
        "std_rate_deltaMP": float(np.std(r.list_rate_deltaMP, ddof=1)),
        "avg_rate_deltaFT": float(np.mean(r.list_rate_deltaFT)),
        "std_rate_deltaFT": float(np.std(r.list_rate_deltaFT, ddof=1)),
        "hist_numAgentReachGoal": np.bincount(r.list_numAgentReachGoal, minlength=r.num_agents + 1).tolist(),
    }
