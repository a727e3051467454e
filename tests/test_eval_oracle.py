"""CPU: the test-loop oracle (oracle/eval_oracle.py evaluate_case / summarize) against whole test sets evaluated by the
reference's own mutliAgent_ActionPolicy + MonitoringMultiAgentPerformance (tests/golden/eval_trace.npz); the host-side
checks of BatchedRollout.setup_cases; evaluation.summarize over chunks."""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("list_reachGoal", "list_noReachGoalSH", "list_findOptimalSolution", "list_collisionFreeSol",
          "list_CollisionPredictedinLoop", "list_MP_predict", "list_MP_target", "list_FT_predict", "list_FT_target",
          "list_numAgentReachGoal")


@pytest.fixture(scope="module")
def trace():
    return np.load(os.path.join(ROOT, "tests", "golden", "eval_trace.npz"), allow_pickle=False)


def _sets(trace):
    for name in trace["sets"]:
        name = str(name)
        yield name, {k[len(name) + 1:]: trace[k] for k in trace.files if k.startswith(name + "_")}


def _records(g):
    from gnn_pathplanning_b200.evaluation import CaseRecords
    return CaseRecords.from_record(np.stack([g[k] for k in FIELDS], axis=1), int(g["cfg"][0]))


def test_oracle_vs_reference_test_loop(trace):
    from oracle import eval_oracle, goal_policy
    policy = goal_policy.GoalSeekingPolicy().eval().numpy_policy()
    keys = [str(k) for k in trace["summary_keys"]]
    for name, g in _sets(trace):
        N = int(g["cfg"][0])
        recs = [eval_oracle.evaluate_case(policy, g["input"][b, 1], g["input"][b, 0], g["map"][b], g["target"][b],
                                         g["makespan"][b]) for b in range(g["input"].shape[0])]
        for k in FIELDS + ("list_rate_deltaMP", "list_rate_deltaFT"):
            assert np.array_equal(np.array([r[k] for r in recs]), g[k]), (name, k)
        s = eval_oracle.summarize(recs, N)
        assert [s[k] for k in keys] == g["summary"].tolist(), name
        assert s["hist_numAgentReachGoal"] == g["hist"].tolist(), name


def test_records_and_summary_vs_reference(trace):
    """CaseRecords' rates and evaluation.summarize over the reference's per-case fields give its summary exactly."""
    from gnn_pathplanning_b200 import evaluation
    keys = [str(k) for k in trace["summary_keys"]]
    for name, g in _sets(trace):
        r = _records(g)
        assert np.array_equal(r.list_rate_deltaMP, g["list_rate_deltaMP"]), name
        assert np.array_equal(r.list_rate_deltaFT, g["list_rate_deltaFT"]), name
        s = evaluation.summarize(r)
        assert [s[k] for k in keys] == g["summary"].tolist(), name
        assert s["hist_numAgentReachGoal"] == g["hist"].tolist() and s["num_cases"] == len(r), name


def test_summarize_over_chunks(trace):
    from gnn_pathplanning_b200 import evaluation
    for name, g in _sets(trace):
        r = _records(g)
        n = len(r)
        fields = [k for k in vars(r) if k != "num_agents"]
        parts = [evaluation.CaseRecords(r.num_agents, **{k: getattr(r, k)[sl] for k in fields})
                 for sl in (slice(0, n // 3), slice(n // 3, n))]
        assert evaluation.summarize(*parts) == evaluation.summarize(r), name
        with pytest.raises(ValueError):
            evaluation.summarize(r, evaluation.CaseRecords(r.num_agents + 1, **{k: getattr(r, k) for k in fields}))


def test_setup_cases_rejects_what_the_reference_crashes_on(trace):
    """Checked on the host before any launch: these run without a GPU."""
    import gnn_pathplanning_b200 as gp
    g = dict(_sets(trace))["a"]
    N = int(g["cfg"][0])
    inp, tgt, mk, maps = g["input"][:4].copy(), g["target"][:4].copy(), g["makespan"][:4].copy(), g["map"][:4]
    ro = gp.BatchedRollout(N)
    bad = inp.copy()
    bad[2, 1, 3] = bad[2, 0, 3]                               # case 2, agent 3 starts on its goal
    with pytest.raises(ValueError, match=r"starts on its goal in cases \[2\]"):
        ro.setup_cases(bad, tgt, mk, maps)
    bad = tgt.copy()
    bad[1, 5] = 0.0
    bad[1, 5, :, 4] = 1.0                                     # case 1, agent 5: the expert never moves
    with pytest.raises(ValueError, match=r"off its goal in cases \[1\]"):
        ro.setup_cases(inp, bad, mk, maps)
    bad = mk.copy()
    bad[[0, 3]] = 0
    with pytest.raises(ValueError, match=r"makespan < 1 in cases \[0, 3\]"):
        ro.setup_cases(inp, tgt, bad, maps)
    with pytest.raises(ValueError, match="expected input"):
        ro.setup_cases(inp[:, :, :5], tgt, mk, maps)
