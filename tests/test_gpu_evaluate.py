"""GPU: per-case evaluation of lock-step rollouts (csrc/evaluate.cu via BatchedRollout.setup_cases / evaluate) against
whole test sets evaluated by the reference's own test loop (tests/golden/eval_trace.npz) and against
oracle/eval_oracle.py fed the same logits -- every per-case field bit-exact, rates and summaries equal."""
import os

import numpy as np
import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("list_reachGoal", "list_noReachGoalSH", "list_findOptimalSolution", "list_collisionFreeSol",
          "list_CollisionPredictedinLoop", "list_MP_predict", "list_MP_target", "list_FT_predict", "list_FT_target",
          "list_numAgentReachGoal", "list_rate_deltaMP", "list_rate_deltaFT")


@pytest.fixture(scope="module")
def eval_trace():
    g = np.load(os.path.join(ROOT, "tests", "golden", "eval_trace.npz"), allow_pickle=False)
    return {str(n): {k[len(str(n)) + 1:]: g[k] for k in g.files if k.startswith(str(n) + "_")} for n in g["sets"]} | \
        {"summary_keys": [str(k) for k in g["summary_keys"]]}


class LogitsRecorder:
    """Wraps a model for evaluate(): keeps every step's [N,B,5] logits on the device."""

    def __init__(self, inner):
        self.inner, self.training, self.logits = inner, False, []

    def addGSO(self, S):
        self.inner.addGSO(S)

    def forward_logits(self, x):
        lg = self.inner.forward_logits(x)
        self.logits.append(lg.clone())
        return lg


class Cfg:
    def __init__(self, n, k):
        self.num_agents, self.nGraphFilterTaps, self.device = n, k, torch.device("cuda")


def test_evaluate_vs_reference_test_loop(eval_trace):
    import gnn_pathplanning_b200 as gp
    from oracle import goal_policy
    policy = goal_policy.GoalSeekingPolicy().eval()
    for name in ("a", "b"):
        g = eval_trace[name]
        ro = gp.BatchedRollout(int(g["cfg"][0])).setup_cases(g["input"], g["target"], g["makespan"], g["map"])
        rec = ro.evaluate(policy, poll_every=4)
        for k in FIELDS:
            assert np.array_equal(getattr(rec, k), g[k]), (name, k)
        s = gp.summarize(rec)
        assert [s[k] for k in eval_trace["summary_keys"]] == g["summary"].tolist(), name
        assert s["hist_numAgentReachGoal"] == g["hist"].tolist(), name


@pytest.mark.parametrize("N,W,B", [(10, 20, 64), (20, 28, 17), (40, 36, 5)])
def test_evaluate_planner_vs_oracle(N, W, B):
    """The CUDA planner drives B cases of mixed makespans (cases freeze at different steps); the oracle's test loop,
    fed each case's logits of the same steps, gives the same per-case records.  N = 20 runs at maxstep = 3 x makespan,
    N = 40 the thread-per-episode move kernel."""
    import gnn_pathplanning_b200 as gp
    from gnn_pathplanning_b200 import synthetic
    from oracle import eval_oracle, planner_oracle as po
    rng = np.random.default_rng(N * W + B)
    maps, starts, goals, target, makespan = synthetic.random_eval_cases(rng, B, N, W, 0.1)
    assert len(set(makespan.tolist())) > 1
    sd = po.init_state_dict(3, seed=3)
    po.randomize_bn_stats(sd, seed=4)
    sd["actionsMLP.0.weight"] = sd["actionsMLP.0.weight"] * 40.0          # a policy that moves
    m = gp.DecentralPlannerNet(Cfg(N, 3))
    m.load_state_dict(sd)
    model = LogitsRecorder(m.cuda().eval())
    ro = gp.BatchedRollout(N).setup_cases(np.stack([goals, starts], axis=1), target, makespan, maps)
    rec = ro.evaluate(model, poll_every=8)
    lg = torch.stack(model.logits).cpu().numpy()                          # [steps,N,B,5]
    for b in range(B):
        r = eval_oracle.evaluate_case(lambda x, S, step: lg[step, :, b], starts[b], goals[b], maps[b], target[b],
                                     makespan[b])
        for k in FIELDS:
            assert getattr(rec, k)[b] == r[k], (b, k)
    s = gp.summarize(rec)
    assert 0.0 <= s["rateReachGoal"] <= 1.0 and sum(s["hist_numAgentReachGoal"]) == B


def test_targets_vs_oracle_ragged_and_maps():
    """gpp_rollout_targets on cases of different expert lengths padded with 'stop' to one T, with a shared [W,W] map
    and with per-case maps: per-agent start / end steps and per-case makespan / flowtime targets as getPathTarget."""
    import gnn_pathplanning_b200 as gp
    from gnn_pathplanning_b200 import synthetic
    from oracle import eval_oracle
    N, W, B = 12, 16, 9
    rng = np.random.default_rng(5)
    parts = [synthetic.random_eval_cases(rng, 3, N, W, d) for d in (0.0, 0.1, 0.2)]
    T = max(p[3].shape[2] for p in parts) + 3                              # ragged: every chunk padded further
    target = np.zeros((B, N, T, 5), dtype=np.float32)
    target[..., 4] = 1.0
    for c, p in enumerate(parts):
        target[3 * c:3 * c + 3, :, :p[3].shape[2]] = p[3]
    starts = np.concatenate([p[1] for p in parts]); goals = np.concatenate([p[2] for p in parts])
    maps = np.concatenate([p[0] for p in parts]); makespan = np.concatenate([p[4] for p in parts])
    inp = np.stack([goals, starts], axis=1)
    want_s, want_e, want_t = [], [], []
    for b in range(B):
        sim = eval_oracle.EvalSimOracle(N).setup(starts[b], goals[b], maps[b], 1)
        want_t.append(list(sim.setup_targets(target[b])) + [1])
        want_s.append(sim.target_start); want_e.append(sim.target_end)
    assert len(set(makespan.tolist())) > 1
    for m in (maps, maps[0]):
        ro = gp.BatchedRollout(N).setup_cases(inp, torch.from_numpy(target).cuda(), makespan, m)
        assert np.array_equal(ro.target_start.cpu().numpy(), np.array(want_s))
        assert np.array_equal(ro.target_end.cpu().numpy(), np.array(want_e))
        assert np.array_equal(ro.targets.cpu().numpy(), np.array(want_t))
        assert np.array_equal(ro.maxstep.cpu().numpy(), makespan * 2)


def test_run_matches_evaluate(eval_trace):
    """run() shares evaluate()'s loop: the same final state on the same cases."""
    import gnn_pathplanning_b200 as gp
    from oracle import goal_policy
    policy = goal_policy.GoalSeekingPolicy().eval()
    g = eval_trace["a"]
    N = int(g["cfg"][0])
    ro = gp.BatchedRollout(N).setup_cases(g["input"], g["target"], g["makespan"], g["map"])
    ro.evaluate(policy)
    ro2 = gp.BatchedRollout(N).setup(g["input"][:, 1], g["input"][:, 0], g["map"], ro.maxstep)
    ro2.run(policy, poll_every=3)
    for k in ("pos", "reached", "start_step", "end_step", "choice_counter", "status", "active"):
        assert np.array_equal(getattr(ro2, k).cpu().numpy(), getattr(ro, k).cpu().numpy()), k
    assert not ro.active.any()
