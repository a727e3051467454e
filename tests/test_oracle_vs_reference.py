"""CPU: the oracle against what the unmodified reference computed on the same inputs (DecentralPlannerNet init, eval and
train-mode forward, BatchLSIGF), stored in tests/golden/reference_checks.npz by tests/golden/make_reference_checks.py."""
import hashlib

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import planner_oracle as po

PLANNER_CASES = [(3, 10, 8), (2, 10, 1), (1, 4, 3), (3, 20, 2)]


def sha256(t):
    return hashlib.sha256(np.ascontiguousarray(t.numpy()).tobytes()).hexdigest()


def graph_filter_inputs():
    """(h, b, S, x) of each BatchLSIGF case."""
    g = torch.Generator().manual_seed(3)
    cases = []
    for (B, N, G, F, K) in [(5, 10, 128, 128, 3), (2, 33, 16, 8, 4)]:
        h = torch.rand(F, 1, K, G, generator=g) - 0.5
        b = torch.rand(F, 1, generator=g)
        S = torch.rand(B, 1, N, N, generator=g)
        x = torch.randn(B, G, N, generator=g)
        cases.append((h, b, S, x))
    return cases


@pytest.mark.parametrize("K,N,B", PLANNER_CASES)
def test_eval_and_train_match_reference(golden, K, N, B):
    g = golden("reference_checks.npz")
    sd = po.init_state_dict(K, seed=1337)
    # the reference's own initial state_dict under torch.manual_seed(1337), bit for bit
    assert sorted(sd) == sorted(str(k) for k in g["init%d_keys" % K])
    for k, h in zip(g["init%d_keys" % K], g["init%d_sha256" % K]):
        assert sha256(sd[str(k)]) == str(h), k
    po.randomize_bn_stats(sd)
    from gnn_pathplanning_b200 import synthetic
    x, S = synthetic.make_batch(B, N, 20, seed=5)
    x, S = torch.from_numpy(x), torch.from_numpy(S)
    p = "planner_%d_%d_%d_" % (K, N, B)
    with torch.no_grad():
        b = torch.stack(po.planner_forward(sd, S.double(), x))
    assert rel_err(b.numpy(), g[p + "eval"]) <= 1e-6
    bn = {k: v.clone() for k, v in sd.items() if "running" in k or "tracked" in k}
    out2 = po.planner_forward(sd, S, x, True, bn)
    assert rel_err(torch.stack(out2).numpy(), g[p + "train"]) <= 1e-6
    for k, v in bn.items():
        assert rel_err(v.double().numpy(), g[p + "bn_" + k].astype(np.float64)) <= 1e-6


def test_graph_filter_matches_reference(golden):
    g = golden("reference_checks.npz")
    for i, (h, b, S, x) in enumerate(graph_filter_inputs()):
        # the stored outputs belong to exactly these inputs
        assert [sha256(t) for t in (h, b, S, x)] == [str(s) for s in g["gf%d_inputs_sha256" % i]]
        assert rel_err(po.batch_lsigf(h, S, x, b).numpy(), g["gf%d_y" % i]) <= 1e-6
