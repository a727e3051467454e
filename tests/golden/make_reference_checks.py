"""Generates tests/golden/reference_checks.npz: what the UNMODIFIED reference computes for the cases of
tests/test_oracle_vs_reference.py (DecentralPlannerNet init / eval / train-mode forward, BatchLSIGF) and of
tests/test_sim_oracle_vs_reference.py (step-by-step rollouts of its simulator, utils/multirobotsim_dcenlocal.py).
Those tests compare the oracle with these vectors, so they run without the reference tree.

Needs a checkout of the reference (found as oracle/ref_shim.py finds it; GNNPP_REFERENCE_ROOT overrides):
    python tests/golden/make_reference_checks.py
"""
import hashlib
import os
import sys
import warnings

import numpy as np
import torch

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from oracle import planner_oracle as po  # noqa: E402
from oracle import ref_agent, ref_shim, ref_sim  # noqa: E402
from gnn_pathplanning_b200 import synthetic  # noqa: E402
import test_oracle_vs_reference as tov  # noqa: E402
import test_sim_oracle_vs_reference as tsv  # noqa: E402


def sha256(t):
    return hashlib.sha256(np.ascontiguousarray(t.numpy()).tobytes()).hexdigest()


def planner_checks(gml, dcp):
    out = {}
    for K in sorted({c[0] for c in tov.PLANNER_CASES}):
        torch.manual_seed(1337)
        sd = dcp.DecentralPlannerNet(ref_shim.Config(10, K)).state_dict()
        out["init%d_keys" % K] = np.array(list(sd.keys()))
        out["init%d_sha256" % K] = np.array([sha256(v) for v in sd.values()])
    for K, N, B in tov.PLANNER_CASES:
        torch.manual_seed(1337)
        m = dcp.DecentralPlannerNet(ref_shim.Config(N, K))
        sd = po.init_state_dict(K, seed=1337)
        po.randomize_bn_stats(sd)
        m.load_state_dict(sd)
        x, S = synthetic.make_batch(B, N, 20, seed=5)
        x, S = torch.from_numpy(x), torch.from_numpy(S)
        p = "planner_%d_%d_%d_" % (K, N, B)
        m.eval()
        m.addGSO(S.double())
        with torch.no_grad():
            out[p + "eval"] = torch.stack(m(x)).numpy()
        m.train()
        m.addGSO(S)
        out[p + "train"] = torch.stack(m(x)).detach().numpy()
        for k, v in m.state_dict().items():
            if "running" in k or "tracked" in k:
                out[p + "bn_" + k] = v.numpy()
    for i, (h, b, S, x) in enumerate(tov.graph_filter_inputs()):
        out["gf%d_inputs_sha256" % i] = np.array([sha256(t) for t in (h, b, S, x)])
        out["gf%d_y" % i] = gml.BatchLSIGF(h, S, x, b).numpy()
    return out


def sim_checks():
    out = {}
    with ref_agent.reference_env(dropin=False) as agmod:
        for N, W, density, makespan, T, seed in tsv.CASES:
            p = tsv.key(N, W, density, makespan, T, seed)
            case = ref_sim.make_case(np.random.default_rng(1000 + seed), N, W, density, makespan)
            out[p + "map"], out[p + "start"], out[p + "goal"] = case[:3]
            for k, v in ref_sim.reference_rollout(agmod, case, T, seed, N).items():
                out[p + k] = v
    return out


if __name__ == "__main__":
    out = planner_checks(*ref_shim.load()[:2])
    out.update(sim_checks())
    path = os.path.join(HERE, "reference_checks.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path))
