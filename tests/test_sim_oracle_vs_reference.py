"""CPU: oracle/sim_oracle.py against the reference's own multiRobotSim (unmodified), step by step on seeded cases -- FOV
tensors, float64 GSOs (incl. the step-0 radius growth), positions, actions, flags, goal / step bookkeeping.  The
reference's rollouts of these cases are stored in tests/golden/reference_checks.npz (tests/golden/
make_reference_checks.py).  `random.choice` is the round-robin contract on both sides (oracle/ref_sim.py)."""
import numpy as np
import pytest

from oracle import ref_sim

CASES = [  # N, W, obstacle density, makespan (-> maxstep = 2x, 3x for N >= 20), steps, seed
    (10, 20, 0.10, 14, 28, 1), (10, 20, 0.10, 6, 12, 2), (5, 8, 0.25, 10, 20, 3), (6, 6, 0.05, 8, 16, 4),
    (20, 28, 0.10, 6, 18, 5), (3, 12, 0.3, 9, 18, 6), (12, 9, 0.0, 5, 10, 7),
]
TRACE_KEYS = ("logits", "x", "S", "pos", "flags", "radius", "last_action", "reached", "maxstep", "start_step", "end_step",
              "choices")


def key(N, W, density, makespan, T, seed):
    return "sim_%d_%d_%g_%d_%d_%d_" % (N, W, density, makespan, T, seed)


@pytest.mark.parametrize("N,W,density,makespan,T,seed", CASES)
def test_oracle_matches_reference_simulator(golden, N, W, density, makespan, T, seed):
    g = golden("reference_checks.npz")
    p = key(N, W, density, makespan, T, seed)
    case = (g[p + "map"], g[p + "start"], g[p + "goal"], makespan)
    got = ref_sim.oracle_rollout(case, T, seed, N)
    assert sorted(got) == sorted(TRACE_KEYS)
    for k in TRACE_KEYS:
        assert np.array_equal(np.asarray(got[k]), g[p + k]), k
    assert (g[p + "last_action"] != 4).any()                     # agents really moved
