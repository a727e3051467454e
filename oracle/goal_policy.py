"""TEST INFRASTRUCTURE -- a small deterministic goal-seeking policy over the field-of-view tensor, used to evaluate the
test loop (tests/golden/make_eval_trace.py through the reference's agent, tests/test_gpu_evaluate.py through
BatchedRollout.evaluate).

Every logit is a small integer held in float32, so the arithmetic is exact on any device and the first-maximum
action (LogSoftmax + argmax in the reference) is the same everywhere.  The policy heads for its goal (or the goal's
projection on the window rim) and steps around an obstacle or agent in its way (sideways beats staying, staying beats
bumping).  Greedy and blind to what other agents do next, it gives a mix of optimal and delayed successes, shielded
collisions and deadlocks that time out."""
from __future__ import annotations

import numpy as np
import torch

from oracle.sim_oracle import CENTER, DELTA, STOP


class GoalSeekingPolicy(torch.nn.Module):
    """Duck-types the planner's interface: addGSO(S), forward(x) -> N tensors [B,5], forward_logits(x) -> [N,B,5]."""

    def __init__(self, obstacle_penalty: float = 6.0, agent_penalty: float = 6.0, stop_penalty: float = 3.0):
        super().__init__()
        self.obstacle_penalty = float(obstacle_penalty)
        self.agent_penalty = float(agent_penalty)
        self.stop_penalty = float(stop_penalty)

    def addGSO(self, S):
        self.S = S

    def forward_logits(self, x):
        """x [B,N,3,11,11] -> logits [N,B,5]: -2 * (distance to the goal after the move) - penalties for moving into
        an obstacle or an agent and for staying off the goal."""
        u = torch.arange(x.shape[-1], dtype=x.dtype, device=x.device)
        goal = x[:, :, 1]
        gu = (goal.sum(-1) * u).sum(-1)
        gv = (goal.sum(-2) * u).sum(-1)
        out = []
        for k, (dx, dy) in enumerate(DELTA):
            nu, nv = CENTER + dx, CENTER + dy
            s = -2.0 * ((gu - nu).abs() + (gv - nv).abs())
            if k != STOP:
                s = s - self.obstacle_penalty * x[:, :, 0, nu, nv] - self.agent_penalty * x[:, :, 2, nu, nv]
            else:
                s = s - self.stop_penalty * (s < 0).to(x.dtype)           # staying put off the goal
            out.append(s)
        return torch.stack(out, -1).permute(1, 0, 2).contiguous()

    def forward(self, x):
        return list(self.forward_logits(x).unbind(0))

    def numpy_policy(self):
        """The same policy as oracle/eval_oracle.evaluate_case's policy(x [N,3,11,11], S, step) -> [N,5]."""
        def policy(x, S, step):
            with torch.no_grad():
                return self.forward_logits(torch.from_numpy(np.asarray(x))[None])[:, 0].numpy()
        return policy
