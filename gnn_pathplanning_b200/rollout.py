"""GPU-resident batched rollouts (SURVEY.md section 8 rows f1 / f2).

The reference rolls ONE episode at a time on the host (agents/decentralplannerlocal.py:535-648): every step it rebuilds
the field-of-view tensor and the graph shift operator with numpy / scipy (`multiRobotSim.getCurrentState`, `.getGSO`),
copies them to the device, runs the model, pulls N tiny argmax results back and moves the agents in Python dicts
(`multiRobotSim.move`).  `BatchedRollout` keeps B episodes on the device and advances them in lock-step: positions never
leave HBM, the per-step work is four library launches (inputs, planner forward, move, track) and there is no per-step
host <-> device copy -- only the `done` flags are read back every `poll_every` steps.

Mirrors the simulator's interface where it has one: `setup`, `getCurrentState`, `getGSO`, `move`, `getMaxstep`,
`count_numAgents_ReachGoal`, plus `run(model)` for the whole loop.  `setup_cases` + `evaluate(model)` replace the
reference's test() loop (agents/decentralplannerlocal.py:484-648): per-case success / makespan / flowtime records,
summarised by `evaluation.summarize`; `failure_cases()` lists the cases the online expert would re-plan.  The only
behavioural difference is the documented tie-break contract of gpp_rollout_move (round-robin instead of
`random.choice`).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib


class BatchedRollout:
    def __init__(self, num_agents: int, comm_radius: float = 6.0, device="cuda"):
        self.N = int(num_agents)
        self.commR = float(comm_radius)               # main.py:70 `--commR`, multirobotsim_dcenlocal.py:242
        self.device = torch.device(device)
        self.lib = _lib.load()
        self.B = 0

    # ------------------------------------------------------------------ setup (multirobotsim_dcenlocal.py:54-143)
    def setup(self, start, goal, maps, maxstep):
        """start, goal: [B,N,2] integer cells; maps: [B,W,W] or [W,W] {0,1}; maxstep: int or [B]
        (the reference: makespanTarget * rate_maxstep, :76-81)."""
        dev = self.device
        self.pos = torch.as_tensor(start).to(dev, torch.int32).contiguous().clone()
        self.goal = torch.as_tensor(goal).to(dev, torch.int32).contiguous()
        self.B = self.pos.shape[0]
        assert tuple(self.pos.shape) == (self.B, self.N, 2) and tuple(self.goal.shape) == (self.B, self.N, 2)
        maps = torch.as_tensor(maps)
        self.map_shared = maps.dim() == 2
        self.map = maps.to(dev, torch.uint8).contiguous()
        self.W = int(self.map.shape[-1])
        assert self.map.shape[-2] == self.W and (self.map_shared or self.map.shape[0] == self.B)
        ms = torch.as_tensor(maxstep)
        self.maxstep = (ms.expand(self.B) if ms.dim() == 0 else ms).to(dev, torch.int32).contiguous()
        B, N = self.B, self.N
        self.radius = torch.full((B,), self.commR, device=dev, dtype=torch.float64)
        self.reached = torch.zeros(B, N, device=dev, dtype=torch.int32)
        self.start_step = torch.full((B, N), -1, device=dev, dtype=torch.int32)
        self.end_step = torch.full((B, N), -1, device=dev, dtype=torch.int32)
        self.last_action = torch.full((B, N), 4, device=dev, dtype=torch.int32)
        self.choice_counter = torch.zeros(B, device=dev, dtype=torch.int32)
        self.flags = torch.zeros(B, 3, device=dev, dtype=torch.int32)
        self.active = torch.ones(B, device=dev, dtype=torch.int32)
        self.connected = torch.zeros(B, device=dev, dtype=torch.int32)
        # {allReachGoal of the last move, collision happened in the loop, collision predicted in the loop, last step}
        self.status = torch.zeros(B, 4, device=dev, dtype=torch.int32)
        self.x = torch.empty(B, N, 3, 11, 11, device=dev, dtype=torch.float32)
        self.S = torch.empty(B, N, N, device=dev, dtype=torch.float64)
        self.step = 0
        self.targets = None
        return self

    def setup_cases(self, input, target, makespan, maps, rate_maxstep: int = 2):
        """B test cases in the test loader's formats, batched (multiRobotSim.setup, multirobotsim_dcenlocal.py:54-143):
        input [B,2,N,2] = (goal, start); target [B,N,T,5] one-hot expert actions (cases with fewer steps padded with
        'stop' rows); makespan [B]; maps [B,W,W] or [W,W].  maxstep = int(makespan) * rate_maxstep, with rate 3 for
        N >= 20 (:76-81).  Replays the expert's actions on the device (getPathTarget, :159-229) for evaluate().

        Raises ValueError, naming the cases, where the reference's test loop would crash: an agent starts on its goal
        (TypeError at :708), the expert's actions leave an agent off its goal (makespanTarget = 0, ZeroDivisionError
        at utils/metrics.py:110), or makespan < 1.  These checks run on the host before anything is launched."""
        inp = _host(input).astype(np.int64)
        tgt = _host(target)
        mk = _host(makespan).reshape(-1).astype(np.int32)
        B = inp.shape[0]
        if inp.shape != (B, 2, self.N, 2) or tgt.ndim != 4 or tgt.shape[:2] != (B, self.N) or tgt.shape[3] != 5 \
                or mk.shape != (B,):
            raise ValueError("setup_cases: expected input [B,2,%d,2], target [B,%d,T,5], makespan [B]; got %s, %s, %s"
                             % (self.N, self.N, inp.shape, tgt.shape, mk.shape))
        goal, start = inp[:, 0], inp[:, 1]
        bad = np.nonzero((start == goal).all(-1).any(-1))[0]
        if bad.size:
            raise ValueError("setup_cases: an agent starts on its goal in cases %s" % bad.tolist())
        bad = np.nonzero(mk < 1)[0]
        if bad.size:
            raise ValueError("setup_cases: makespan < 1 in cases %s" % bad.tolist())
        # the expert's path is start + the running sum of its moves (getPathTarget ignores map and other agents)
        path = start[:, :, None, :] + np.cumsum(_DELTA[tgt.argmax(-1)], axis=2)
        bad = np.nonzero(~(path == goal[:, :, None, :]).all(-1).any(-1).all(-1))[0]
        if bad.size:
            raise ValueError("setup_cases: the expert's actions leave an agent off its goal in cases %s" % bad.tolist())
        rate = 3 if self.N >= 20 else int(rate_maxstep)
        self.setup(start, goal, maps, torch.from_numpy(mk.astype(np.int64) * rate))
        dev, N, T = self.device, self.N, tgt.shape[2]
        target_dev = torch.as_tensor(target).to(dev, torch.float32).contiguous()
        self.target_start = torch.empty(B, N, device=dev, dtype=torch.int32)
        self.target_end = torch.empty(B, N, device=dev, dtype=torch.int32)
        self.targets = torch.empty(B, 3, device=dev, dtype=torch.int32)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.gpp_rollout_targets(
                target_dev.data_ptr(), self.pos.data_ptr(), self.goal.data_ptr(), self.target_start.data_ptr(),
                self.target_end.data_ptr(), self.targets.data_ptr(), B, N, T, self._stream()))
        return self

    def getMaxstep(self):
        return self.maxstep

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    # ------------------------------------------------------------------ inputs of one step (f2)
    def build_inputs(self, step: int):
        """getCurrentState + getGSO of every episode in one launch: returns (x [B,N,3,11,11] f32, S [B,N,N] f64)."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.gpp_rollout_build_inputs(
                self.pos.data_ptr(), self.goal.data_ptr(), self.map.data_ptr(), int(self.map_shared),
                self.radius.data_ptr(), int(step == 0), self.x.data_ptr(), self.S.data_ptr(), 1,
                self.connected.data_ptr(), self.B, self.N, self.W, self._stream()))
        return self.x, self.S

    def getCurrentState(self):
        return self.x

    def getGSO(self, step: int):
        return self.build_inputs(step)[1]

    # ------------------------------------------------------------------ move (f1)
    def move(self, logits, currentstep: int):
        """logits: the planner's [N,B,5] tensor (or its list of N [B,5] views).  Returns the [B,3] int32 device tensor
        {allReachGoal before the move, check_moveCollision, check_predictCollsion} (multirobotsim_dcenlocal.py:723)."""
        if isinstance(logits, (list, tuple)):
            base = getattr(logits[0], "_base", None)
            logits = base if base is not None and base.dim() == 3 else torch.stack(list(logits))
        logits = logits.contiguous()
        assert tuple(logits.shape) == (self.N, self.B, 5) and logits.dtype == torch.float32
        with torch.cuda.device(self.device):
            _lib.check(self.lib.gpp_rollout_move(
                logits.data_ptr(), self.pos.data_ptr(), self.goal.data_ptr(), self.map.data_ptr(), int(self.map_shared),
                self.maxstep.data_ptr(), self.active.data_ptr(), self.reached.data_ptr(), self.start_step.data_ptr(),
                self.end_step.data_ptr(), self.last_action.data_ptr(), self.choice_counter.data_ptr(),
                self.flags.data_ptr(), int(currentstep), self.B, self.N, self.W, self._stream()))
        return self.flags

    def count_numAgents_ReachGoal(self):
        return self.reached.sum(dim=1)

    # ------------------------------------------------------------------ the rollout loop (agents/...local.py:560-592)
    def track(self, flags, currentstep: int):
        """The loop body after the move (agents/decentralplannerlocal.py:593-606) for every episode that was active
        for it: ORs the move's collision flags into `status`, records its allReachGoal and step, and retires the
        episode (active = 0) once all agents had reached their goals or maxstep is reached."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.gpp_rollout_track(
                flags.data_ptr(), self.active.data_ptr(), self.status.data_ptr(), self.maxstep.data_ptr(),
                int(currentstep), self.B, self._stream()))

    def run(self, model, max_steps: int = None, poll_every: int = 8):
        """Advances all episodes until every one has finished (all agents at their goals, or its maxstep reached).
        Per step: build_inputs -> model.addGSO + forward_logits -> move -> track, all on the device; an episode stops
        being moved once the reference's loop would have left it (:606-613).  Returns the number of steps taken."""
        assert not model.training
        limit = int(self.maxstep.max().item()) if max_steps is None else int(max_steps)
        with torch.no_grad():
            for step in range(limit):
                x, S = self.build_inputs(step)
                model.addGSO(S)
                logits = model.forward_logits(x)
                self.track(self.move(logits, step + 1), step + 1)
                self.step = step + 1
                if (step + 1) % poll_every == 0 and not bool(self.active.any().item()):
                    break
        return self.step

    # ------------------------------------------------------------------ the test loop (agents/...local.py:484-648)
    def evaluate(self, model, poll_every: int = 8):
        """Runs the cases given to setup_cases to the end and returns their per-case records (CaseRecords): what
        mutliAgent_ActionPolicy hands to MonitoringMultiAgentPerformance.update for each case.  The only host copies
        are the `active.any()` poll every `poll_every` steps and the records at the end."""
        from .evaluation import CaseRecords
        assert self.targets is not None, "evaluate() needs the cases' expert targets: call setup_cases() first"
        self.run(model, poll_every=poll_every)
        record = torch.empty(self.B, 10, device=self.device, dtype=torch.int32)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.gpp_rollout_evaluate_finish(
                self.status.data_ptr(), self.targets.data_ptr(), self.maxstep.data_ptr(), self.reached.data_ptr(),
                self.start_step.data_ptr(), self.end_step.data_ptr(), record.data_ptr(), self.B, self.N,
                self._stream()))
        return CaseRecords.from_record(record.cpu().numpy(), self.N)

    def failure_cases(self):
        """After evaluate(): the cases whose loop ended at maxstep (currentStep >= maxstep, a success on the last step
        included) -- the ones the reference's online expert hands to its solver (agents/
        decentralplannerlocal_OnlineExpert.py:536-539).  Returns (case indices [F] int64, the agents' final cells
        [F,N,2] int64) on the host, for `dataset.write_failure_cases`."""
        assert self.targets is not None and self.step > 0, "failure_cases() needs a finished evaluate()"
        ids = torch.nonzero(self.status[:, 3] >= self.maxstep).reshape(-1)
        return ids.cpu().numpy(), self.pos[ids].long().cpu().numpy()


_DELTA = np.array([[-1, 0], [0, -1], [1, 0], [0, 1], [0, 0]], dtype=np.int64)    # multirobotsim_dcenlocal.py:21-25


def _host(a) -> np.ndarray:
    return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
