"""Training batches built on the device from expert schedules, and the online expert's file formats (SURVEY.md
section 8 row f3).

The original project turns every expert solution into a .mat file (onlineExpert/DataTransformer_local_onlineExpert.py:
`obtainSchedule`, `computeAdjacencyMatrix`, `pathtransformer_RelativeCoordinate`) holding per step a 363-float field of
view per agent, a float64 GSO and one-hot targets, and its train loader calls `scipy.io.loadmat` once per sample
(dataloader/Dataloader_dcplocal_notTF_onlineExpert.py:142-157).  Every one of those tensors is a pure function of the
schedule's integer cells, the goals and the map, so `ExpertDataset` keeps only those on the device (about 60 MB for
21,000 cases of 10 agents, instead of about 9 GB of field-of-view tensors) and builds each batch in one kernel launch
(csrc/dataset.cu) at the moment it is needed.

The online expert (agents/decentralplannerlocal_OnlineExpert.py:289-310, DAgger-style data aggregation) closes the loop:
`ExpertDataset.test_cases` -> `BatchedRollout.setup_cases` / `evaluate` / `failure_cases` -> `write_failure_cases` ->
an external ECBS solver -> `read_ecbs_solutions` -> `ExpertDataset.add`.  `read_mat_cases` reads the reference's
existing training files.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import _lib

DELTA = np.array([[-1, 0], [0, -1], [1, 0], [0, 1], [0, 0]], dtype=np.int64)   # up, left, down, right, stop


def _check(rc: int) -> None:
    if rc == _lib.GPP_ERR_UNSUPPORTED:
        raise ValueError("libgnnpp_b200: " + _lib.load().gpp_last_error().decode("utf-8", "replace"))
    _lib.check(rc)


def _host(a) -> np.ndarray:
    return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def _integral(a, what: str) -> np.ndarray:
    a = _host(a)
    if a.dtype.kind == "f":
        if not np.isfinite(a).all() or (a != np.round(a)).any():
            raise ValueError("%s: cells must be whole numbers" % what)
    elif a.dtype.kind not in "iub":
        raise ValueError("%s: expected integer cells, got dtype %s" % (what, a.dtype))
    return np.ascontiguousarray(a, dtype=np.int64)


def _map01(maps) -> np.ndarray:
    return np.ascontiguousarray(maps != 0, dtype=np.uint8)       # .mat arrays arrive in Fortran order


def validate_cases(positions, goals, maps, num_agents=None, names=None):
    """Checks C cases on the host and returns them as (list of int64 [T_c,N,2], int64 goals [C,N,2], uint8 maps
    [C,W,W] or [W,W]).  Raises ValueError naming the offending cases (by `names`, else by index) for fewer than two
    agents or a number other than `num_agents`, an empty schedule, a non-square map, a cell or goal outside the map, and
    a move between consecutive rows (or from the last row to the goal) that is not one of up, left, down, right, stop
    -- where the reference's DataTransformer raises ValueError (`delta.index`)."""
    goals = _integral(goals, "goals")
    C = goals.shape[0] if goals.ndim == 3 else -1
    if goals.ndim != 3 or goals.shape[2] != 2:
        raise ValueError("goals: expected [C,N,2], got %s" % (goals.shape,))
    maps = _host(maps)
    if C == 0:
        return [], goals, _map01(maps)
    names = list(range(C)) if names is None else list(names)
    if isinstance(positions, (np.ndarray, torch.Tensor)) and _host(positions).ndim == 4:
        positions = list(_host(positions))
    positions = [_integral(p, "positions") for p in positions]
    if len(positions) != C:
        raise ValueError("positions: %d cases but %d goal sets" % (len(positions), C))
    N = goals.shape[1]
    if N < 2:
        raise ValueError("cases %s: %d agent(s); the communication graph needs at least 2" % (names, N))
    if num_agents is not None and N != num_agents:
        raise ValueError("cases %s: %d agents, the dataset has %d" % (names, N, num_agents))
    if maps.ndim not in (2, 3) or maps.shape[-1] != maps.shape[-2]:
        raise ValueError("maps: expected square [C,W,W] or [W,W] maps, got %s" % (maps.shape,))
    if maps.ndim == 3 and maps.shape[0] != C:
        raise ValueError("maps: %d maps for %d cases" % (maps.shape[0], C))
    W = maps.shape[-1]
    bad_shape = [names[c] for c, p in enumerate(positions) if p.ndim != 3 or p.shape[0] < 1 or p.shape[1:] != (N, 2)]
    if bad_shape:
        raise ValueError("cases %s: expected positions [T>=1,%d,2]" % (bad_shape, N))
    outside = [names[c] for c, p in enumerate(positions)
               if (p < 0).any() or (p >= W).any() or (goals[c] < 0).any() or (goals[c] >= W).any()]
    if outside:
        raise ValueError("cases %s: a cell or goal lies outside the %dx%d map" % (outside, W, W))
    bad_move = []
    for c, p in enumerate(positions):
        d = np.concatenate([p[1:], goals[c][None]]) - p
        if (np.abs(d).sum(-1) > 1).any():
            bad_move.append(names[c])
    if bad_move:
        raise ValueError("cases %s: a move is not one of up, left, down, right, stop" % bad_move)
    return positions, goals, _map01(maps)


class ExpertDataset:
    """Expert schedules on the device; every row (step) of every case is one training sample, as
    `search_target_files_withStep` lists them.  `batch(rows)` returns what the reference's train loader stacks:
    x [B,N,3,11,11] f32, S [B,N,N] f32 and target [B,N,5] int64 -- the arguments of `DecentralPlannerNet.addGSO` /
    `forward_logits` and `planner_loss`.  Host <-> device copies happen only in `add`, `test_cases` and in what the
    caller passes to `batch`."""

    def __init__(self, num_agents: int, comm_radius: float = 5.0, device="cuda"):
        self.N = int(num_agents)
        self.r0 = float(comm_radius)             # DataTransformer.communicationRadius
        self.device = torch.device(device)
        self.lib = _lib.load()
        dev = self.device
        self.pos = torch.empty(0, self.N, 2, device=dev, dtype=torch.int32)
        self.row_case = torch.empty(0, device=dev, dtype=torch.int32)
        self.case_first_row = torch.zeros(1, device=dev, dtype=torch.int32)
        self.goal = torch.empty(0, self.N, 2, device=dev, dtype=torch.int32)
        self.radius = torch.empty(0, device=dev, dtype=torch.float64)
        self.map = None
        self.map_shared = True
        self.W = None
        self._T = np.zeros(0, dtype=np.int64)       # rows per case (host: sizes only)

    def __len__(self) -> int:
        return int(self._T.sum())

    @property
    def num_cases(self) -> int:
        return int(self._T.size)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def add(self, positions, goals, maps):
        """Appends C cases: positions = per case the expert's cells [T_c,N,2] for steps 0 .. makespan (a list, or one
        [C,T,N,2] array), goals [C,N,2], maps [C,W,W] or one [W,W] map shared by the C cases.  Validates on the host
        (`validate_cases`), uploads, and computes the new cases' communication thresholds on the device.  Returns
        self."""
        positions, goals, maps = validate_cases(positions, goals, maps, self.N)
        C, W = goals.shape[0], maps.shape[-1]
        if C == 0:
            return self
        if self.W is not None and W != self.W:
            raise ValueError("maps: %dx%d, the dataset's maps are %dx%d" % (W, W, self.W, self.W))
        dev, C0, R0 = self.device, self.num_cases, len(self)
        T = np.array([p.shape[0] for p in positions], dtype=np.int64)
        first = R0 + np.concatenate([[0], np.cumsum(T)])
        self.pos = torch.cat([self.pos, torch.from_numpy(np.concatenate(positions).astype(np.int32)).to(dev)])
        self.row_case = torch.cat([self.row_case, torch.from_numpy(np.repeat(np.arange(C0, C0 + C), T).astype(np.int32)).to(dev)])
        self.case_first_row = torch.cat([self.case_first_row, torch.from_numpy(first[1:].astype(np.int32)).to(dev)])
        self.goal = torch.cat([self.goal, torch.from_numpy(goals.astype(np.int32)).to(dev)])
        new_map = torch.from_numpy(maps).to(dev).contiguous()
        if self.map is None:
            self.map, self.map_shared = new_map, maps.ndim == 2
        elif self.map_shared and maps.ndim == 2 and torch.equal(self.map, new_map):
            pass
        else:
            old = self.map.expand(C0, W, W) if self.map_shared else self.map
            self.map = torch.cat([old, new_map.expand(C, W, W) if maps.ndim == 2 else new_map]).contiguous()
            self.map_shared = False
        self.W = W
        self.radius = torch.cat([self.radius, torch.empty(C, device=dev, dtype=torch.float64)])
        self._T = np.concatenate([self._T, T])
        with torch.cuda.device(dev):
            _check(self.lib.gpp_dataset_prepare(
                self.pos.data_ptr(), self.case_first_row[C0:].data_ptr(), self.r0, self.radius[C0:].data_ptr(), C,
                self.N, self._stream()))
        return self

    def batch(self, rows, out=None):
        """Builds the samples `rows` (int64 indices into [0, len)) in one launch.  Returns (x, S, target); with
        `out` = such a triple of the right shapes, writes into it instead of allocating.  Host indices are range-checked
        (IndexError); a device index outside the range gives an all-zero sample."""
        rows = torch.as_tensor(rows)
        if not rows.is_cuda:                      # device indices are not read back: that would stall the stream
            r = rows.reshape(-1)
            if r.numel() and (int(r.min()) < 0 or int(r.max()) >= len(self)):
                raise IndexError("batch: row indices must lie in [0, %d)" % len(self))
        rows = rows.to(self.device, torch.int64).reshape(-1).contiguous()
        B, N, dev = rows.numel(), self.N, self.device
        if out is None:
            out = (torch.empty(B, N, 3, 11, 11, device=dev, dtype=torch.float32),
                   torch.empty(B, N, N, device=dev, dtype=torch.float32),
                   torch.empty(B, N, 5, device=dev, dtype=torch.int64))
        x, S, target = out
        assert tuple(x.shape) == (B, N, 3, 11, 11) and tuple(S.shape) == (B, N, N) and tuple(target.shape) == (B, N, 5)
        assert x.dtype == torch.float32 and S.dtype == torch.float32 and target.dtype == torch.int64
        assert x.is_contiguous() and S.is_contiguous() and target.is_contiguous()
        if self.map is None:
            if B:
                raise IndexError("batch: the dataset is empty")
            return x, S, target
        with torch.cuda.device(dev):
            _check(self.lib.gpp_dataset_batch(
                self.pos.data_ptr(), self.row_case.data_ptr(), self.case_first_row.data_ptr(), self.goal.data_ptr(),
                self.map.data_ptr(), int(self.map_shared), self.radius.data_ptr(), rows.data_ptr(), x.data_ptr(),
                S.data_ptr(), target.data_ptr(), B, N, self.W, len(self), self._stream()))
        return x, S, target

    def batches(self, batch_size: int, generator=None):
        """One epoch in a random order drawn on the device (torch.randperm; `generator` must live on the dataset's
        device), ending with a partial batch, as DataLoader(shuffle=True) does."""
        order = torch.randperm(len(self), device=self.device, generator=generator)
        for i in range(0, len(self), int(batch_size)):
            yield self.batch(order[i:i + int(batch_size)])

    def test_cases(self, case_ids=None):
        """The test loader's view of the cases (`load_data_during_training`): (input [C,2,N,2] = (goal, start),
        target [C,N,T,5] int64 one-hot expert actions, cases shorter than the longest padded with 'stop', makespan [C]
        = T_c, maps [C,W,W] or the shared [W,W]) -- the arguments of `BatchedRollout.setup_cases`."""
        dev = self.device
        ids = np.arange(self.num_cases) if case_ids is None else np.asarray(case_ids, dtype=np.int64).reshape(-1)
        if ids.size and (ids.min() < 0 or ids.max() >= self.num_cases):
            raise IndexError("test_cases: case ids must lie in [0, %d)" % self.num_cases)
        Tc = self._T[ids]
        Tmax = int(Tc.max()) if ids.size else 1
        ids_d = torch.from_numpy(ids).to(dev)
        first = self.case_first_row[ids_d].long()
        Tc_d = torch.from_numpy(Tc).to(dev)
        t = torch.arange(Tmax, device=dev)
        rows = first[:, None] + torch.minimum(t[None], Tc_d[:, None] - 1)                   # [C,T]
        last = (rows + 1 == self.case_first_row[ids_d + 1].long()[:, None])
        p = self.pos[rows].long()                                                           # [C,T,N,2]
        goal = self.goal[ids_d].long()
        nxt = torch.where(last[..., None, None], goal[:, None], self.pos[(rows + 1).clamp(max=max(len(self) - 1, 0))].long())
        d = nxt - p
        key = torch.full(d.shape[:-1], 4, device=dev, dtype=torch.long)
        for k, (dx, dy) in enumerate(DELTA[:4].tolist()):
            key[(d[..., 0] == dx) & (d[..., 1] == dy)] = k
        key[t[None].expand(len(ids), Tmax) >= Tc_d[:, None]] = 4                             # padding: stop
        target = torch.nn.functional.one_hot(key, 5).permute(0, 2, 1, 3).contiguous()        # [C,N,T,5]
        inp = torch.stack([goal, self.pos[first].long()], dim=1)                            # [C,2,N,2]
        maps = self.map if self.map_shared else self.map[ids_d]
        return inp, target, torch.from_numpy(Tc.copy()), maps


# ---------------------------------------------------------------------------------------------------------------------
# the online expert's files
# ---------------------------------------------------------------------------------------------------------------------
def failure_case_yaml(map_hw, cells, goals) -> str:
    """The solver input multiRobotSim.save_failure_cases writes (utils/multirobotsim_dcenlocal_onlineExpert.py:705-730):
    the map's dimensions, its obstacles in row-major order and every agent's final cell as its start."""
    m = _host(map_hw)
    out = ["map:\n", "    dimensions: [%d, %d]\n" % m.shape, "    obstacles:\n"]
    out += ["    - [%d, %d]\n" % (x, y) for x, y in np.argwhere(m != 0).tolist()]
    out.append("agents:\n")
    for i, (c, g) in enumerate(zip(_host(cells).tolist(), _host(goals).tolist())):
        out.append("  - name: agent%d\n    start: [%d, %d]\n    goal: [%d, %d]\n" % (i, c[0], c[1], g[0], g[1]))
    return "".join(out)


def write_failure_cases(directory, case_ids, maps, cells, goals):
    """Writes `failureCases_ID{id:05d}.yaml` for each failed case into the existing `directory`: case_ids [F], maps
    [F,W,W] or one shared [W,W], cells [F,N,2] (BatchedRollout.failure_cases), goals [F,N,2].  Deletes nothing (the
    reference empties its folder first; that is the caller's decision).  Returns the paths written."""
    if not os.path.isdir(directory):
        raise FileNotFoundError("write_failure_cases: %s is not a directory" % directory)
    ids, maps, cells, goals = _host(case_ids).reshape(-1), _host(maps), _host(cells), _host(goals)
    paths = []
    for f, cid in enumerate(ids.tolist()):
        path = os.path.join(directory, "failureCases_ID{:05d}.yaml".format(int(cid)))
        with open(path, "w") as fh:
            fh.write(failure_case_yaml(maps if maps.ndim == 2 else maps[f], cells[f], goals[f]))
        paths.append(path)
    return paths


def _yaml_files(directory):
    out = []
    for root, _, names in sorted(os.walk(directory)):
        out += [os.path.join(root, n) for n in names if n.endswith(".yaml")]
    return out


def read_ecbs_solutions(input_dir, solution_dir):
    """Reads the solver's outputs in `solution_dir` and their inputs in `input_dir`, paired as the reference's
    DataTransformer.load_ExpertSolution does (a solution `..._ID<id>.yaml` goes with `<prefix>ID<id>.yaml`, the prefix
    taken from the first input file), in sorted solution order.  Each case has T = statistics.makespan + 1 rows: an
    agent's cell is its planned cell while the plan lasts, then its goal.  Returns (positions, goals, maps) for
    `ExpertDataset.add`, validated; raises ValueError naming the solution files that the reference would reject or
    that a solver never writes (a plan longer than makespan + 1 steps)."""
    import yaml
    sols = sorted(_yaml_files(solution_dir))
    inputs = _yaml_files(input_dir)
    if not sols:
        return [], np.zeros((0, 0, 2), dtype=np.int64), np.zeros((0, 0, 0), dtype=np.uint8)
    if not inputs:
        raise ValueError("read_ecbs_solutions: no input files in %s" % input_dir)
    prefix = os.path.basename(inputs[0]).split("ID")[0]
    positions, goals, maps, too_long = [], [], [], []
    for path in sols:
        cid = os.path.basename(path).split("_ID")[-1].split(".yaml")[0]
        with open(os.path.join(input_dir, prefix + "ID{}.yaml".format(cid))) as fh:
            cfg = yaml.safe_load(fh)
        with open(path) as fh:
            sol = yaml.safe_load(fh)
        W, H = (int(v) for v in cfg["map"]["dimensions"])
        m = np.zeros((W, H), dtype=np.uint8)
        for x, y in cfg["map"]["obstacles"] or []:
            m[int(x), int(y)] = 1
        g = np.array([a["goal"] for a in cfg["agents"]], dtype=np.int64)
        T = int(sol["statistics"]["makespan"]) + 1
        p = np.empty((T, len(g), 2), dtype=np.int64)
        for i in range(len(g)):
            plan = [(int(s["x"]), int(s["y"])) for s in sol["schedule"]["agent%d" % i]]
            if len(plan) > T:
                too_long.append(path)
            for t in range(T):
                p[t, i] = plan[t] if t < len(plan) else g[i]
        positions.append(p)
        goals.append(g)
        maps.append(m)
    if too_long:
        raise ValueError("solutions %s: a plan is longer than makespan + 1 steps" % sorted(set(too_long)))
    if len({g.shape for g in goals}) != 1 or len({m.shape for m in maps}) != 1:
        raise ValueError("solutions %s: the cases differ in their number of agents or map size" % sols)
    return validate_cases(positions, np.stack(goals), np.stack(maps), names=sols)


def read_mat_cases(paths):
    """Reads training-set .mat files the reference's DataTransformer wrote: only `map`, `goal` and `inputState`
    [T,N,2] (everything else is regenerated on the device).  Returns (positions, goals, maps) for
    `ExpertDataset.add`, validated; raises ValueError naming test-format files (a 2-D inputState) and invalid cases."""
    import scipy.io
    paths = list(paths)
    positions, goals, maps, test_format = [], [], [], []
    for path in paths:
        d = scipy.io.loadmat(path, variable_names=("map", "goal", "inputState"))
        if d["inputState"].ndim != 3:
            test_format.append(path)
            continue
        positions.append(d["inputState"])
        goals.append(d["goal"])
        maps.append(d["map"])
    if test_format:
        raise ValueError("files %s: a 2-D inputState (test-set format) has no schedule" % test_format)
    if not paths:
        return [], np.zeros((0, 0, 2), dtype=np.int64), np.zeros((0, 0, 0), dtype=np.uint8)
    if len({np.shape(g) for g in goals}) != 1 or len({np.shape(m) for m in maps}) != 1:
        raise ValueError("files %s: the cases differ in their number of agents or map size" % paths)
    return validate_cases(positions, np.stack(goals), np.stack(maps), names=paths)
