"""Synthetic rollout-like inputs for the planner hot path (SURVEY.md section 8d).

Vectorised numpy builders for the two tensors the reference hands to
DecentralPlannerNet every step:

  * the per-agent field-of-view tensor  x [N,3,11,11] f32 in {0,1}
    (map / goal-or-projected-goal / agents-in-view), same semantics as
    AgentState.toInputTensor (/root/reference/dataloader/statetransformer.py:82-130,
    projected goal :47-66), and
  * the graph shift operator  S = D^-1/2 A D^-1/2,  A = (pairwise distance < r)
    with zero diagonal and the zero-degree guard
    (/root/reference/utils/multirobotsim_dcenlocal.py:338-348).

These are input PRODUCERS (SURVEY.md section 8 rows a11/f1/f2), written from the
behaviour of the reference, pinned against it by tests/golden (the reference
itself is not available on the GPU box).  They run on the host; nothing here is
timed as part of the hot path.
"""
from __future__ import annotations

import numpy as np

FOV = 9                 # statetransformer.py:11
FOV_HALF = FOV // 2     # :12
BORDER = 1              # :13
WIN = FOV + 2 * BORDER  # 11 (:14-15)
CENTER = WIN // 2       # 5  (:16,20-21)


def fov_tensor(map_hw: np.ndarray, goals: np.ndarray, states: np.ndarray) -> np.ndarray:
    """map_hw [W,H] {0,1} obstacles; goals/states [N,2] integer (x,y) cells.
    Returns float32 [N,3,11,11]: channel 0 = obstacle window (outside the map counts
    as obstacle), 1 = goal (inside the 9x9 view, else projected onto the 11x11 rim),
    2 = all agents inside the 9x9 view; each 9x9 window sits inside a zero border."""
    map_hw = np.asarray(map_hw)
    N = states.shape[0]
    pad_map = np.pad(map_hw, FOV_HALF, constant_values=1)
    occ = np.zeros_like(map_hw, dtype=np.int64)
    occ[states[:, 0].astype(int), states[:, 1].astype(int)] = 1
    pad_occ = np.pad(occ, FOV_HALF, constant_values=0)
    out = np.zeros((N, 3, WIN, WIN), dtype=np.float32)
    for i in range(N):
        cx, cy = int(states[i, 0]), int(states[i, 1])
        gx, gy = int(goals[i, 0]), int(goals[i, 1])
        out[i, 0, BORDER:-BORDER, BORDER:-BORDER] = pad_map[cx:cx + FOV, cy:cy + FOV]
        out[i, 2, BORDER:-BORDER, BORDER:-BORDER] = pad_occ[cx:cx + FOV, cy:cy + FOV]
        dx, dy = gx - cx, gy - cy
        if abs(dx) <= FOV_HALF and abs(dy) <= FOV_HALF:
            out[i, 1, CENTER + dx, CENTER + dy] = 1.0
        else:
            # goal outside the view: project along the bearing onto the window rim
            ang = np.arctan2(float(dy), float(dx))
            if (np.pi / 4 <= ang <= 3 * np.pi / 4) or (-3 * np.pi / 4 <= ang <= -np.pi / 4):
                py = int(CENTER * (np.sign(dy) + 1))
                px = int(CENTER + np.round(CENTER * float(dx) / abs(float(dy))))
            else:
                px = int(CENTER * (np.sign(dx) + 1))
                py = int(CENTER + np.round(CENTER * float(dy) / abs(float(dx))))
            out[i, 1, px, py] = 1.0
    return out


def gso_from_positions(pos: np.ndarray, comm_radius: float, zero_tol: float = 1e-9) -> np.ndarray:
    """pos [N,2] -> float64 [N,N] normalised adjacency D^-1/2 A D^-1/2 with
    A[i,j] = (||p_i - p_j|| < r), A[i,i] = 0; zero-degree nodes keep an all-zero row."""
    p = np.asarray(pos, dtype=np.float64)
    d = np.sqrt(((p[:, None, :] - p[None, :, :]) ** 2).sum(-1))
    A = (d < comm_radius).astype(np.float64)
    np.fill_diagonal(A, 0.0)
    deg = A.sum(axis=1)
    iso = np.abs(deg) < zero_tol
    deg[iso] = 1.0
    inv_sqrt = np.sqrt(1.0 / deg)
    inv_sqrt[iso] = 0.0
    return (inv_sqrt[:, None] * A) * inv_sqrt[None, :]


def random_episode(rng: np.random.Generator, num_agents: int, map_w: int, density: float = 0.1):
    """One random case: W x W map with `density` obstacles, N distinct free start
    cells and N distinct free goal cells (uniform)."""
    while True:
        m = (rng.random((map_w, map_w)) < density).astype(np.int64)
        free = np.argwhere(m == 0)
        if free.shape[0] >= 2 * num_agents:
            break
    starts = free[rng.choice(free.shape[0], num_agents, replace=False)]
    goals = free[rng.choice(free.shape[0], num_agents, replace=False)]
    return m, starts, goals


def make_batch(batch: int, num_agents: int, map_w: int, seed: int = 1337,
               comm_radius: float = 6.0, density: float = 0.1, gso_dtype=np.float32):
    """B independent episodes -> (x [B,N,3,11,11] f32, S [B,N,N] gso_dtype)."""
    rng = np.random.default_rng(seed)
    x = np.empty((batch, num_agents, 3, WIN, WIN), dtype=np.float32)
    S = np.empty((batch, num_agents, num_agents), dtype=np.float64)
    for b in range(batch):
        m, starts, goals = random_episode(rng, num_agents, map_w, density)
        x[b] = fov_tensor(m, goals, starts)
        S[b] = gso_from_positions(starts, comm_radius)
    return x, S.astype(gso_dtype)


_MOVES = ((-1, 0), (0, -1), (1, 0), (0, 1))   # up, left, down, right (multirobotsim_dcenlocal.py:21-25); 4 = stop


def _bfs_distance(map_hw: np.ndarray, goal) -> np.ndarray:
    """Steps from every free cell to `goal` over free cells (4-connected); -1 = unreachable."""
    W = map_hw.shape[0]
    dist = np.full(map_hw.shape, -1, dtype=np.int64)
    dist[goal[0], goal[1]] = 0
    frontier = [(int(goal[0]), int(goal[1]))]
    while frontier:
        nxt = []
        for x, y in frontier:
            for dx, dy in _MOVES:
                u, v = x + dx, y + dy
                if 0 <= u < W and 0 <= v < W and map_hw[u, v] == 0 and dist[u, v] < 0:
                    dist[u, v] = dist[x, y] + 1
                    nxt.append((u, v))
        frontier = nxt
    return dist


def random_eval_cases(rng: np.random.Generator, batch: int, num_agents: int, map_w: int, density: float = 0.1):
    """B test cases in the test loader's content: maps [B,W,W] int64, starts / goals [B,N,2] int64 with no agent
    starting on its goal, one-hot expert actions [B,N,T,5] float32 and makespan [B] int64.  The expert is each agent's
    own shortest path (breadth-first search; the first shortest move in action order), ignoring the other agents --
    enough for the target makespan / flowtime the test loop replays.  makespan = the longest of a case's paths;
    T = the longest over the batch, shorter paths are padded with 'stop'."""
    maps, starts, goals, paths = [], [], [], []
    while len(maps) < batch:
        m, st, gl = random_episode(rng, num_agents, map_w, density)
        if (st == gl).all(axis=1).any():
            continue
        acts = []
        for s, g in zip(st, gl):
            dist = _bfs_distance(m, g)
            if dist[s[0], s[1]] < 0:
                break
            x, y, a = int(s[0]), int(s[1]), []
            while dist[x, y] > 0:
                k = next(k for k, (dx, dy) in enumerate(_MOVES)
                         if 0 <= x + dx < map_w and 0 <= y + dy < map_w and dist[x + dx, y + dy] == dist[x, y] - 1)
                a.append(k)
                x, y = x + _MOVES[k][0], y + _MOVES[k][1]
            acts.append(a)
        if len(acts) < num_agents:
            continue                                  # some goal unreachable: draw the case again
        maps.append(m); starts.append(st); goals.append(gl); paths.append(acts)
    makespan = np.array([max(len(a) for a in p) for p in paths], dtype=np.int64)
    T = int(makespan.max())
    target = np.zeros((batch, num_agents, T, 5), dtype=np.float32)
    target[..., 4] = 1.0
    for b, p in enumerate(paths):
        for i, a in enumerate(p):
            target[b, i, np.arange(len(a)), 4] = 0.0
            target[b, i, np.arange(len(a)), a] = 1.0
    return np.stack(maps), np.stack(starts), np.stack(goals), target, makespan


def random_targets(batch: int, num_agents: int, seed: int = 1337) -> np.ndarray:
    """Uniform random one-hot action targets [B,N,5] (int64), the training label
    format of Dataloader_dcplocal_notTF_onlineExpert.py:142-157."""
    rng = np.random.default_rng(seed + 1)
    idx = rng.integers(0, 5, size=(batch, num_agents))
    return np.eye(5, dtype=np.int64)[idx]


def random_schedules(rng: np.random.Generator, cases: int, num_agents: int, map_w: int, density: float = 0.1,
                     max_len: int = 31, p_wait: float = 0.2):
    """Expert-schedule-like cases for `ExpertDataset.add`: per case [T_c,N,2] int64 cells, goals [C,N,2] int64 and maps
    [C,W,W] int64.  Each agent walks from a distinct free cell for 1 .. max_len - 1 moves (random free neighbour, or a
    wait with probability p_wait or when boxed in) and then stays; its goal is its last cell and T_c is the case's
    longest walk + 1 -- the rows a solver's schedule turns into.  Agents may share cells: the transformer never checks."""
    C, N, W = cases, num_agents, map_w
    maps = (rng.random((C, W, W)) < density).astype(np.int64)
    pos = np.empty((C, N, 2), dtype=np.int64)
    for c in range(C):
        free = np.flatnonzero(maps[c] == 0)
        cell = rng.choice(free, N, replace=False)
        pos[c, :, 0], pos[c, :, 1] = cell // W, cell % W
    length = rng.integers(1, max_len, size=(C, N))                 # moves per agent
    traj = [pos.copy()]
    ci = np.arange(C)[:, None]
    for t in range(max_len - 1):
        k = rng.integers(0, 4, size=(C, N))
        nxt = pos + np.asarray(_MOVES)[k]
        inside = ((nxt >= 0) & (nxt < W)).all(-1)
        ok = inside & (maps[ci, nxt[..., 0].clip(0, W - 1), nxt[..., 1].clip(0, W - 1)] == 0)
        ok &= (rng.random((C, N)) >= p_wait) & (t < length)
        pos = np.where(ok[..., None], nxt, pos)
        traj.append(pos.copy())
    traj = np.stack(traj, axis=1)                                   # [C,max_len,N,2]
    T = length.max(axis=1) + 1
    return [traj[c, :T[c]] for c in range(C)], traj[np.arange(C), T - 1], maps
