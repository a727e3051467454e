"""GPU: training batches built on the device (csrc/dataset.cu via gnn_pathplanning_b200.ExpertDataset) against the
files the original project's DataTransformer wrote (tests/golden/schedule_trace.npz) and against oracle/dataset_oracle.py
-- field of view, GSO and targets bit-exact -- and the online expert's round on the eval-trace sets: test_cases ->
setup_cases / evaluate -> failure_cases -> write_failure_cases, against the files the reference's agent wrote."""
import os

import numpy as np
import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def trace():
    g = np.load(os.path.join(ROOT, "tests", "golden", "schedule_trace.npz"), allow_pickle=False)
    return {k: g[k] for k in g.files}


@pytest.fixture(scope="module")
def eval_trace():
    g = np.load(os.path.join(ROOT, "tests", "golden", "eval_trace.npz"), allow_pickle=False)
    return {k: g[k] for k in g.files}


def case(trace, name):
    return {k[len(name) + 1:]: v for k, v in trace.items() if k.startswith(name + "_")}


def check_all_rows(ds, cases, order=None):
    """Every sample of the dataset, in `order` (default: all rows at once), against the files' contents."""
    x_ref = np.concatenate([c["inputTensor"].astype(np.float32) for c in cases])
    S_ref = np.concatenate([c["GSO"].astype(np.float32) for c in cases])
    t_ref = np.concatenate([c["target"].astype(np.int64) for c in cases])
    rows = torch.arange(len(ds), device="cuda") if order is None else order
    x, S, t = ds.batch(rows)
    r = rows.cpu().numpy()
    assert np.array_equal(x.cpu().numpy(), x_ref[r])
    assert np.array_equal(S.cpu().numpy(), S_ref[r])
    assert np.array_equal(t.cpu().numpy(), t_ref[r])


def test_batch_vs_reference_files(trace):
    import gnn_pathplanning_b200 as gp
    names = [str(n) for n in trace["cases"]]
    groups = {}
    for n in names:
        c = case(trace, n)
        groups.setdefault((c["goal"].shape[0], c["map"].shape[0]), []).append(c)
    assert {N for N, _ in groups} >= {5, 10, 20, 64}
    for (N, W), cases in groups.items():
        ds = gp.ExpertDataset(N).add([c["inputState"] for c in cases], np.stack([c["goal"] for c in cases]),
                                     np.stack([c["map"] for c in cases]))
        assert len(ds) == sum(int(c["makespan"]) for c in cases) and not ds.map_shared
        assert ds.radius.cpu().numpy().tolist() == [float(c["threshold"]) for c in cases], (N, W)
        check_all_rows(ds, cases)
        check_all_rows(ds, cases, torch.randperm(len(ds), device="cuda", generator=torch.Generator("cuda").manual_seed(N)))
    shared = [case(trace, n) for n in names if n.startswith("n10_shared")]
    assert len(shared) >= 2 and all(np.array_equal(c["map"], shared[0]["map"]) for c in shared)
    ds = gp.ExpertDataset(10).add([c["inputState"] for c in shared], np.stack([c["goal"] for c in shared]), shared[0]["map"])
    assert ds.map_shared
    check_all_rows(ds, shared)


def oracle_samples(positions, goals, maps, r0=5.0):
    from oracle import dataset_oracle
    xs, Ss, ts, thr = [], [], [], []
    for p, g, m in zip(positions, goals, maps):
        o = dataset_oracle.transform(m, g, p, r0)
        xs.append(o["inputTensor"]); Ss.append(o["GSO"].astype(np.float32)); ts.append(o["target"].astype(np.int64))
        thr.append(o["threshold"])
    return np.concatenate(xs), np.concatenate(Ss), np.concatenate(ts), thr


@pytest.mark.parametrize("N,W,C", [(10, 20, 24), (20, 28, 8), (40, 36, 4), (64, 40, 3)])
def test_random_sets_vs_oracle(N, W, C):
    import gnn_pathplanning_b200 as gp
    from gnn_pathplanning_b200 import synthetic
    rng = np.random.default_rng(N * 100 + W)
    pos, goals, maps = synthetic.random_schedules(rng, C, N, W, 0.1, max_len=20)
    h = C // 2
    ds = gp.ExpertDataset(N).add(pos[:h], goals[:h], maps[:h])
    first = [t.cpu().clone() for t in ds.batch(torch.arange(len(ds), device="cuda"))]
    R0 = len(ds)
    ds.add(pos[h:], goals[h:], maps[h:])                                 # appending leaves earlier samples unchanged
    assert len(ds) == sum(p.shape[0] for p in pos) and ds.num_cases == C
    again = ds.batch(torch.arange(R0, device="cuda"))
    assert all(torch.equal(a.cpu(), b) for a, b in zip(again, first))
    x_ref, S_ref, t_ref, thr = oracle_samples(pos, goals, maps)
    assert ds.radius.cpu().numpy().tolist() == thr
    gen = torch.Generator("cuda").manual_seed(7)
    order = torch.randperm(len(ds), device="cuda", generator=gen)
    for lo in range(0, len(ds), 13):                                      # partial last batch
        rows = order[lo:lo + 13]
        x, S, t = ds.batch(rows)
        r = rows.cpu().numpy()
        assert np.array_equal(x.cpu().numpy(), x_ref[r]) and np.array_equal(S.cpu().numpy(), S_ref[r])
        assert np.array_equal(t.cpu().numpy(), t_ref[r])
    x, S, t = ds.batch([5])                                               # batch size 1, host indices
    assert np.array_equal(x.cpu().numpy(), x_ref[5:6]) and np.array_equal(t.cpu().numpy(), t_ref[5:6])


def test_batches_visit_every_sample_once():
    """batches() walks one device-side permutation of all samples, a partial batch last: the same batches as
    batch() over torch.randperm with an identically seeded generator, and every sample's content exactly once."""
    import collections
    import gnn_pathplanning_b200 as gp
    from gnn_pathplanning_b200 import synthetic
    pos, goals, maps = synthetic.random_schedules(np.random.default_rng(3), 30, 10, 20)
    ds = gp.ExpertDataset(10).add(pos, goals, maps)
    assert len(ds) % 64 != 0
    order = torch.randperm(len(ds), device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    assert torch.equal(order.sort().values, torch.arange(len(ds), device="cuda"))
    fp = lambda x, S, t: [hash(r.numpy().tobytes()) for r in torch.cat([x.flatten(1), S.flatten(1), t.flatten(1).float()], 1).cpu()]
    want = collections.Counter(fp(*ds.batch(torch.arange(len(ds), device="cuda"))))
    got, sizes = collections.Counter(), []
    for k, (x, S, t) in enumerate(ds.batches(64, generator=torch.Generator("cuda").manual_seed(1))):
        ref = ds.batch(order[64 * k:64 * (k + 1)])
        assert all(torch.equal(a, b) for a, b in zip((x, S, t), ref)), k
        sizes.append(x.shape[0])
        got.update(fp(x, S, t))
    assert sizes == [64] * (len(ds) // 64) + [len(ds) % 64] and got == want


def test_envelope_and_out_buffers():
    import gnn_pathplanning_b200 as gp
    from gnn_pathplanning_b200 import synthetic
    pos, goals, maps = synthetic.random_schedules(np.random.default_rng(4), 3, 10, 20)
    with pytest.raises(ValueError):
        gp.ExpertDataset(10).add(pos, goals, maps[:, :, :19])
    ds = gp.ExpertDataset(10).add(pos, goals, maps)
    with pytest.raises(ValueError):
        ds.add(*synthetic.random_schedules(np.random.default_rng(5), 2, 10, 24))
    with pytest.raises(IndexError):
        ds.batch([len(ds)])
    out = (torch.empty(4, 10, 3, 11, 11, device="cuda"), torch.empty(4, 10, 10, device="cuda"),
           torch.empty(4, 10, 5, device="cuda", dtype=torch.int64))
    rows = torch.tensor([0, 3, 1, len(ds) - 1], device="cuda")
    got = ds.batch(rows, out=out)
    assert all(a is b for a, b in zip(got, out))
    ref = ds.batch(rows)
    assert all(torch.equal(a, b) for a, b in zip(got, ref))
    p65, g65, m65 = synthetic.random_schedules(np.random.default_rng(6), 1, 65, 40)
    with pytest.raises(ValueError):
        gp.ExpertDataset(65).add(p65, g65, m65)


def eval_cases_as_schedules(g):
    """The eval-trace cases whose expert moves span exactly `makespan` steps, as schedules whose test-loader view is
    the same cases: rows = the cells before each expert move."""
    D = np.array([[-1, 0], [0, -1], [1, 0], [0, 1], [0, 0]])
    keep, pos = [], []
    for b in range(g["input"].shape[0]):
        goal, start, m = g["input"][b, 0], g["input"][b, 1], int(g["makespan"][b])
        moves = D[g["target"][b].argmax(-1)]                                  # [N,T,2]
        cells = start[:, None] + np.concatenate([np.zeros_like(moves[:, :1]), np.cumsum(moves, 1)], 1)
        if m <= moves.shape[1] and (cells[:, m] == goal).all() and (g["target"][b][:, m:, 4] == 1).all():
            keep.append(b)
            pos.append(cells[:, :m].transpose(1, 0, 2))
    return np.array(keep), pos


def test_online_expert_round_vs_reference(trace, eval_trace, tmp_path):
    import gnn_pathplanning_b200 as gp
    from oracle import goal_policy
    policy = goal_policy.GoalSeekingPolicy().eval()
    for s in ("a", "b"):
        g = {k[2:]: v for k, v in eval_trace.items() if k.startswith(s + "_")}
        N = int(g["cfg"][0])
        ids_ref, cells_ref = trace["fail_%s_ids" % s], trace["fail_%s_cells" % s]
        names_ref, texts_ref = [str(n) for n in trace["fail_%s_names" % s]], [str(t) for t in trace["fail_%s_texts" % s]]
        # the dataset's view of the cases equals the test loader's
        keep, pos = eval_cases_as_schedules(g)
        assert len(keep) >= g["input"].shape[0] - 1
        ds = gp.ExpertDataset(N).add(pos, g["input"][keep, 0], g["map"][keep])
        inp, target, makespan, maps = ds.test_cases()
        T = target.shape[2]
        assert np.array_equal(inp.cpu().numpy(), g["input"][keep])
        assert np.array_equal(makespan.numpy(), g["makespan"][keep])
        want = g["target"][keep][:, :, :T]
        assert np.array_equal(target.cpu().numpy(), want.astype(np.int64)) and (g["target"][keep][:, :, T:, 4] == 1).all()
        ro = gp.BatchedRollout(N).setup_cases(inp, target, makespan, maps)
        ro.evaluate(policy, poll_every=4)
        ids, cells = ro.failure_cases()
        orig = keep[ids]
        sel = np.isin(ids_ref, keep)
        assert np.array_equal(orig, ids_ref[sel]) and np.array_equal(cells, cells_ref[sel]), s
        d = tmp_path / s
        d.mkdir()
        gp.write_failure_cases(str(d), orig, g["map"][orig], cells, g["input"][orig, 0])
        for n, t in zip(names_ref, texts_ref):
            if int(n.split("ID")[1][:5]) in orig:
                assert (d / n).read_text() == t, (s, n)
        # every case, including ones a schedule cannot express (a success exactly at maxstep), through setup_cases
        ro = gp.BatchedRollout(N).setup_cases(g["input"], g["target"], g["makespan"], g["map"])
        ro.evaluate(policy, poll_every=4)
        ids, cells = ro.failure_cases()
        assert np.array_equal(ids, ids_ref) and np.array_equal(cells, cells_ref), s
        d = tmp_path / (s + "_all")
        d.mkdir()
        paths = gp.write_failure_cases(str(d), ids, g["map"][ids], cells, g["input"][ids, 0])
        assert sorted(os.path.basename(p) for p in paths) == names_ref
        for n, t in zip(names_ref, texts_ref):
            assert (d / n).read_bytes() == t.encode(), (s, n)


class Cfg:
    def __init__(self, n, k):
        self.num_agents, self.nGraphFilterTaps, self.device = n, k, torch.device("cuda")


def test_train_step_on_batch_vs_oracle_tensors():
    """One planner_loss training step fed by ExpertDataset.batch gives the loss and gradients of the same step fed
    with the oracle's tensors."""
    import gnn_pathplanning_b200 as gp
    from gnn_pathplanning_b200 import synthetic
    from oracle import planner_oracle as po
    N = 10
    pos, goals, maps = synthetic.random_schedules(np.random.default_rng(11), 6, N, 20)
    ds = gp.ExpertDataset(N).add(pos, goals, maps)
    x_ref, S_ref, t_ref, _ = oracle_samples(pos, goals, maps)
    rows = torch.randperm(len(ds), device="cuda", generator=torch.Generator("cuda").manual_seed(2))[:48]
    r = rows.cpu().numpy()
    sd = po.init_state_dict(3, seed=5)
    results = []
    for x, S, t in (ds.batch(rows), tuple(torch.from_numpy(a[r]).cuda() for a in (x_ref, S_ref, t_ref))):
        m = gp.DecentralPlannerNet(Cfg(N, 3))
        m.load_state_dict(sd)
        m = m.cuda().train()
        m.addGSO(S)
        loss = gp.planner_loss(m.forward_logits(x), t)
        loss.backward()
        results.append((loss.item(), {k: p.grad.detach().cpu().numpy() for k, p in m.named_parameters()}))
    (l0, g0), (l1, g1) = results
    assert abs(l0 - l1) <= 1e-5 * abs(l1)
    for k in g1:
        # conv biases feed a train-mode BatchNorm: their true gradient is 0, both sides hold rounding noise
        den = 1.0 if k in ("ConvLayers.%d.bias" % ci for ci in (0, 4, 7, 11, 14)) else max(float(np.abs(g1[k]).max()), 1e-30)
        assert float(np.abs(g0[k] - g1[k]).max()) / den <= 1e-5, k
