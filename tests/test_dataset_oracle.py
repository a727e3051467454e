"""CPU: the training-data restatement (oracle/dataset_oracle.py), the readers and the failure-case writer of
gnn_pathplanning_b200/dataset.py against what the original project's DataTransformer and online-expert agent wrote
(tests/golden/schedule_trace.npz) -- bit for bit, byte for byte -- and the host-side rejections."""
import os

import numpy as np
import pytest
import scipy.io
import yaml

from gnn_pathplanning_b200 import dataset
from oracle import dataset_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def trace():
    g = np.load(os.path.join(ROOT, "tests", "golden", "schedule_trace.npz"), allow_pickle=False)
    return {k: g[k] for k in g.files}


def case(trace, name):
    return {k[len(name) + 1:]: v for k, v in trace.items() if k.startswith(name + "_")}


def plans_of(solution_yaml, N):
    s = yaml.safe_load(solution_yaml)
    return [[(c["x"], c["y"]) for c in s["schedule"]["agent%d" % i]] for i in range(N)], s["statistics"]["makespan"]


def test_oracle_vs_reference_transformer(trace):
    names = [str(n) for n in trace["cases"]]
    assert len(names) >= 10
    grew_later = False
    for name in names:
        c = case(trace, name)
        N = c["goal"].shape[0]
        plans, makespan = plans_of(str(c["solution_yaml"]), N)
        pos, tgt = dataset_oracle.obtain_schedule(plans, c["goal"], makespan)
        assert np.array_equal(pos, c["inputState"]) and np.array_equal(tgt, c["target"]), name
        assert int(c["makespan"]) == makespan + 1 == pos.shape[0], name
        out = dataset_oracle.transform(c["map"], c["goal"], pos)
        assert out["threshold"] == float(c["threshold"]), name
        assert np.array_equal(out["GSO"], c["GSO"]), name
        assert np.array_equal(out["inputTensor"], c["inputTensor"].astype(np.float32)), name
        assert np.array_equal(out["target"], c["target"]), name
        if dataset_oracle.schedule_threshold(pos[:1]) < float(c["threshold"]):
            grew_later = True
    assert grew_later, "no case whose threshold grows after step 0"


def write_solutions(tmp, trace, names):
    inp, sol = tmp / "input", tmp / "output_ECBS"
    inp.mkdir()
    sol.mkdir()
    for k, name in enumerate(names):
        c = case(trace, name)
        (inp / ("failureCases_ID%05d.yaml" % k)).write_text(str(c["input_yaml"]))
        (sol / ("failureCases_solved_ID%05d.yaml" % k)).write_text(str(c["solution_yaml"]))
    return str(inp), str(sol)


def groups(trace):
    out = {}
    for name in (str(n) for n in trace["cases"]):
        c = case(trace, name)
        out.setdefault((c["goal"].shape[0], c["map"].shape[0]), []).append(name)
    return out


def test_read_ecbs_solutions(trace, tmp_path):
    for (N, W), names in groups(trace).items():
        d = tmp_path / ("n%d_w%d" % (N, W))
        d.mkdir()
        pos, goals, maps = dataset.read_ecbs_solutions(*write_solutions(d, trace, names))
        assert len(pos) == len(names) and maps.shape == (len(names), W, W)
        for k, name in enumerate(names):
            c = case(trace, name)
            assert np.array_equal(pos[k], c["inputState"]) and np.array_equal(goals[k], c["goal"]), name
            assert np.array_equal(maps[k], c["map"]), name


def test_read_mat_cases(trace, tmp_path):
    """Files written as the reference's DataTransformer.save does (scipy.io.savemat of the same fields)."""
    for (N, W), names in groups(trace).items():
        paths = []
        for name in names:
            c = case(trace, name)
            p = str(tmp_path / ("train_%s_MP%d.mat" % (name, int(c["makespan"]))))
            scipy.io.savemat(p, {"map": c["map"].astype(np.float64), "goal": c["goal"].astype(np.float64),
                                 "inputState": c["inputState"].astype(np.float64),
                                 "inputTensor": c["inputTensor"].astype(np.float32),
                                 "target": c["target"].astype(np.float64), "GSO": c["GSO"],
                                 "makespan": int(c["makespan"]), "HashIDs": np.zeros(N)})
            paths.append(p)
        pos, goals, maps = dataset.read_mat_cases(paths)
        for k, name in enumerate(names):
            c = case(trace, name)
            assert np.array_equal(pos[k], c["inputState"]) and np.array_equal(goals[k], c["goal"]), name
            assert np.array_equal(maps[k], c["map"]), name


def test_reader_rejections(trace, tmp_path):
    # a two-cell jump: the reference's transformer raises ValueError on it too
    (tmp_path / "a").mkdir()
    inp, sol = tmp_path / "a" / "input", tmp_path / "a" / "output_ECBS"
    inp.mkdir()
    sol.mkdir()
    (inp / "failureCases_ID00007.yaml").write_text(str(trace["invalid_input_yaml"]))
    (sol / "failureCases_solved_ID00007.yaml").write_text(str(trace["invalid_solution_yaml"]))
    with pytest.raises(ValueError, match="failureCases_solved_ID00007"):
        dataset.read_ecbs_solutions(str(inp), str(sol))
    # a plan longer than makespan + 1 steps
    c = case(trace, "n10_shared0")
    s = yaml.safe_load(str(c["solution_yaml"]))
    s["statistics"]["makespan"] = max(len(p) for p in s["schedule"].values()) - 2
    (tmp_path / "b").mkdir()
    inp, sol = tmp_path / "b" / "input", tmp_path / "b" / "output_ECBS"
    inp.mkdir()
    sol.mkdir()
    (inp / "failureCases_ID00003.yaml").write_text(str(c["input_yaml"]))
    (sol / "failureCases_solved_ID00003.yaml").write_text(yaml.safe_dump(s))
    with pytest.raises(ValueError, match="failureCases_solved_ID00003.*longer"):
        dataset.read_ecbs_solutions(str(inp), str(sol))
    # a test-format file: 2-D inputState
    p = str(tmp_path / "test_ID00001_MP5.mat")
    scipy.io.savemat(p, {"map": c["map"].astype(np.float64), "goal": c["goal"].astype(np.float64),
                         "inputState": c["inputState"][0].astype(np.float64)})
    with pytest.raises(ValueError, match="test_ID00001"):
        dataset.read_mat_cases([p])


def test_validate_cases_rejections(trace):
    c = case(trace, "n10_shared0")
    pos, goal, m = c["inputState"], c["goal"], c["map"]
    ok = dataset.validate_cases([pos, pos], np.stack([goal, goal]), m, 10)
    assert len(ok[0]) == 2 and ok[2].shape == m.shape
    jump = pos.copy()
    jump[3, 2] = jump[2, 2] + np.array([2, 0]) if jump[2, 2, 0] + 2 < m.shape[0] else jump[2, 2] - np.array([2, 0])
    with pytest.raises(ValueError, match=r"cases \[1\]: a move"):
        dataset.validate_cases([pos, jump, pos], np.stack([goal] * 3), m, 10)
    bad_goal = goal.copy()
    bad_goal[4] += np.array([0, 3]) if goal[4, 1] + 3 < m.shape[0] else np.array([0, -3])
    with pytest.raises(ValueError, match=r"cases \[0\]: a move"):
        dataset.validate_cases([pos, pos], np.stack([bad_goal, goal]), m, 10)
    with pytest.raises(ValueError, match="at least 2"):
        dataset.validate_cases([pos[:, :1]], goal[None, :1], m)
    with pytest.raises(ValueError, match="square"):
        dataset.validate_cases([pos], goal[None], np.zeros((m.shape[0], m.shape[0] + 1)))
    with pytest.raises(ValueError, match="the dataset has 12"):
        dataset.validate_cases([pos], goal[None], m, 12)
    out = pos.copy()
    out[:, 0] = [-1, 0]
    with pytest.raises(ValueError, match=r"cases \[0\]: a cell or goal lies outside"):
        dataset.validate_cases([out], goal[None], m)
    with pytest.raises(ValueError, match="whole numbers"):
        dataset.validate_cases([pos + 0.5], goal[None], m)


def test_write_failure_cases_vs_reference(trace, tmp_path):
    ev = np.load(os.path.join(ROOT, "tests", "golden", "eval_trace.npz"), allow_pickle=False)
    seen_at_maxstep = False
    for s in ("a", "b"):
        ids, cells = trace["fail_%s_ids" % s], trace["fail_%s_cells" % s]
        names, texts = [str(n) for n in trace["fail_%s_names" % s]], [str(t) for t in trace["fail_%s_texts" % s]]
        goals, maps = ev[s + "_input"][ids, 0], ev[s + "_map"][ids]
        d = tmp_path / s
        d.mkdir()
        paths = dataset.write_failure_cases(str(d), ids, maps, cells, goals)
        assert sorted(os.path.basename(p) for p in paths) == names
        for n, t in zip(names, texts):
            assert (d / n).read_bytes() == t.encode(), (s, n)
        for k in range(len(ids)):
            assert dataset_oracle.failure_case_text(maps[k], cells[k], goals[k]) == texts[k], (s, k)
        # a success that lands exactly on maxstep is dumped too
        reach = ev[s + "_list_reachGoal"][ids]
        seen_at_maxstep |= bool(reach.any())
    assert seen_at_maxstep
    # a shared [W,W] map writes the same text; the directory must exist; nothing else in it is touched
    keep = tmp_path / "a" / "other.txt"
    keep.write_text("x")
    ids, cells = trace["fail_a_ids"][:1], trace["fail_a_cells"][:1]
    dataset.write_failure_cases(str(tmp_path / "a"), ids, ev["a_map"][ids[0]], cells, ev["a_input"][ids, 0])
    assert keep.read_text() == "x"
    with pytest.raises(FileNotFoundError):
        dataset.write_failure_cases(str(tmp_path / "missing"), ids, ev["a_map"][ids], cells, ev["a_input"][ids, 0])


def test_validate_cases_returns_c_order(trace):
    """.mat arrays arrive in Fortran order; the device kernels read raw C-order buffers."""
    c = case(trace, "n10_shared0")
    pos, goals, maps = dataset.validate_cases([np.asfortranarray(c["inputState"])], np.asfortranarray(c["goal"][None]),
                                              np.asfortranarray(np.stack([c["map"]])))
    assert pos[0].flags.c_contiguous and goals.flags.c_contiguous and maps.flags.c_contiguous
