"""K5 at four objectives through the C ABI and the Python API, against the literal restatement of the reference's
hypervolume (tests/hv_ref.py). Bar: bit-exact hypervolume, sparsity, picks and virtual front (float64, the reference's
operations in the reference's order)."""
import os

import numpy as np
import pytest

import hv_ref
from oracle import selection_oracle as so

pytestmark = pytest.mark.gpu

MAX_FRONT_4D = 2202          # the 4-D scorer's shared-memory layout (csrc/k5_select.cu, include/pgmorl_b200.h)


def _sphere(rng, n, r=80.0):
    v = np.abs(rng.normal(size=(n, 4))) + 0.05
    return v / np.linalg.norm(v, axis=1, keepdims=True) * r


def _metrics_ref(pts):
    return hv_ref.hv(pts), so.sparsity_md(pts)


def test_front_metrics_random_sets():
    from pgmorl_b200 import kernels as K
    rng = np.random.RandomState(7)
    for n in (1, 2, 3, 17, 64, 300):
        for pts in (rng.uniform(0, 50, (n, 4)), _sphere(rng, n)):
            if n > 3:
                pts[2, 0] = pts[1, 0]; pts[3, 1:] = pts[1, 1:]
            assert K.front_metrics(pts) == _metrics_ref(pts), n


def test_front_metrics_integer_sets_and_area_reuse():
    """Ties, duplicates, dominated points, zero and negative coordinates; the inputs reach the sweep's area-reuse
    branch, including the sets where two points agree in objectives 0-2 (tests/test_oracle_hv_md.py)."""
    from pgmorl_b200 import kernels as K
    rng = np.random.RandomState(3)
    hv_ref.reset_reuse_count()
    for it in range(120):
        pts = rng.randint(0, 6, (rng.randint(1, 40), 4)).astype(np.float64)
        if it % 4 == 3:
            pts[rng.rand(len(pts)) < 0.2, rng.randint(4)] = -1.0
        assert K.front_metrics(pts) == _metrics_ref(pts), it
    assert hv_ref.reuse_count > 0
    hv_ref.reset_reuse_count()
    for it in range(20):                                       # real-valued fronts with dominated points mixed in
        pts = np.vstack([_sphere(rng, 60), rng.uniform(0, 45, (30, 4))])
        rng.shuffle(pts)
        assert K.front_metrics(pts) == _metrics_ref(pts), it
    assert hv_ref.reuse_count > 0


def _check_greedy(ep, cand, alpha, num_tasks):
    from pgmorl_b200 import kernels as K
    best, hv, sp, front = K.select_greedy(ep, cand, alpha, num_tasks)
    ob, ohv, osp, ofront = hv_ref.greedy_select_md(ep, cand, alpha, num_tasks)
    assert best.tolist() == ob + [-1] * (num_tasks - len(ob))
    for r in range(len(ohv)):
        assert np.array_equal(hv[r], ohv[r]), r
        assert np.array_equal(sp[r], osp[r]), r
    assert np.array_equal(front, np.array(ofront, dtype=np.float64).reshape(-1, 4))
    return best, hv, sp


def _product_classes():
    from pgmorl_b200.ep import EP
    from pgmorl_b200.opt_graph import OptGraph
    from pgmorl_b200.population_3d import Population
    from pgmorl_b200.scalarization_methods import WeightedSumScalarization
    return dict(EP=EP, Population=Population, OptGraph=OptGraph, Scalarization=WeightedSumScalarization)


def _capture_k5(monkeypatch):
    """Record every call of kernels.select_greedy (inputs and outputs) the product makes."""
    from pgmorl_b200 import kernels as K
    calls, real = [], K.select_greedy

    def spy(ep, cand, alpha, num_tasks):
        out = real(ep, cand, alpha, num_tasks)
        calls.append(dict(ep=np.array(ep, dtype=np.float64), cand=np.array(cand, dtype=np.float64), alpha=alpha,
                          num_tasks=num_tasks, out=out))
        return out
    monkeypatch.setattr(K, "select_greedy", spy)
    return calls


@pytest.mark.parametrize("seed", [0, 1])
def test_greedy_selection_on_synthetic_histories(monkeypatch, seed):
    """The virtual front and candidate predictions K5 receives in every generation of a 4-objective selection
    history: every round's hv / sparsity, every pick and the final front equal greedy_select_md."""
    import synth_envs
    calls = _capture_k5(monkeypatch)
    args = synth_envs.SelectionArgs(4, pbuffer_num=6, delta_weight=0.5, num_tasks=6)
    synth_envs.run_selection_history(_product_classes(), args, 3, seed)
    greedy = [c for c in calls if c["num_tasks"] == args.num_tasks]
    assert len(greedy) == 3
    for c in greedy:
        assert len(c["cand"]) > args.num_tasks
        _check_greedy(c["ep"], c["cand"], c["alpha"], c["num_tasks"])


def test_greedy_edge_cases():
    rng = np.random.RandomState(2)
    ep = _sphere(rng, 12, 10.0)
    ep = ep[np.argsort(ep[:, 0], kind="stable")]
    cand = np.vstack([rng.uniform(0, 12, (5, 4)), ep[3], [4.0, -1.0, 8.0, 8.0], [9.0, 9.0, 9.0, 9.5]])
    _check_greedy(np.zeros((0, 4)), cand, 1e6, 3)                         # empty archive
    best, _, _ = _check_greedy(ep, cand[:2], 1e6, 4)                       # fewer candidates than tasks
    assert best.tolist()[2:] == [-1, -1]
    _check_greedy(ep, cand, 1e6, 5)                                        # equal point, negative coordinate
    big = np.vstack([ep, [[8.0, 8.0, 8.0, 8.0]]])                          # dominates most of the archive
    _check_greedy(ep, big[::-1].copy(), 1.0, 4)
    dup = rng.randint(0, 4, (30, 4)).astype(np.float64)                    # ties and duplicates everywhere
    _check_greedy(dup[:10], dup[10:], 1.0, 5)


def test_size_limit():
    """The largest front the 4-D layout admits is scored exactly; one more point is refused with the library's error."""
    from pgmorl_b200 import kernels as K
    from pgmorl_b200._lib import PgmError
    n = MAX_FRONT_4D
    i = np.arange(n, dtype=np.float64)
    pts = np.stack([i, n - i, i + 1.0, 2.0 * i + 3.0], axis=1)             # mutually non-dominated
    assert K.front_metrics(pts) == _metrics_ref(pts)
    with pytest.raises(PgmError, match="4-D scorer's shared memory"):
        K.front_metrics(np.vstack([pts, pts[:1] + 0.5]))
    with pytest.raises(PgmError, match="4-D scorer's shared memory"):
        K.select_greedy(pts[:n - 1], pts[:1], 1.0, 1)                      # archive + num_tasks + 1 > limit
    K.select_greedy(pts[:n - 2], pts[:1], 1.0, 1)                          # exactly at the limit


def test_full_size_selection(monkeypatch):
    """make_selection_state(4, 420, 500) through prediction_guided_selection: a sample of round-0 candidates scored
    exactly as the restatement scores them, and the first pick is the arg-max of the product's own scores."""
    import synth_envs
    from pgmorl_b200.scalarization_methods import WeightedSumScalarization
    calls = _capture_k5(monkeypatch)
    args, graph, pop, ep = synth_envs.make_selection_state(4, 420, 500)
    np.random.seed(0)
    template = WeightedSumScalarization(num_objs=4, weights=np.ones(4) / 4)
    elites, scals, predicted = pop.prediction_guided_selection(args, 0, ep, graph, template)
    assert len(elites) == args.num_tasks
    (c,) = [c for c in calls if c["num_tasks"] == args.num_tasks]
    best, hv, sp, _ = c["out"]
    assert len(c["cand"]) > 2500 and len(c["ep"]) == 500
    rng = np.random.RandomState(1)
    for i in rng.choice(len(c["cand"]), 40, replace=False):
        front = so.update_ep(c["ep"], c["cand"][i])
        assert hv[0][i] == hv_ref.hv(front) and sp[0][i] == so.sparsity_md(front), i
    score = hv[0] - c["alpha"] * sp[0]
    assert best[0] == int(np.argmax(score))
    assert np.array_equal(predicted[0], c["cand"][best[0]])


def test_python_api():
    from pgmorl_b200 import kernels as K
    from pgmorl_b200 import utils
    from pgmorl_b200._lib import PgmError
    from pgmorl_b200.hypervolume import InnerHyperVolume
    rng = np.random.RandomState(4)
    for n in (1, 5, 40):
        pts = np.vstack([_sphere(rng, n), rng.uniform(-5, 40, (n, 4))])
        assert InnerHyperVolume(np.zeros(4)).compute(pts) == hv_ref.hv(pts)
        assert utils.compute_sparsity(pts) == so.sparsity_md(pts)
        front = _sphere(rng, n)
        front = front[np.argsort(front[:, 0], kind="stable")]
        for new in (rng.uniform(0, 80, 4), front[0], np.array([1.0, -1.0, 2.0, 3.0])):
            got = utils.update_ep(front, new)
            ref = so.update_ep(front, new)
            assert np.array_equal(np.array(got).reshape(-1, 4), np.array(ref).reshape(-1, 4))
    p5 = rng.uniform(0, 1, (6, 5))
    for call in (lambda: InnerHyperVolume(np.zeros(5)).compute(p5), lambda: utils.compute_sparsity(p5),
                 lambda: utils.update_ep(p5, p5[0])):
        with pytest.raises(NotImplementedError, match="4 objectives"):
            call()
    with pytest.raises(PgmError, match="2 to 4 objectives"):
        K.front_metrics(p5)
    with pytest.raises(PgmError, match="2 to 4 objectives"):
        K.select_greedy(p5, p5, 1.0, 1)


def _run_args_4d(save_dir, method):
    import synth_envs
    args = synth_envs.run_args_2d(str(save_dir))
    args.obj_num, args.delta_weight, args.pbuffer_num, args.sparsity = 4, 0.5, 6, 1e6
    args.selection_method = method
    return args


class _ToyEvalEnv4:
    """synth_envs.ToyEvalEnv with four objectives: one smooth function of the mean action per third of the action."""

    def __init__(self, dims):
        import synth_envs
        self.env = synth_envs.ToyEvalEnv(dims)
        self.observation_space, self.action_space = self.env.observation_space, self.env.action_space

    def seed(self, s):
        self.env.seed(s)

    def reset(self):
        return self.env.reset()

    def step(self, action):
        ob, r, done, _ = self.env.step(action)
        a = np.asarray(action, dtype=np.float64).reshape(-1)
        obj = np.array([1.0 + np.tanh(a[0:2].sum()), 1.0 + np.tanh(a[2:4].sum()), 1.0 + np.tanh(a[4:6].sum()), 1.0])
        return ob, r, done, {"obj": obj}

    def close(self):
        pass


def _run(save_dir, method):
    import synth_envs
    from pgmorl_b200 import mopg, morl
    from pgmorl_b200.layout import NetDims
    d = NetDims(17, 6, 4)
    args = _run_args_4d(save_dir, method)
    mopg.set_env_hooks(
        make_vec_envs=lambda **kw: synth_envs.SeededReplayVecEnv(d, args.num_steps, args.num_processes,
                                                                 [1.3, 0.7, 1.0, 0.9], base_seed=500),
        gym_make=lambda name: _ToyEvalEnv4(d))
    return args, morl.run(args, device="cuda")


def _files(root):
    out = {}
    for dirpath, _, names in os.walk(root):
        for name in names:
            if name.endswith(".txt"):
                path = os.path.join(dirpath, name)
                out[os.path.relpath(path, root)] = open(path, "rb").read()
    return out


def test_whole_run_prediction_guided(tmp_path, monkeypatch):
    """warm-up + 2 generations at 4 objectives: 4-column result files, every generation's picks equal greedy_select_md
    on that generation's archive and the product's own predictions, and a second identical run writes the same bytes."""
    calls = _capture_k5(monkeypatch)
    args, (ep, population, graph, timings) = _run(tmp_path / "a", "prediction-guided")
    assert len(timings) == 3
    files = _files(tmp_path / "a")
    gens = sorted((d for d in os.listdir(tmp_path / "a") if d.isdigit()), key=int)
    greedy = [c for c in calls if c["num_tasks"] == args.num_tasks]
    assert len(greedy) == len(gens) >= 2
    for c, gen in zip(greedy, gens):
        for sub in ("ep/objs.txt", "population/objs.txt", "elites/predictions.txt"):
            rows = files[os.path.join(gen, sub)].decode().strip().splitlines()
            assert rows and all(len(r.split(",")) == 4 for r in rows), (gen, sub)
        best, _, _ = _check_greedy(c["ep"], c["cand"], c["alpha"], c["num_tasks"])
        rows = files[os.path.join(gen, "elites", "predictions.txt")].decode().strip().splitlines()
        got = np.array([[float(x) for x in r.split(",")] for r in rows])
        assert np.allclose(got, c["cand"][best[best >= 0]], rtol=0, atol=5e-7), gen
    _run(tmp_path / "b", "prediction-guided")
    assert _files(tmp_path / "b") == files


@pytest.mark.parametrize("method", ["moead", "ra", "random"])
def test_whole_run_other_modes(tmp_path, method):
    _run(tmp_path, method)
    rows = open(os.path.join(tmp_path, "final", "objs.txt")).read().strip().splitlines()
    assert rows and all(len(r.split(",")) == 4 for r in rows)


def test_whole_run_pfa_refuses(tmp_path):
    with pytest.raises(NotImplementedError):
        _run(tmp_path, "pfa")
