"""K5 at three objectives past the shared-memory layouts: the global-memory path (csrc/k5_select.cu, PGM_SEL_GLOBAL).

Two bars:
  * where both paths run, the global path gives the same bits as the shared-memory kernels (every round's hv and
    sparsity, the picks, the final front, front_metrics);
  * past the old limits (2 111 points for select_greedy, 3 936 for front_metrics) the results equal a vectorised
    restatement of oracle/selection_oracle.hv3d_raw / sparsity_md / update_ep, which is pinned bit for bit to the
    oracle on small fronts below, and an exact integer computation on integer fronts.
The restatement tests at the top need no GPU."""
import os

import numpy as np
import pytest

from oracle import selection_oracle as so

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
OLD_GREEDY_LIMIT = 2111          # archive + num_tasks + 1 of the shared-memory incremental scorer
OLD_METRICS_LIMIT = 3936         # points of the shared-memory one-front scorer


# ---------------------------------------------------------------------------------------------------------------------
# the restatement: hypervolume.py:106-153 at dimIndex 2 (as so.hv3d_raw), vectorised across the z-slices
# ---------------------------------------------------------------------------------------------------------------------
def hv3d_raw_fast(front):
    """so.hv3d_raw with every slice's operations in the original order; the slices advance together. Slice k holds the
    first k+1 points of the z list; walking the y list, the point of z rank r joins slices r..n-1."""
    pts = -np.asarray(front, dtype=np.float64).reshape(-1, 3)
    pts = pts[(pts <= 0.0).all(axis=1)]
    n = len(pts)
    if n == 0:
        return 0.0
    x, y, z = pts[:, 0], pts[:, 1], pts[:, 2]
    ylist = np.lexsort((x, y))                       # stable sorts by x, then y (ties keep the input order)
    zlist = ylist[np.argsort(z[ylist], kind="stable")]
    zr = np.empty(n, dtype=np.int64)
    zr[zlist] = np.arange(n)
    h = np.zeros(n); acc = np.zeros(n); prev = np.zeros(n); seen = np.zeros(n, dtype=bool)
    for j in ylist:
        r = zr[j]
        xj, yj = x[j], y[j]
        s = seen[r:]
        hh = h[r:]
        acc[r:] = np.where(s, acc[r:] + hh * (prev[r:] - yj), acc[r:])
        h[r:] = np.where(s & (xj >= hh), hh, xj)
        prev[r:] = yj
        seen[r:] = True
    area = acc + h * prev
    hv = 0.0
    zs = z[zlist]
    for k in range(1, n):
        hv += float(area[k - 1]) * (float(zs[k]) - float(zs[k - 1]))
    hv -= float(area[n - 1]) * float(zs[n - 1])
    return hv


def sparsity_fast(front):
    """so.sparsity_md: the same squared gaps, summed in the same order."""
    front = np.asarray(front, dtype=np.float64)
    if len(front) < 2:
        return 0.0
    s = 0.0
    for dim in range(front.shape[1]):
        v = np.sort(front[:, dim])
        for g2 in np.square(v[1:] - v[:-1]).tolist():
            s += g2
    return s / (len(front) - 1)


def update_ep_fast(ep, new):
    """so.update_ep (utils.py:42-65) with the comparisons done on whole arrays."""
    new = np.asarray(new, dtype=np.float64)
    ep = np.asarray(ep, dtype=np.float64).reshape(-1, len(new))
    if (new < 0).any():
        return [p for p in ep]
    on_ep = not ((ep >= new - 1e-5).all(axis=1) & (ep > new + 1e-5).any(axis=1)).any()
    out = ep[~(new >= ep).all(axis=1)]
    if on_ep:
        after = np.nonzero(new[0] < out[:, 0])[0]
        pos = int(after[0]) if len(after) else len(out)
        out = np.insert(out, pos, new, axis=0)
    return [p for p in out]


def hv3d_exact_int(front):
    """Exact hypervolume of integer points >= 0: unit cells (a, b) of the x-y plane are covered up to the largest z
    among the points with x > a and y > b."""
    p = np.asarray(front, dtype=np.int64).reshape(-1, 3)
    p = p[(p > 0).all(axis=1)]
    if len(p) == 0:
        return 0
    top = np.zeros((p[:, 0].max(), p[:, 1].max()), dtype=np.int64)
    np.maximum.at(top, (p[:, 0] - 1, p[:, 1] - 1), p[:, 2])
    top = np.maximum.accumulate(top[::-1], axis=0)[::-1]
    top = np.maximum.accumulate(top[:, ::-1], axis=1)[:, ::-1]
    return int(top.sum())


def sparsity_exact_int(front):
    p = np.asarray(front, dtype=np.int64)
    s = sum(int(np.square(np.diff(np.sort(p[:, d]))).sum()) for d in range(p.shape[1]))
    return float(s) / (len(p) - 1)


def _sphere(rng, n, r=80.0):
    v = np.abs(rng.normal(size=(n, 3))) + 0.05
    v = v / np.linalg.norm(v, axis=1, keepdims=True) * r
    return v[np.argsort(v[:, 0], kind="stable")]


def _int_plane(rng, n, s=260):
    """n distinct integer points with x + y + z = s (mutually non-dominated), ordered by x."""
    a = np.array([(x, y, s - x - y) for x in range(1, s - 1) for y in range(1, s - x)], dtype=np.float64)
    p = a[rng.choice(len(a), n, replace=False)]
    return p[np.argsort(p[:, 0], kind="stable")]


def _small_sets(rng):
    for n in (1, 2, 3, 7, 40, 150):
        yield rng.uniform(0, 50, (n, 3))
        yield _sphere(rng, n)
        yield rng.randint(0, 5, (n, 3)).astype(np.float64)                # ties and duplicates
    p = _sphere(rng, 60)
    p[5, 0] = p[4, 0]; p[9, 1:] = p[8, 1:]; p[20] = p[21]
    yield p
    yield np.vstack([_sphere(rng, 30), rng.uniform(-5, 40, (20, 3))])    # negative coordinates, dominated points


# ---------------------------------------------------------------------------------------------------------------------
# the restatement is the oracle (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def test_restatement_matches_oracle_bit_for_bit():
    rng = np.random.RandomState(11)
    for it, pts in enumerate(_small_sets(rng)):
        assert hv3d_raw_fast(pts) == so.hv3d_raw(pts), it
        assert sparsity_fast(pts) == so.sparsity_md(pts), it
        ep = pts[np.argsort(pts[:, 0], kind="stable")][: len(pts) // 2]
        for new in (pts[-1], ep[0] if len(ep) else pts[0], ep[-1] + 5e-6 if len(ep) else pts[0],
                    np.array([3.0, -1.0, 2.0]), rng.uniform(0, 60, 3)):
            got, ref = update_ep_fast(ep, new), so.update_ep(ep, new)
            assert np.array_equal(np.array(got).reshape(-1, 3), np.array(ref).reshape(-1, 3)), it


def test_exact_integer_metrics_match_restatement():
    rng = np.random.RandomState(12)
    for n in (1, 5, 60, 400):
        pts = rng.randint(0, 9, (n, 3)).astype(np.float64)
        assert hv3d_raw_fast(pts) == float(hv3d_exact_int(pts)), n
        if n >= 2:
            assert sparsity_fast(pts) == sparsity_exact_int(pts), n
    pts = _int_plane(rng, 500)
    assert hv3d_raw_fast(pts) == float(hv3d_exact_int(pts))


@pytest.fixture
def restated_oracle(monkeypatch):
    """so.greedy_select_3d / greedy_select_2d_fork with the fast restatement plugged in."""
    monkeypatch.setattr(so, "hv3d_raw", hv3d_raw_fast)
    monkeypatch.setattr(so, "sparsity_md", sparsity_fast)
    monkeypatch.setattr(so, "update_ep", update_ep_fast)
    return so


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the two paths agree where both run
# ---------------------------------------------------------------------------------------------------------------------
def _both_paths(ep, cand, alpha, num_tasks):
    from pgmorl_b200 import kernels as K
    a = K.select_greedy(ep, cand, alpha, num_tasks)
    b = K.select_greedy(ep, cand, alpha, num_tasks, force_global=True)
    assert np.array_equal(a[0], b[0])
    for r in range(num_tasks):
        assert np.array_equal(a[1][r], b[1][r]), r
        assert np.array_equal(a[2][r], b[2][r]), r
    assert np.array_equal(a[3], b[3])
    return a


def _metrics_both(pts):
    from pgmorl_b200 import kernels as K
    a = K.front_metrics(pts)
    assert K.front_metrics(pts, force_global=True) == a
    return a


@pytest.mark.gpu
def test_paths_agree_on_the_recorded_history():
    z = np.load(os.path.join(GOLDEN, "selection_3d.npz"))
    alpha = float(z["args_f"][0]); num_tasks = int(z["args"][0])
    for g in range(int(z["meta"][1])):
        best, hv, sp, _ = _both_paths(z[f"g{g}_round0_vep"], z[f"g{g}_cand_pred"], alpha, num_tasks)
        for r in range(num_tasks):
            assert np.array_equal(hv[r], z[f"g{g}_round{r}_hv"]) and np.array_equal(sp[r], z[f"g{g}_round{r}_sparsity"])
            _metrics_both(z[f"g{g}_round{r}_vep"])


@pytest.mark.gpu
def test_paths_agree_at_full_size(monkeypatch):
    """make_selection_state(3, 420, 500): the product's own selection call, then both paths on its inputs."""
    import synth_envs
    from pgmorl_b200 import kernels as K
    from pgmorl_b200.scalarization_methods import WeightedSumScalarization
    calls, real = [], K.select_greedy

    def spy(ep, cand, alpha, num_tasks, **kw):
        calls.append((np.array(ep, dtype=np.float64), np.array(cand, dtype=np.float64), alpha, num_tasks))
        return real(ep, cand, alpha, num_tasks, **kw)
    monkeypatch.setattr(K, "select_greedy", spy)
    args, graph, pop, ep = synth_envs.make_selection_state(3, 420, 500)
    np.random.seed(0)
    pop.prediction_guided_selection(args, 0, ep, graph, WeightedSumScalarization(num_objs=3, weights=np.ones(3) / 3))
    monkeypatch.setattr(K, "select_greedy", real)
    (c,) = [c for c in calls if c[3] == args.num_tasks]
    assert len(c[1]) > 2500 and len(c[0]) == 500
    _both_paths(*c)
    _metrics_both(c[0])


@pytest.mark.gpu
def test_paths_agree_on_2000_point_fronts():
    rng = np.random.RandomState(5)
    ep = _sphere(rng, 2000)
    cand = np.vstack([_sphere(rng, 60, 80.5), rng.uniform(0, 60, (30, 3)), ep[rng.choice(2000, 10)]])
    _both_paths(ep, cand, 1e6, 8)
    _both_paths(ep, cand, 0.0, 3)
    _metrics_both(ep)
    _metrics_both(np.vstack([ep, _sphere(rng, 1900, 79.0)]))          # dominated points and 3 900 of them


@pytest.mark.gpu
def test_paths_agree_on_edge_sets():
    rng = np.random.RandomState(6)
    ep = _sphere(rng, 25, 10.0)
    tol = ep[7] + np.array([4e-6, -3e-6, 9e-6])                       # within update_ep's 1e-5 of an archive point
    cand = np.vstack([rng.uniform(0, 12, (8, 3)), ep[3], ep[3], tol, [4.0, -1.0, 8.0], [-0.0, 2.0, 3.0],
                      [9.0, 9.0, 9.0], ep[10] * 0.5])
    _both_paths(np.zeros((0, 3)), cand, 1e6, 4)                       # empty archive
    best = _both_paths(ep, cand[:2], 1e6, 4)[0]                       # fewer candidates than tasks
    assert best.tolist()[2:] == [-1, -1]
    _both_paths(ep, cand, 1e6, 6)
    _both_paths(ep, cand[::-1].copy(), 1.0, 6)
    _both_paths(ep, cand[[11, 12, 14]], 1.0, 3)                       # negative coordinate, dominated candidates
    dup = rng.randint(0, 4, (40, 3)).astype(np.float64)               # ties and duplicates everywhere
    _both_paths(dup[:15], dup[15:], 1.0, 6)
    _both_paths(dup[:15], dup[15:], 1e6, 6)
    for pts in _small_sets(np.random.RandomState(7)):
        _metrics_both(pts[(pts >= 0).all(axis=1)])


@pytest.mark.gpu
def test_paths_agree_on_the_fork_scorer(monkeypatch):
    """The fork's 2-objective scorer lifts the fronts to z = 1 and calls the 3-D select_greedy: with the global path
    forced it still reproduces the fork golden's every round."""
    import torch
    from tests.helpers import rebuild_selection_state
    from pgmorl_b200 import kernels as K
    real = K.select_greedy
    monkeypatch.setattr(K, "select_greedy", lambda *a, **kw: real(*a, force_global=True, **kw))
    z = np.load(os.path.join(GOLDEN, "selection_2d_fork.npz"))
    alpha = float(z["args_f"][0]); num_tasks = int(z["args"][0])
    torch.set_default_dtype(torch.float64)
    try:
        for g in range(int(z["meta"][1])):
            args, graph, pop, ep = rebuild_selection_state(z, g, 2)
            args.fork_scoring = True
            pred = z[f"g{g}_cand_pred"]
            best, hv, sp = pop._greedy_fork(z[f"g{g}_round0_vep"], pred, alpha, num_tasks)
            for r in range(num_tasks):
                assert np.array_equal(hv[r], z[f"g{g}_round{r}_hv"]), (g, r)
                assert np.array_equal(sp[r], z[f"g{g}_round{r}_sparsity"]), (g, r)
    finally:
        torch.set_default_dtype(torch.float32)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: correct past the old limits
# ---------------------------------------------------------------------------------------------------------------------
SIZES = [OLD_GREEDY_LIMIT + 1, OLD_METRICS_LIMIT + 1, 5000, 20000]


@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES)
def test_front_metrics_past_the_old_limits(n):
    from pgmorl_b200 import kernels as K
    rng = np.random.RandomState(n)
    pts = _sphere(rng, n)
    assert K.front_metrics(pts) == (round(hv3d_raw_fast(pts), 4), sparsity_fast(pts))
    ip = _int_plane(rng, n)
    rng.shuffle(ip)
    assert K.front_metrics(ip) == (float(hv3d_exact_int(ip)), sparsity_exact_int(ip))


def _check_greedy_vs_restated(oracle, ep, cand, alpha, num_tasks):
    from pgmorl_b200 import kernels as K
    best, hv, sp, front = K.select_greedy(ep, cand, alpha, num_tasks)
    ob, ohv, osp = oracle.greedy_select_3d(ep, cand, alpha, num_tasks)
    assert best.tolist() == ob + [-1] * (num_tasks - len(ob))
    for r in range(len(ohv)):
        assert np.array_equal(hv[r], ohv[r]), r
        assert np.array_equal(sp[r], osp[r]), r
    vep = [p for p in np.asarray(ep, dtype=np.float64)]
    for b in ob:
        vep = update_ep_fast(vep, cand[b])
    assert np.array_equal(front, np.array(vep).reshape(-1, 3))


@pytest.mark.gpu
@pytest.mark.parametrize("n,n_cand,rounds", [(OLD_GREEDY_LIMIT + 1, 24, 3), (OLD_METRICS_LIMIT + 1, 16, 2),
                                             (5000, 16, 2), (20000, 8, 2)])
def test_select_greedy_past_the_old_limits(restated_oracle, n, n_cand, rounds):
    rng = np.random.RandomState(n + 1)
    ep = _sphere(rng, n)
    k = n_cand // 3
    cand = np.vstack([_sphere(rng, k, 80.4), rng.uniform(0, 70, (n_cand - k - 2, 3)), ep[n // 2] + 4e-6,
                      [50.0, -1.0, 50.0]])
    _check_greedy_vs_restated(restated_oracle, ep, cand, 1e6, rounds)
    ip = _int_plane(rng, n)
    icand = np.vstack([ip[rng.choice(n, 2)] + 1.0, rng.randint(1, 120, (n_cand - 2, 3))]).astype(np.float64)
    _check_greedy_vs_restated(restated_oracle, ip, icand, 1.0, rounds)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the public interface
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_utils_and_hypervolume_on_a_5000_point_front():
    from pgmorl_b200 import utils
    from pgmorl_b200.hypervolume import InnerHyperVolume
    rng = np.random.RandomState(21)
    front = _sphere(rng, 5000)
    hv = round(hv3d_raw_fast(front), 4)
    assert utils.compute_hypervolume(front) == hv
    assert InnerHyperVolume(np.zeros(3)).compute(front) == hv
    assert utils.compute_sparsity(front) == sparsity_fast(front)
    for new in (_sphere(rng, 1, 80.3)[0], front[17], front[40] + 3e-6, np.array([1.0, -1.0, 2.0]), np.full(3, 60.0)):
        got = utils.update_ep(front, new)
        assert np.array_equal(np.array(got).reshape(-1, 3), np.array(update_ep_fast(front, new)).reshape(-1, 3))


@pytest.mark.gpu
def test_prediction_guided_selection_with_a_5000_point_archive(monkeypatch):
    import synth_envs
    from pgmorl_b200 import kernels as K
    from pgmorl_b200.scalarization_methods import WeightedSumScalarization
    calls, real = [], K.select_greedy

    def spy(ep, cand, alpha, num_tasks, **kw):
        out = real(ep, cand, alpha, num_tasks, **kw)
        calls.append((np.array(ep, dtype=np.float64), np.array(cand, dtype=np.float64), alpha, num_tasks, out))
        return out
    monkeypatch.setattr(K, "select_greedy", spy)
    args, graph, pop, ep = synth_envs.make_selection_state(3, 60, 5000)
    np.random.seed(0)
    elites, scals, predicted = pop.prediction_guided_selection(args, 0, ep, graph,
                                                              WeightedSumScalarization(num_objs=3, weights=np.ones(3) / 3))
    assert len(elites) == args.num_tasks
    (c,) = [c for c in calls if c[3] == args.num_tasks]
    e, cand, alpha, _, (best, hv, sp, _) = c
    assert len(e) == 5000 and len(cand) >= 4 * 60
    for i in np.random.RandomState(1).choice(len(cand), 12, replace=False):
        front = update_ep_fast(e, cand[i])
        assert hv[0][i] == round(hv3d_raw_fast(front), 4) and sp[0][i] == sparsity_fast(front), i
    assert best[0] == int(np.argmax(hv[0] - alpha * sp[0]))
    assert np.array_equal(predicted[0], cand[best[0]])


@pytest.mark.gpu
def test_fork_scoring_selection_over_a_3000_point_archive(restated_oracle):
    import torch
    import synth_envs
    from pgmorl_b200.scalarization_methods import WeightedSumScalarization
    torch.set_default_dtype(torch.float64)
    try:
        args, graph, pop, ep = synth_envs.make_selection_state(2, 30, 3000, fork_scoring=True)
        np.random.seed(0)
        elites, _, predicted = pop.prediction_guided_selection(args, 0, ep, graph,
                                                               WeightedSumScalarization(num_objs=2, weights=np.ones(2) / 2))
    finally:
        torch.set_default_dtype(torch.float32)
    assert len(elites) == args.num_tasks
    cand = np.asarray(pop.last_candidates.prediction, dtype=np.float64)
    hv, sp = np.asarray(pop.last_hv), np.asarray(pop.last_sparsity)
    vep = [np.asarray(p, dtype=np.float64) for p in ep.obj_batch]
    for i in np.random.RandomState(2).choice(len(cand), 10, replace=False):
        front = restated_oracle.update_ep(vep, cand[i])
        assert hv[0][i] == restated_oracle.hv2d_inner(front) and sp[0][i] == sparsity_fast(front), i


# ---------------------------------------------------------------------------------------------------------------------
# GPU: up to morl.run
# ---------------------------------------------------------------------------------------------------------------------
def _run_3d(save_dir):
    import synth_envs
    from pgmorl_b200 import mopg, morl
    from pgmorl_b200.layout import NetDims
    d = NetDims(17, 6, 3)
    args = synth_envs.run_args_2d(str(save_dir))
    args.obj_num, args.delta_weight, args.pbuffer_num, args.sparsity = 3, 0.5, 6, 1e6
    mopg.set_env_hooks(
        make_vec_envs=lambda **kw: synth_envs.SeededReplayVecEnv(d, args.num_steps, args.num_processes, [1.3, 0.7, 1.0],
                                                                 base_seed=500),
        gym_make=lambda name: synth_envs.ToyEvalEnv(d))
    return morl.run(args, device="cuda")


def _files(root):
    out = {}
    for dirpath, _, names in os.walk(root):
        for name in names:
            if name.endswith(".txt"):
                path = os.path.join(dirpath, name)
                out[os.path.relpath(path, root)] = open(path, "rb").read()
    return out


@pytest.mark.gpu
def test_whole_run_on_the_global_path_writes_the_same_files(tmp_path, monkeypatch):
    from pgmorl_b200 import kernels as K
    _run_3d(tmp_path / "default")
    real_sel, real_met = K.select_greedy, K.front_metrics
    used = []

    def sel(ep, cand, alpha, num_tasks):
        used.append(np.asarray(cand).shape[1])
        return real_sel(ep, cand, alpha, num_tasks, force_global=True)
    monkeypatch.setattr(K, "select_greedy", sel)
    monkeypatch.setattr(K, "front_metrics", lambda pts: real_met(pts, force_global=True))
    _run_3d(tmp_path / "global")
    assert used and set(used) == {3}
    a, b = _files(tmp_path / "default"), _files(tmp_path / "global")
    assert a and any("ep" in k for k in a)
    assert a == b
