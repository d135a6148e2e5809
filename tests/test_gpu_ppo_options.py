"""The non-default PPO options on the GPU: every return branch of compute_returns in K2 (both kernels) and the unclipped
value loss in every K3 kernel family, against the float64 restatements of tests/ppo_options_ref.py, and through the
public API (RolloutStorage, PPO, MOPG_worker, mopg_population_update, morl.run). Tolerances as in test_gpu_kernels.py
(norm-wise, max|a-b| <= tol * max|b| per tensor)."""
import queue
import threading

import numpy as np
import pytest
import torch

import ppo_options_ref as ref
import synth_envs
from oracle import mopg_oracle as orc
from pgmorl_b200 import synthetic
from pgmorl_b200.layout import NetDims
from tests.helpers import rel_err
from tests.test_gpu_kernels import DIMS, TAIL0, TAIL2, TAILBP, TAILEP, TAILGL, TAILMC, TAILNB, make_case

pytestmark = pytest.mark.gpu


def dev(x, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(x)).to(device="cuda", dtype=dtype).contiguous()


# ---------------------------------------------------------------------------------------------------------------------
# K2
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("use_gae,use_ptl", ref.BRANCHES)
@pytest.mark.parametrize("P,T,N,M", [(3, 2048, 4, 1), (3, 2048, 4, 2), (3, 2048, 4, 3),    # segmented kernel
                                     (2, 1030, 3, 2),                                       # segmented, ragged last segment
                                     (3, 2048, 4, 5),                                       # M > 4: one warp per column
                                     (70, 300, 4, 2), (70, 200, 2, 3), (2, 7, 1, 1), (4, 50, 4, 5)])
def test_k2_return_branches_match_oracle(use_gae, use_ptl, P, T, N, M):
    from pgmorl_b200 import kernels as K
    rng = np.random.RandomState(T + M)
    rewards = rng.randn(P, T, N, M)
    value = rng.randn(P, T + 1, N, M) * 3
    masks = (rng.uniform(size=(P, T + 1, N)) > 0.03).astype(np.float32)
    bad = (rng.uniform(size=(P, T + 1, N)) > 0.03).astype(np.float32)
    masks[:, T, 0] = 0.0; bad[:, T, -1] = 0.0                          # zeros in the bootstrap slot
    boot = rng.randn(P, N, M) * 3
    weights, obj_var = rng.dirichlet(np.ones(M), P), rng.uniform(0.5, 2.0, (P, M))
    args = (dev(rewards), dev(value), dev(masks), dev(bad), 0.995, 0.95)
    kw = dict(use_gae=use_gae, use_proper_time_limits=use_ptl, weights=dev(weights), obj_var=dev(obj_var))
    ret, adv = K.returns_adv(*args, boot=None if use_gae else dev(boot), **kw)
    # boot = NULL means value row T; an explicit copy of that row gives the same bits
    r_row, a_row = K.returns_adv(*args, **kw)
    r_exp, a_exp = K.returns_adv(*args, boot=dev(value[:, T]), **kw)
    if use_gae and use_ptl:      # branch A through the new entry point == pgm_gae_adv_f32, bit for bit
        r_old, a_old = K.gae_adv(*args, weights=dev(weights), obj_var=dev(obj_var))
    torch.cuda.synchronize()
    assert torch.equal(r_row, r_exp) and torch.equal(a_row, a_exp)
    if use_gae and use_ptl:
        assert torch.equal(ret, r_old) and torch.equal(adv, a_old)
    f64 = lambda a: dev(a).cpu().numpy().astype(np.float64)            # the kernel saw float32-rounded inputs
    rw, v32, b32, mk, bd = f64(rewards), f64(value), f64(boot), masks.astype(np.float64), bad.astype(np.float64)
    for p in range(P):
        r = ref.returns_np(rw[p], v32[p], mk[p], bd[p], 0.995, 0.95, use_gae, use_ptl,
                           next_value=None if use_gae else b32[p])
        a = orc.advantages(r, v32[p], weights[p], obj_var[p])
        assert rel_err(ret[p].cpu().numpy(), r) < 1e-5          # returns: 1e-5
        assert rel_err(adv[p].cpu().numpy(), a) < 1e-4          # normalised advantage: 1e-4


# ---------------------------------------------------------------------------------------------------------------------
# K3
# ---------------------------------------------------------------------------------------------------------------------
def _unclipped_inputs(d, P, T, N, seed):
    """PPO inputs whose old value predictions sit far enough from the current ones that the clip of the value loss is
    active for most (row, objective) elements: the clipped and unclipped losses then differ."""
    params, traj, eps, perm, weights, obj_var, out = make_case(d, P, T, N, seed)
    rng = np.random.RandomState(seed + 1)
    cur = params + rng.randn(*params.shape) * 0.02
    S = T * N
    pk = dict(obs=traj["obs"].reshape(P, (T + 1) * N, d.obs),
              action=np.stack([r["action"].reshape(S, d.act) for r in out]),
              logp=np.stack([r["logp"].reshape(S) for r in out]),
              value=np.stack([r["value"].reshape((T + 1) * N, d.obj) for r in out]) + rng.randn(P, (T + 1) * N, d.obj) * 0.4,
              returns=np.stack([r["returns"].reshape(S, d.obj) for r in out]),
              adv=np.stack([r["adv"].reshape(S) for r in out]))
    for p in range(P):
        v, _, _ = orc.forward(orc.Net(cur[p].copy(), d.obs, d.act, d.obj), pk["obs"][p][:S].astype(np.float64))
        assert (np.abs(v - pk["value"][p][:S]) > 0.2).mean() >= 0.2
    return cur, pk, perm


K3_CASES = [("walker", c) for c in (1, 2, 4, 8, 16, 32, 64)] + [("hopper3", c) for c in (1, 2, 4, 8, 16, 32, 64)] + \
           [("humanoid", c) for c in (8, 32, 64, 128)] + \
           [("s45_16_3", c) for c in (2, 4, 8)] + [("s60_6_2", 16), ("ant", 2), ("s33_17_2", 1)]   # generic DB, TM = 2 fallback, big


@pytest.mark.parametrize("name,cluster", K3_CASES)
def test_k3_unclipped_gradient_matches_oracle(name, cluster):
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    P, T, N, mb = (2, 64, 8, 384) if name == "humanoid" else (2, 64, 4, 200)
    cur, pk, _ = _unclipped_inputs(d, P, T, N, seed=31)
    S = T * N
    idx = np.random.RandomState(0).permutation(S)[:mb]
    hyper = K.PpoHyper(entropy_coef=0.01)
    ins = (dev(cur), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]), dev(pk["returns"]),
           dev(pk["adv"]), dev(idx, torch.int32), d)
    g, losses = K.ppo_grad(*ins, hyper=hyper, cluster=cluster, clipped_value_loss=False)
    g_clip, _ = K.ppo_grad(*ins, hyper=hyper, cluster=cluster)
    torch.cuda.synchronize()
    for p in range(P):
        net = orc.Net(cur[p].copy(), d.obs, d.act, d.obj)
        rows = lambda a: a[p][:S][idx].astype(np.float64)
        gref, lref = ref.ppo_grad_np(net, rows(pk["obs"]), rows(pk["action"]), rows(pk["logp"]), rows(pk["value"]),
                                     rows(pk["returns"]), rows(pk["adv"]), ecoef=0.01, clipped_value_loss=False)
        gcl, _ = orc.ppo_grad(net, rows(pk["obs"]), rows(pk["action"]), rows(pk["logp"]), rows(pk["value"]),
                              rows(pk["returns"]), rows(pk["adv"]), ecoef=0.01)
        assert rel_err(gref, gcl) > 10 * 5e-5                  # not vacuous: the two losses have different gradients
        assert rel_err(g[p].cpu().numpy(), gref) < 5e-5
        assert rel_err(g_clip[p].cpu().numpy(), gcl) < 5e-5
        assert rel_err(losses[p].cpu().numpy(), np.array(lref)) < 1e-4


@pytest.mark.parametrize("name,cluster", K3_CASES)
def test_k3_unclipped_update_matches_oracle(name, cluster):
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    P, T, N, B = (2, 48, 8, 3) if name == "humanoid" else (2, 64, 4, 4)
    cur, pk, perm = _unclipped_inputs(d, P, T, N, seed=37)
    rng = np.random.RandomState(2)
    m0, v0 = rng.randn(P, d.n_par) * 1e-3, rng.rand(P, d.n_par) * 1e-5
    step0, lr = np.array([0, 7], dtype=np.int32), np.array([3e-4, 2.5e-4])
    gp, gm, gv, gstep = dev(cur), dev(m0), dev(v0), dev(step0, torch.int32)
    losses = K.ppo_update(gp, gm, gv, gstep, dev(lr, torch.float64), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]),
                          dev(pk["value"]), dev(pk["returns"]), dev(pk["adv"]), dev(perm[None], torch.int32), B, d,
                          cluster=cluster, clipped_value_loss=False)
    torch.cuda.synchronize()
    for p in range(P):
        flat, m, v = (dev(t[p]).cpu().numpy().astype(np.float64) for t in (cur, m0, v0))
        step, lref = ref.ppo_update_np(flat, m, v, int(step0[p]), lr[p], (d.obs, d.act, d.obj),
                                       pk["obs"][p].reshape(T + 1, N, d.obs).astype(np.float64),
                                       pk["action"][p].reshape(T, N, -1), pk["logp"][p].reshape(T, N),
                                       pk["value"][p].reshape(T + 1, N, -1), pk["returns"][p].reshape(T, N, -1),
                                       pk["adv"][p].reshape(T, N), perm, B, clipped_value_loss=False)
        assert int(gstep[p]) == step
        assert rel_err(gp[p].cpu().numpy(), flat) < 1e-5          # parameters
        assert rel_err(gm[p].cpu().numpy(), m) < 1e-4 and rel_err(gv[p].cpu().numpy(), v) < 1e-4
        assert rel_err(losses[p].cpu().numpy(), np.array(lref)) < 1e-4


@pytest.mark.parametrize("cluster", [4, 8, 16])
@pytest.mark.parametrize("name,P,T,N,B", [("walker", 3, 64, 4, 4), ("hopper3", 2, 48, 2, 3)])
def test_k3_unclipped_step_tails_bit_identical(name, P, T, N, B, cluster):
    """test_k3_step_tails_bit_identical with the unclipped value loss"""
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    cur, pk, perm = _unclipped_inputs(d, P, T, N, seed=17)
    hyper = K.PpoHyper(entropy_coef=0.01)
    lr = dev(np.array([3e-4, 2.5e-4, 1e-4][:P]), torch.float64)
    out = []
    for cl in (cluster, cluster | TAIL0, cluster | TAIL2, cluster | TAILMC, cluster | TAILGL, cluster | TAILBP,
               cluster | TAILNB, cluster | TAILEP):
        gp, gm, gv = dev(cur), torch.zeros(P, d.n_par, device="cuda"), torch.zeros(P, d.n_par, device="cuda")
        gstep = torch.zeros(P, dtype=torch.int32, device="cuda")
        losses = K.ppo_update(gp, gm, gv, gstep, lr, dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]),
                              dev(pk["returns"]), dev(pk["adv"]), dev(perm[None], torch.int32), B, d, hyper=hyper, cluster=cl,
                              clipped_value_loss=False)
        idx = np.random.RandomState(0).permutation(T * N)[:T * N // B]
        g, gl = K.ppo_grad(dev(cur), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]),
                           dev(pk["returns"]), dev(pk["adv"]), dev(idx, torch.int32), d, hyper=hyper, cluster=cl,
                           clipped_value_loss=False)
        torch.cuda.synchronize()
        out.append((gp, gm, gv, gstep, losses, g, gl))
    for other in out[1:]:
        for x, y in zip(out[0], other):
            assert torch.equal(x, y)


# ---------------------------------------------------------------------------------------------------------------------
# API
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("use_gae,use_ptl", ref.BRANCHES)
def test_rollout_storage_compute_returns_all_branches(use_gae, use_ptl):
    from pgmorl_b200.a2c_ppo_acktr.storage import RolloutStorage
    T, N, M = 40, 4, 3
    rng = np.random.RandomState(9)
    st = RolloutStorage(T, N, (5,), synth_envs._Box(2), 1, obj_num=M)
    st.rewards.copy_(dev(rng.randn(T, N, M)))
    st.value_preds.copy_(dev(rng.randn(T + 1, N, M)))
    st.masks.copy_(dev((rng.uniform(size=(T + 1, N, 1)) > 0.1)))
    st.bad_masks.copy_(dev((rng.uniform(size=(T + 1, N, 1)) > 0.1)))
    before = st.value_preds.clone()
    nv = dev(rng.randn(N, M))
    st.compute_returns(nv, use_gae, 0.99, 0.9, use_ptl)
    torch.cuda.synchronize()
    if use_gae:
        assert torch.equal(st.value_preds[-1], nv)
    else:                        # n-step: bootstrap in returns[-1], value_preds untouched (storage.py:95-116)
        assert torch.equal(st.value_preds, before) and torch.equal(st.returns[-1], nv)
    f = lambda t: t.cpu().numpy().astype(np.float64)
    want = ref.returns_np(f(st.rewards), f(st.value_preds), f(st.masks)[..., 0], f(st.bad_masks)[..., 0], 0.99, 0.9,
                          use_gae, use_ptl, next_value=f(nv))
    assert rel_err(f(st.returns[:-1]), want) < 1e-5


def _replay_args(T, N, E, B, use_gae, use_ptl):
    from types import SimpleNamespace
    return SimpleNamespace(env_name="replay", seed=0, num_processes=N, gamma=0.995, obj_rms=True, ob_rms=True, num_steps=T,
                           obj_num=2, num_env_steps=10 * T * N, use_linear_lr_decay=True, lr_decay_ratio=1.0, lr=3e-4,
                           use_gae=use_gae, gae_lambda=0.95, use_proper_time_limits=use_ptl, rl_log_interval=0,
                           update_iter=1, eval_num=1, raw=True, ppo_epoch=E, num_mini_batch=B)


def _task(d, seed, weights, E, B, clipped):
    from pgmorl_b200.a2c_ppo_acktr.algo import PPO
    from pgmorl_b200.a2c_ppo_acktr.model import Policy
    from pgmorl_b200.sample import Sample, Task
    from pgmorl_b200.scalarization_methods import WeightedSumScalarization
    torch.manual_seed(seed)
    pol = Policy((d.obs,), synth_envs._Box(d.act), base_kwargs={"layernorm": False}, obj_num=d.obj)
    agent = PPO(pol, 0.2, E, B, 0.5, 0.0, lr=3e-4, eps=1e-5, max_grad_norm=0.5, use_clipped_value_loss=clipped)
    sample = Sample({"ob_rms": None, "ret_rms": None, "obj_rms": None}, pol, agent, objs=np.zeros(d.obj), optgraph_id=-1)
    return Task(sample, WeightedSumScalarization(num_objs=d.obj, weights=weights))


OPTIONS = [(False, True, True), (True, False, True), (False, False, True), (True, True, False)]   # + unclipped value loss


@pytest.mark.parametrize("use_gae,use_ptl,clipped", OPTIONS)
def test_worker_and_population_update_match_the_torch_port(tmp_path, use_gae, use_ptl, clipped):
    """One MOPG iteration on replayed trajectories with a non-default option: MOPG_worker (RolloutStorage.compute_returns +
    PPO.update) against the float64 torch port (1e-4), and mopg_population_update -- host-normalised and with the
    normalisation on the device (K6) -- against MOPG_worker (1e-4)."""
    from pgmorl_b200 import mopg
    from pgmorl_b200.sample import Task
    d = NetDims(17, 6, 2)
    T, N, E, B, P, j = 32, 4, 2, 4, 3, 1
    args = _replay_args(T, N, E, B, use_gae, use_ptl)
    traj = {k: v.numpy() for k, v in synthetic.make_trajectories(P, T, N, d, seed=40, p_done=0.08).items()}
    traj["bad_masks"][:, T, 1] = 0.0
    obj_var = np.array([1.3, 0.7])
    wts = [np.array([0.2, 0.8]), np.array([0.5, 0.5]), np.array([0.9, 0.1])]
    tasks = [_task(d, 1000 + p, wts[p], E, B, clipped) for p in range(P)]
    init = [t.sample.actor_critic.flat.cpu().numpy().astype(np.float64) for t in tasks]
    order = iter(range(10 ** 6))

    def replay_env(**kw):                     # the environments of task i replay trajectory i
        i = next(order) % P
        return synth_envs.ReplayVecEnv({k: v[i] for k, v in traj.items()}, d, obj_var)

    mopg.set_env_hooks(make_vec_envs=replay_env, gym_make=lambda name: synth_envs.ToyEvalEnv(d), make_raw_vec_envs=False)
    worker = []
    for p in range(P):
        order = iter([p] * 10)
        q, ev = queue.Queue(), threading.Event()
        ev.set()
        mopg.MOPG_worker(args, p, _task(d, 1000 + p, wts[p], E, B, clipped), torch.device("cuda"), j, 1, 0.0, q, ev)
        worker.append(q.get_nowait()["offspring_batch"][0].actor_critic.flat.cpu().numpy().astype(np.float64))
    from oracle.mopg_torch_port import PortPolicy
    for p in range(P):
        pol = PortPolicy(init[p], d.obs, d.act, d.obj)
        opt = torch.optim.Adam(pol.ordered(), lr=3e-4, eps=1e-5)
        lr = synthetic.linear_lr(3e-4, j, 1.0, 10)
        ref.mopg_iteration_torch(pol, opt, {k: v[p] for k, v in traj.items()}, j, lr, wts[p], obj_var, ppo_epoch=E,
                                 num_mini_batch=B, use_gae=use_gae, use_proper_time_limits=use_ptl,
                                 clipped_value_loss=clipped)
        assert rel_err(worker[p], pol.flat()) < 1e-4
    # the population path, host-normalised replay environments
    order = iter(range(10 ** 6))
    pop = mopg.mopg_population_update(args, tasks, torch.device("cuda"), j, 1)
    for p in range(P):
        assert rel_err(pop[p][0].actor_critic.flat.cpu().numpy(), worker[p]) < 1e-4
    # ... and with the running normalisation on the device: identical to the host-normalised loop (test_gpu_vecnorm.py)
    from pgmorl_b200 import warm_up
    from tests.test_gpu_vecnorm import _HostNormalised, _RawEnv
    args = synth_envs.run_args_2d(str(tmp_path), T=T, N=N)
    args.use_gae, args.use_proper_time_limits = use_gae, use_ptl
    mopg.set_env_hooks(make_vec_envs=lambda **kw: _HostNormalised(_RawEnv(N, d.obs, d.obj), d, args.gamma))
    torch.manual_seed(0)
    elites, scals = warm_up.initialize_warm_up_batch(args, "cuda")
    for e in elites:
        e.agent.use_clipped_value_loss = clipped
    host = mopg.mopg_population_update(args, [Task(e, s) for e, s in zip(elites[:3], scals[:3])], torch.device("cuda"), 0, 2)
    mopg.set_env_hooks(make_raw_vec_envs=lambda **kw: _RawEnv(N, d.obs, d.obj))
    try:
        fused = mopg.mopg_population_update(args, [Task(e, s) for e, s in zip(elites[:3], scals[:3])], torch.device("cuda"), 0, 2)
    finally:
        mopg.set_env_hooks(make_raw_vec_envs=False)
    for hs, fs in zip(host, fused):
        assert len(hs) == len(fs) == 2
        for a, b in zip(hs, fs):
            assert torch.equal(a.actor_critic.flat, b.actor_critic.flat)
            assert torch.equal(a.agent.optimizer.exp_avg_sq, b.agent.optimizer.exp_avg_sq)


def test_population_cache_is_keyed_by_the_options():
    """a shard built for one return branch / value loss is never reused for another"""
    from pgmorl_b200 import mopg
    from pgmorl_b200._lib import PpoHyper
    d = NetDims(17, 6, 2)
    pops = []
    for use_gae, use_ptl, clipped in OPTIONS[:3] + [(True, True, True)]:
        args = _replay_args(16, 4, 1, 2, use_gae, use_ptl)
        pop = mopg._population(d, 2, args, PpoHyper(), torch.device("cuda"), 0, clipped)["pop"]
        assert (pop.use_gae, pop.use_proper_time_limits, pop.clipped_value_loss) == (use_gae, use_ptl, clipped)
        pops.append(pop)
    pop = mopg._population(d, 2, args, PpoHyper(), torch.device("cuda"), 0, False)["pop"]
    assert pop.clipped_value_loss is False and all(pop is not q for q in pops)
    assert mopg._population(d, 2, args, PpoHyper(), torch.device("cuda"), 0, True)["pop"] is pops[-1]   # cache hit
    assert len({id(q) for q in pops}) == len(pops)


def test_run_without_gae_reaches_the_kernels(tmp_path):
    """a two-generation morl.run with use_gae=False completes, and its offspring differ from the use_gae=True run"""
    import os
    from pgmorl_b200 import mopg, morl
    d = NetDims(17, 6, 2)
    out = {}
    for use_gae in (True, False):
        save = str(tmp_path / f"gae{int(use_gae)}")
        args = synth_envs.run_args_2d(save)
        args.use_gae = use_gae
        mopg.set_env_hooks(
            make_vec_envs=lambda **kw: synth_envs.SeededReplayVecEnv(d, args.num_steps, args.num_processes, [1.3, 0.7],
                                                                     base_seed=500),
            gym_make=lambda name: synth_envs.ToyEvalEnv(d))
        ep, population, opt_graph, timings = morl.run(args, device="cuda")
        assert len(timings) == 3
        out[use_gae] = open(os.path.join(save, "2", "elites", "offsprings.txt")).read()
    assert out[True] != out[False]
