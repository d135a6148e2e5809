"""Policies of hidden width 32 and 128 on the device: K1 (every action mode, trajectory and per-step), K3's raw gradient and
update on the generic cluster kernel, the refusals at these widths, the _h entry points at 64, and whole MOPG iterations
up to morl.run.

The float64 pin is the numpy oracle at width H (oracle/mopg_oracle.Net takes it; tests/hidden_ref.py repeats its update
loop at width H), which tests/test_oracle_hidden.py checks against the torch port. Gates are the ones of the width-64
tests (tests/test_gpu_kernels.py, tests/test_gpu_shapes.py)."""
import ctypes
import os
import pickle
import queue
import threading

import numpy as np
import pytest
import torch

import hidden_ref
import ppo_options_ref as ref
import synth_envs
from oracle import mopg_oracle as orc
from pgmorl_b200 import synthetic
from pgmorl_b200._lib import PgmError
from pgmorl_b200.layout import ENV_SHAPES, NetDims, param_layout
from tests.helpers import rel_err
from tests.test_gpu_kernels import dev

pytestmark = pytest.mark.gpu

WIDTHS = (32, 128)
SHAPES = dict(ENV_SHAPES, s33_17_2=NetDims(33, 17, 2))   # (33,17,2): A > 16, the generic kernel's wide-head variant


def _fits(name, H):
    return not (name == "humanoid" and H == 128)        # Humanoid's W1 alone is 194 KB at width 128


def _dims(name, H):
    d = SHAPES[name]
    return NetDims(d.obs, d.act, d.obj, H)


def _params(d, P, seed):
    rng = np.random.RandomState(seed)
    params = np.stack([synthetic.init_policy_flat(d, seed=seed * 100 + p).numpy() for p in range(P)])
    params[:, -d.act:] = rng.uniform(-0.5, 0.3, (P, d.act))
    return params


def _net(d, flat):
    return orc.Net(np.asarray(flat, dtype=np.float64).copy(), d.obs, d.act, d.obj, d.hidden)


# ------------------------------------------------------------------------------------------------------------------ K1
K1_CASES = [(n, H, T) for H in WIDTHS for n in SHAPES if n != "s33_17_2" and _fits(n, H) for T in (40,)] + \
           [("walker2d", H, 300) for H in WIDTHS] + [("hopper3", H, 300) for H in WIDTHS]   # >= 1024 rows: FFMA, not tcgen05


@pytest.mark.parametrize("name,H,T", K1_CASES)
def test_k1_all_modes_match_oracle(name, H, T):
    from pgmorl_b200 import kernels as K
    d = _dims(name, H)
    P, N = 2, 4
    params = _params(d, P, seed=3)
    traj = {k: v.numpy() for k, v in synthetic.make_trajectories(P, T, N, d, seed=3).items()}
    eps, _ = synthetic.host_rng_streams(3, T, N, d.act, 1)
    eps = eps.numpy()
    obs = dev(traj["obs"]).reshape(P, (T + 1) * N, d.obs)
    gp = dev(params)
    value, action, logp = K.policy_forward(gp, obs, d, eps=dev(eps).reshape(1, T * N, d.act), rows_a=T * N)
    v_det, a_det, lp_det = K.policy_forward(gp, obs, d, mode=K.ACT_DETERMINISTIC)
    torch.cuda.synchronize()
    for p in range(P):
        net = _net(d, params[p])
        v, a, lp = orc.rollout(net, traj["obs"][p].astype(np.float64), eps)
        # FP32 forward of a 3-layer MLP: 2e-5 norm-wise
        assert rel_err(value[p].cpu().numpy().reshape(T + 1, N, -1), v) < 2e-5
        assert rel_err(action[p].cpu().numpy().reshape(T, N, -1), a) < 2e-5
        assert rel_err(logp[p].cpu().numpy().reshape(T, N), lp) < 2e-5
        vv, mean, _ = orc.forward(net, traj["obs"][p].reshape(-1, d.obs).astype(np.float64))
        assert rel_err(a_det[p].cpu().numpy(), mean) < 2e-5 and rel_err(v_det[p].cpu().numpy(), vv) < 2e-5
        assert rel_err(lp_det[p].cpu().numpy(), orc.log_prob(net, mean, mean)) < 2e-5
    given = action.contiguous()
    _, _, lp_ev = K.policy_forward(gp, obs, d, action=given, mode=K.ACT_EVALUATE, rows_a=T * N)
    v0, _, _ = K.policy_forward(gp, obs, d, rows_a=0, mode=K.ACT_DETERMINISTIC)
    torch.cuda.synchronize()
    assert rel_err(lp_ev.cpu().numpy(), logp.cpu().numpy()) < 2e-5
    assert torch.equal(v0, v_det)


@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("staged", [True, False])
def test_k1_per_step_matches_oracle(H, staged):
    """pgm_policy_step_h_f32: one environment step of every task written into time slot t of the rollout buffers"""
    from pgmorl_b200 import kernels as K
    d = _dims("ant", H)
    P, N, T, t = 3, 8, 5, 2
    params = _params(d, P, seed=8)
    rng = np.random.RandomState(4)
    x = rng.randn(P, N, d.obs)
    eps = rng.randn(1, N, d.act)
    obs_buf = torch.zeros(P, (T + 1) * N, d.obs, device="cuda")
    if not staged:
        obs_buf[:, t * N:(t + 1) * N] = dev(x)
    value_buf = torch.zeros(P, (T + 1) * N, d.obj, device="cuda")
    action_buf = torch.zeros(P, T * N, d.act, device="cuda")
    logp_buf = torch.zeros(P, T * N, device="cuda")
    act_out = torch.zeros(P, N, d.act, device="cuda")
    ctl = torch.tensor([t, 1], dtype=torch.int32, device="cuda")
    K.policy_step(dev(params), ctl, dev(x) if staged else None, dev(eps), obs_buf, value_buf, action_buf, logp_buf,
                  act_out, N, d)
    torch.cuda.synchronize()
    for p in range(P):
        v, a, lp = orc.rollout(_net(d, params[p]), np.concatenate([x[p][None], x[p][None]]), eps)
        rows = slice(t * N, (t + 1) * N)
        assert rel_err(value_buf[p, rows].cpu().numpy(), v[0]) < 2e-5
        assert rel_err(action_buf[p, rows].cpu().numpy(), a[0]) < 2e-5
        assert rel_err(logp_buf[p, rows].cpu().numpy(), lp[0]) < 2e-5
        assert torch.equal(act_out[p], action_buf[p, rows])
        assert rel_err(obs_buf[p, rows].cpu().numpy(), x[p]) < 1e-7


# ------------------------------------------------------------------------------------------------------- K3 gradient
def _grad_inputs(d, P, mb, seed):
    rng = np.random.RandomState(seed)
    S = 4 * mb
    params = _params(d, P, seed)
    cur = params + rng.randn(*params.shape) * 0.02
    obs = rng.randn(P, S, d.obs)
    act = rng.randn(P, S, d.act)
    value = np.stack([orc.forward(_net(d, params[p]), obs[p])[0] for p in range(P)])
    pk = dict(obs=obs, action=act, logp=rng.randn(P, S) * 0.3 - 6.0, value=value + rng.randn(P, S, d.obj) * 0.4,
              returns=value + rng.randn(P, S, d.obj), adv=rng.randn(P, S))
    return cur, pk, rng.permutation(S)[:mb]


GRAD_CASES = [(n, H, c) for H in WIDTHS for n in ("walker2d", "ant", "humanoid", "s33_17_2") if _fits(n, H)
              for c in (2, 4, 8, 16, 0)]


@pytest.mark.parametrize("vu", [False, True])
@pytest.mark.parametrize("name,H,cluster", GRAD_CASES)
def test_k3_gradient_per_tensor(name, H, cluster, vu):
    from pgmorl_b200 import kernels as K
    d = _dims(name, H)
    P, mb = 2, 256
    cur, pk, idx = _grad_inputs(d, P, mb, seed=41)
    g, losses = K.ppo_grad(dev(cur), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]),
                           dev(pk["returns"]), dev(pk["adv"]), dev(idx, torch.int32), d,
                           hyper=K.PpoHyper(entropy_coef=0.01), cluster=cluster, clipped_value_loss=not vu)
    torch.cuda.synchronize()
    g, losses = g.cpu().numpy(), losses.cpu().numpy()
    layout, _ = param_layout(d)
    for p in range(P):
        f = lambda a: a[p][idx].astype(np.float64)
        gref, lref = ref.ppo_grad_np(_net(d, dev(cur[p]).cpu().numpy()), f(pk["obs"]), f(pk["action"]), f(pk["logp"]),
                                     f(pk["value"]), f(pk["returns"]), f(pk["adv"]), ecoef=0.01, clipped_value_loss=not vu)
        assert rel_err(losses[p], np.array(lref)) < 1e-4
        for tname, (off, shape) in layout.items():         # per tensor: 2e-5 (tests/test_gpu_shapes.py)
            n = int(np.prod(shape))
            assert rel_err(g[p][off:off + n], gref[off:off + n]) < 2e-5, (tname, rel_err(g[p][off:off + n], gref[off:off + n]))


# --------------------------------------------------------------------------------------------------------- K3 update
@pytest.mark.parametrize("name,H,P,cluster", [("walker2d", H, P, 0) for H in WIDTHS for P in (6, 40)] +
                         [("ant", H, 3, 2) for H in WIDTHS] + [("humanoid", 32, 2, 0)])
def test_k3_update_matches_oracle(name, H, P, cluster):
    from pgmorl_b200 import kernels as K
    d = _dims(name, H)
    T, N, B = 32, 4, 2
    params = _params(d, P, seed=13)
    traj = {k: v.numpy() for k, v in synthetic.make_trajectories(P, T, N, d, seed=13, p_done=0.05).items()}
    eps, perm = synthetic.host_rng_streams(13, T, N, d.act, 2)
    eps, perm = eps.numpy(), perm.numpy()
    rng = np.random.RandomState(2)
    S = T * N
    pk = {k: [] for k in ("action", "logp", "value", "returns", "adv")}
    for p in range(P):
        net = _net(d, params[p])
        value, action, logp = orc.rollout(net, traj["obs"][p].astype(np.float64), eps)
        ret = orc.gae_returns(traj["rewards"][p].astype(np.float64), value, traj["masks"][p].astype(np.float64),
                              traj["bad_masks"][p].astype(np.float64), 0.995, 0.95)
        adv = orc.advantages(ret, value, np.full(d.obj, 1.0 / d.obj), np.ones(d.obj))
        for k, v in zip(pk, (action, logp, value, ret, adv)):
            pk[k].append(v)
    pk = {k: np.stack(v) for k, v in pk.items()}
    cur = params + rng.randn(*params.shape) * 0.02
    m0, v0 = rng.randn(P, d.n_par) * 1e-3, rng.rand(P, d.n_par) * 1e-5
    step0 = np.resize(np.array([0, 7, 640], dtype=np.int32), P)
    lr = np.resize(np.array([3e-4, 2.5e-4, 1e-4]), P)
    gp, gm, gv, gstep = dev(cur), dev(m0), dev(v0), dev(step0, torch.int32)
    losses = K.ppo_update(gp, gm, gv, gstep, dev(lr, torch.float64), dev(traj["obs"]).reshape(P, (T + 1) * N, d.obs),
                          dev(pk["action"]).reshape(P, S, d.act), dev(pk["logp"]).reshape(P, S),
                          dev(pk["value"]).reshape(P, (T + 1) * N, d.obj), dev(pk["returns"]).reshape(P, S, d.obj),
                          dev(pk["adv"]).reshape(P, S), dev(perm[None], torch.int32), B, d, cluster=cluster)
    torch.cuda.synchronize()
    for p in range(P):
        flat = dev(cur[p]).cpu().numpy().astype(np.float64)
        m = dev(m0[p]).cpu().numpy().astype(np.float64)
        v = dev(v0[p]).cpu().numpy().astype(np.float64)
        f32 = lambda a: dev(a).cpu().numpy().astype(np.float64)
        step, lref = hidden_ref.ppo_update(flat, m, v, int(step0[p]), lr[p], d, f32(traj["obs"][p]), f32(pk["action"][p]),
                                           f32(pk["logp"][p]), f32(pk["value"][p]), f32(pk["returns"][p]),
                                           f32(pk["adv"][p]), perm, B)
        assert int(gstep[p]) == step
        assert rel_err(gp[p].cpu().numpy(), flat) < 1e-5       # parameters
        assert rel_err(gm[p].cpu().numpy(), m) < 1e-4          # Adam first moment
        assert rel_err(gv[p].cpu().numpy(), v) < 1e-4          # Adam second moment
        assert rel_err(losses[p].cpu().numpy(), np.array(lref)) < 1e-4


# ---------------------------------------------------------------------------------------------------------- refusals
@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("cluster", [1, 32, 64, 128])
def test_k3_refuses_kernels_built_for_width_64(H, cluster):
    from pgmorl_b200 import kernels as K
    d = _dims("walker2d", H)
    cur, pk, idx = _grad_inputs(d, 1, 64, seed=5)
    with pytest.raises(PgmError, match=f"hidden width {H}"):
        K.ppo_grad(dev(cur), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]), dev(pk["returns"]),
                   dev(pk["adv"]), dev(idx, torch.int32), d, cluster=cluster)


def test_humanoid_at_width_128_is_refused_by_k1_and_k3():
    from pgmorl_b200 import kernels as K
    d = _dims("humanoid", 128)
    params = dev(_params(d, 1, seed=2))
    obs = torch.randn(1, 64, d.obs, device="cuda")
    with pytest.raises(PgmError, match="shared memory at hidden width 128"):
        K.policy_forward(params, obs, d, mode=K.ACT_DETERMINISTIC)
    cur, pk, idx = _grad_inputs(d, 1, 64, seed=5)
    for cluster in (0, 2, 16):
        with pytest.raises(PgmError, match="of shared memory .*hidden width 128"):
            K.ppo_grad(dev(cur), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]),
                       dev(pk["returns"]), dev(pk["adv"]), dev(idx, torch.int32), d, cluster=cluster)
    torch.cuda.synchronize()                          # nothing was launched: the context is healthy
    assert torch.ones(1, device="cuda").item() == 1.0


@pytest.mark.parametrize("name,rows", [("walker2d", 40 * 4), ("walker2d", 300 * 4), ("humanoid", 150 * 8), ("ant", 300 * 4)])
def test_h_entry_points_at_64_equal_the_old_ones(name, rows):
    """the _h entry points at width 64 run what the functions without `hidden` run, bit for bit (forward, per-step,
    gradient at every plan family, update)"""
    from pgmorl_b200 import kernels as K
    from pgmorl_b200._lib import PpoHyper, check, lib, ptr
    d = ENV_SHAPES[name]
    P = 2
    gp = dev(_params(d, P, seed=6))
    obs = torch.randn(P, rows, d.obs, device="cuda")
    eps = torch.randn(1, rows, d.act, device="cuda")
    st = K._stream()
    outs = []
    for h in (None, 64):
        value = torch.empty(P, rows, d.obj, device="cuda"); act = torch.empty(P, rows, d.act, device="cuda")
        logp = torch.empty(P, rows, device="cuda")
        a = (ptr(gp), ptr(obs), ptr(eps), 1, ptr(act), ptr(value), ptr(logp), 0, P, rows, rows, d.obs, d.act, d.obj)
        check(lib().pgm_policy_forward_f32(*a, st) if h is None else lib().pgm_policy_forward_h_f32(*a, h, st))
        outs.append((value, act, logp))
    for x, y in zip(*outs):
        assert torch.equal(x, y)
    mb = 256
    cur, pk, idx = _grad_inputs(d, P, mb, seed=9)
    gcur, gidx, t = dev(cur), dev(idx, torch.int32), {k: dev(v) for k, v in pk.items()}
    for cluster in ((0, 2, 8, 1, 32) if name != "humanoid" else (0, 2, 8, 32)):
        if name == "ant" and cluster == 32:
            continue
        grads = []
        for h in (None, 64):
            ws = K.ppo_workspace(P, 4 * mb, d, "cuda", cluster)
            wp, wn = K._aligned(ws)
            g = torch.zeros(P, d.n_par, device="cuda"); ls = torch.empty(P, 3, device="cuda")
            a = (ptr(gcur), ptr(t["obs"]), t["obs"].stride(0), ptr(t["action"]), ptr(t["logp"]), ptr(t["value"]),
                 t["value"].stride(0), ptr(t["returns"]), ptr(t["adv"]), ptr(gidx), mb,
                 ctypes.byref(PpoHyper()), ptr(g), ptr(ls), wp, wn, cluster, P, 4 * mb, d.obs, d.act, d.obj)
            check(lib().pgm_ppo_grad_f32(*a, st) if h is None else lib().pgm_ppo_grad_h_f32(*a, h, st))
            torch.cuda.synchronize()
            grads.append((g, ls))
        assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1]), cluster
    assert lib().pgm_ppo_workspace_bytes(P, 1024, d.obs, d.act, d.obj, 0) == \
        lib().pgm_ppo_workspace_bytes_h(P, 1024, d.obs, d.act, d.obj, 0, 64)


# --------------------------------------------------------------------------------------------------- whole iterations
def _task(d, seed, weights, E, B):
    from pgmorl_b200.a2c_ppo_acktr.algo import PPO
    from pgmorl_b200.a2c_ppo_acktr.model import Policy
    from pgmorl_b200.sample import Sample, Task
    from pgmorl_b200.scalarization_methods import WeightedSumScalarization
    torch.manual_seed(seed)
    pol = Policy((d.obs,), synth_envs._Box(d.act), base_kwargs={"layernorm": False, "hidden_size": d.hidden},
                 obj_num=d.obj)
    agent = PPO(pol, 0.2, E, B, 0.5, 0.0, lr=3e-4, eps=1e-5, max_grad_norm=0.5)
    sample = Sample({"ob_rms": None, "ret_rms": None, "obj_rms": None}, pol, agent, objs=np.zeros(d.obj), optgraph_id=-1)
    return Task(sample, WeightedSumScalarization(num_objs=d.obj, weights=weights))


def test_worker_and_population_update_match_the_torch_port_at_128(tmp_path):
    """One MOPG iteration at width 128 on replayed trajectories: MOPG_worker against the float64 torch port (1e-4), and
    mopg_population_update -- host-normalised and with the normalisation on the device (K6) -- against MOPG_worker and
    against each other (bit for bit)."""
    from oracle.mopg_torch_port import PortPolicy, mopg_iteration_port
    from pgmorl_b200 import mopg, warm_up
    from pgmorl_b200.sample import Task
    from tests.test_gpu_ppo_options import _replay_args
    from tests.test_gpu_vecnorm import _HostNormalised, _RawEnv
    d = NetDims(17, 6, 2, 128)
    T, N, E, B, P, j = 32, 4, 2, 4, 3, 1
    args = _replay_args(T, N, E, B, True, True)
    traj = {k: v.numpy() for k, v in synthetic.make_trajectories(P, T, N, d, seed=40, p_done=0.08).items()}
    obj_var = np.array([1.3, 0.7])
    wts = [np.array([0.2, 0.8]), np.array([0.5, 0.5]), np.array([0.9, 0.1])]
    tasks = [_task(d, 1000 + p, wts[p], E, B) for p in range(P)]
    assert all(t.sample.actor_critic.dims == d for t in tasks)
    init = [t.sample.actor_critic.flat.cpu().numpy().astype(np.float64) for t in tasks]
    order = iter(range(10 ** 6))

    def replay_env(**kw):
        i = next(order) % P
        return synth_envs.ReplayVecEnv({k: v[i] for k, v in traj.items()}, d, obj_var)

    mopg.set_env_hooks(make_vec_envs=replay_env, gym_make=lambda name: synth_envs.ToyEvalEnv(d), make_raw_vec_envs=False)
    worker = []
    for p in range(P):
        order = iter([p] * 10)
        q, ev = queue.Queue(), threading.Event()
        ev.set()
        mopg.MOPG_worker(args, p, _task(d, 1000 + p, wts[p], E, B), torch.device("cuda"), j, 1, 0.0, q, ev)
        off = q.get_nowait()["offspring_batch"][0]
        assert off.actor_critic.dims == d
        worker.append(off.actor_critic.flat.cpu().numpy().astype(np.float64))
    for p in range(P):
        pol = PortPolicy(init[p], d.obs, d.act, d.obj, 128)
        opt = torch.optim.Adam(pol.ordered(), lr=3e-4, eps=1e-5)
        mopg_iteration_port(pol, opt, {k: v[p] for k, v in traj.items()}, j, synthetic.linear_lr(3e-4, j, 1.0, 10),
                            wts[p], obj_var, ppo_epoch=E, num_mini_batch=B)
        assert rel_err(worker[p], pol.flat()) < 1e-4
    order = iter(range(10 ** 6))
    pop = mopg.mopg_population_update(args, tasks, torch.device("cuda"), j, 1)
    for p in range(P):
        assert rel_err(pop[p][0].actor_critic.flat.cpu().numpy(), worker[p]) < 1e-4
    args = synth_envs.run_args_2d(str(tmp_path), T=T, N=N)
    args.hidden_size = 128
    mopg.set_env_hooks(make_vec_envs=lambda **kw: _HostNormalised(_RawEnv(N, d.obs, d.obj), d, args.gamma))
    torch.manual_seed(0)
    elites, scals = warm_up.initialize_warm_up_batch(args, "cuda")
    assert elites[0].actor_critic.dims == d
    host = mopg.mopg_population_update(args, [Task(e, s) for e, s in zip(elites[:3], scals[:3])], torch.device("cuda"), 0, 2)
    mopg.set_env_hooks(make_raw_vec_envs=lambda **kw: _RawEnv(N, d.obs, d.obj))
    try:
        fused = mopg.mopg_population_update(args, [Task(e, s) for e, s in zip(elites[:3], scals[:3])], torch.device("cuda"), 0, 2)
    finally:
        mopg.set_env_hooks(make_raw_vec_envs=False)
    for hs, fs in zip(host, fused):
        for a, b in zip(hs, fs):
            assert torch.equal(a.actor_critic.flat, b.actor_critic.flat)
            assert torch.equal(a.agent.optimizer.exp_avg_sq, b.agent.optimizer.exp_avg_sq)


@pytest.mark.parametrize("H", WIDTHS)
def test_run_at_width_completes_and_saves_its_width(tmp_path, H):
    """warm-up + 2 generations of morl.run with hidden_size = H; the archive's policies are saved at width H"""
    from pgmorl_b200 import mopg, morl
    d = NetDims(17, 6, 2, H)
    args = synth_envs.run_args_2d(str(tmp_path))
    args.hidden_size = H
    mopg.set_env_hooks(
        make_vec_envs=lambda **kw: synth_envs.SeededReplayVecEnv(d, args.num_steps, args.num_processes, [1.3, 0.7],
                                                                 base_seed=500),
        gym_make=lambda name: synth_envs.ToyEvalEnv(d))
    ep, population, opt_graph, timings = morl.run(args, device="cuda")
    assert len(timings) == 3
    assert all(s.actor_critic.dims == d for s in population.sample_batch)
    final = os.path.join(str(tmp_path), "final")
    pols = [f for f in os.listdir(final) if f.startswith("EP_policy_")]
    assert pols
    for f in pols:
        sd = torch.load(os.path.join(final, f))
        assert tuple(sd["base.actor.0.weight"].shape) == (H, 17) and tuple(sd["base.critic.0.weight"].shape) == (H, 17)
        assert tuple(sd["base.actor.2.weight"].shape) == (H, H) and tuple(sd["base.critic.2.weight"].shape) == (H, H)
        assert tuple(sd["dist.fc_mean.weight"].shape) == (6, H)


def test_two_gpu_run_at_width_32_equals_single_gpu_run(tmp_path):
    """the sharded run at width 32 writes the same files as the single-GPU run, bit for bit: elites that migrate between
    the GPUs carry their width-32 state (dist.sample_state_len follows the policy's dims)"""
    import subprocess
    import sys
    from tests.test_gpu_dist_run import _free_port, _tree
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 visible GPUs")
    here = os.path.dirname(os.path.abspath(__file__))
    trees = []
    for nproc in (1, 2):
        save = str(tmp_path / f"w{nproc}")
        os.makedirs(save)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr",
               "127.0.0.1", "--master-port", str(_free_port()), os.path.join(here, "dist_run_hidden_worker.py"), save,
               "prediction-guided", "32"]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        trees.append(_tree(save))
    one, two = trees
    assert sorted(one) == sorted(two) and any(k.startswith("final") for k in one)
    for k in sorted(one):                          # compared as tests/test_gpu_dist_run.py compares them
        if k.endswith(".txt"):
            assert open(one[k]).read() == open(two[k]).read(), k
        elif k.endswith(".pt"):
            x, y = torch.load(one[k]), torch.load(two[k])
            assert list(x) == list(y) and all(torch.equal(x[n], y[n]) for n in x), k
            if "base.actor.2.weight" in x:
                assert tuple(x["base.actor.2.weight"].shape) == (32, 32)
        elif k.endswith(".pkl"):
            x, y = pickle.load(open(one[k], "rb")), pickle.load(open(two[k], "rb"))
            for key in ("ob_rms", "ret_rms", "obj_rms"):
                if x[key] is None:
                    assert y[key] is None
                    continue
                assert np.array_equal(np.asarray(x[key].mean), np.asarray(y[key].mean)), (k, key)
                assert np.array_equal(np.asarray(x[key].var), np.asarray(y[key].var)), (k, key)
