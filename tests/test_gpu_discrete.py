"""Categorical heads (Discrete(n) actions) on the device: K1 (every action mode, trajectory and per-step), K3's raw
gradient and update on the generic cluster kernel, the refusals, the Gaussian path of the _x entry points, and whole MOPG
iterations up to morl.run.

The float64 pin is tests/discrete_ref.py (numpy with a hand-derived backward), which tests/test_oracle_discrete.py checks
against torch.distributions.Categorical with autograd. Gates are the ones of the width-64 tests. A sampled or greedy
action is compared only where the float64 oracle's top-two margin (r1 - r2) / r1 is at least 1e-4: below that, FP32
logits may legitimately pick the other index. Such rows are counted over all the rows a test compares, reported, and
must stay under 0.1 % of them."""
import ctypes
import os
import queue
import threading

import numpy as np
import pytest
import torch

import discrete_ref as dref
import synth_envs
from pgmorl_b200 import synthetic
from pgmorl_b200._lib import PgmError
from pgmorl_b200.layout import DIST_CATEGORICAL, NetDims, param_layout
from tests.helpers import rel_err
from tests.test_gpu_kernels import dev

pytestmark = pytest.mark.gpu

MARGIN = 1e-4
# (O, n, M): Deep-Sea-Treasure-like, mid, wide head (n > 16: the wide variant of K3), O > 64, and the three (O, n, M)
# that equal Gaussian shapes with tensor-core kernels (a categorical policy must never reach those)
SHAPES = {"dst": (2, 4, 2), "mid": (11, 9, 3), "wide_head": (33, 18, 2), "wide_obs": (70, 5, 2),
          "tc_walker": (17, 6, 2), "tc_hopper3": (11, 3, 3), "tcw_humanoid": (376, 17, 2)}


def _fits(name, H):
    return not (name == "tcw_humanoid" and H == 128)     # a width-128 half with O = 376 exceeds 227 KB of shared memory


def _dims(name, H):
    return NetDims(*SHAPES[name], H, DIST_CATEGORICAL)


def _params(d, P, seed, head_scale=0.5):
    """init_policy_flat, with the logits head scaled up so that the softmax is far from uniform"""
    rng = np.random.RandomState(seed)
    params = np.stack([synthetic.init_policy_flat(d, seed=seed * 100 + p).numpy() for p in range(P)])
    off, _ = param_layout(d)[0]["dist.linear.weight"]
    k = d.act * d.hidden
    params[:, off:off + k] = rng.randn(P, k) * head_scale
    params[:, off + k:] = rng.randn(P, d.act) * 0.3
    return params


def _net(d, flat):
    return dref.net_of(np.asarray(flat, dtype=np.float64).copy(), d)


def _check_actions(got, want, margin, what):
    """Equal actions on every row that clears the margin; returns (rows below the margin, rows compared)."""
    ok = margin >= MARGIN
    assert np.array_equal(got[ok], want[ok]), what
    return np.array([int((~ok).sum()), ok.size])


def _report_below(counts, what):
    below, rows = counts
    print(f"{what}: {below} of {rows} rows below the margin")
    assert below < 1e-3 * rows, (what, below, rows)


# ------------------------------------------------------------------------------------------------------------------ K1
K1_CASES = [(n, H, 100) for H in (32, 64, 128) for n in SHAPES if _fits(n, H)] + \
           [(n, 64, 300) for n in ("tc_walker", "tc_hopper3")] + [("tcw_humanoid", 64, 150)]   # >= 1024 rows


@pytest.mark.parametrize("name,H,T", K1_CASES)
def test_k1_all_modes_match_oracle(name, H, T):
    from pgmorl_b200 import kernels as K
    d = _dims(name, H)
    P, N = 2, 8
    params = _params(d, P, seed=3)
    traj = {k: v.numpy() for k, v in synthetic.make_trajectories(P, T, N, d, seed=3).items()}
    q, _ = synthetic.host_rng_streams(3, T, N, d.act, 1, categorical=True)
    q = q.numpy()
    obs = dev(traj["obs"]).reshape(P, (T + 1) * N, d.obs)
    gp = dev(params)
    ent = torch.empty(P, T * N, device="cuda")
    value, action, logp = K.policy_forward(gp, obs, d, eps=dev(q).reshape(1, T * N, d.act), rows_a=T * N, entropy=ent)
    ent_det = torch.empty(P, (T + 1) * N, device="cuda")
    v_det, a_det, lp_det = K.policy_forward(gp, obs, d, mode=K.ACT_DETERMINISTIC, entropy=ent_det)
    torch.cuda.synchronize()
    assert action.shape == (P, T * N, 1)
    below = np.zeros(2, dtype=np.int64)
    for p in range(P):
        net = _net(d, dev(params[p]).cpu().numpy())
        x = traj["obs"][p].astype(np.float64)
        v, a, _, margin = dref.rollout(net, x, q)
        _, z, _ = dref.forward(net, x.reshape(-1, d.obs))
        lsm = dref.log_softmax(z)
        assert rel_err(value[p].cpu().numpy().reshape(T + 1, N, -1), v) < 2e-5
        ga = action[p, :, 0].cpu().numpy().astype(np.int64)
        below += _check_actions(ga, a.reshape(-1), margin.reshape(-1), "sample")
        # log-prob of the action the device took (identical to the oracle's wherever the actions agree)
        assert rel_err(logp[p].cpu().numpy(), lsm[np.arange(T * N), ga]) < 2e-5
        assert rel_err(ent[p].cpu().numpy(), dref.entropy_rows(z[:T * N])) < 2e-5
        am, mm = dref.mode(z)
        gd = a_det[p, :, 0].cpu().numpy().astype(np.int64)
        below += _check_actions(gd, am, mm, "mode")
        assert rel_err(lp_det[p].cpu().numpy(), lsm[np.arange(len(gd)), gd]) < 2e-5
        assert rel_err(ent_det[p].cpu().numpy(), dref.entropy_rows(z)) < 2e-5
        assert rel_err(v_det[p].cpu().numpy(), v.reshape(-1, d.obj)) < 2e-5
    _report_below(below, f"{name} H={H} T={T}")
    _, _, lp_ev = K.policy_forward(gp, obs, d, action=action.contiguous(), mode=K.ACT_EVALUATE, rows_a=T * N)
    torch.cuda.synchronize()
    assert torch.equal(lp_ev, logp)


@pytest.mark.parametrize("H", [32, 64, 128])
@pytest.mark.parametrize("staged", [True, False])
def test_k1_per_step_matches_oracle(H, staged):
    """pgm_policy_step_x_f32: one environment step of every task written into time slot t of the rollout buffers, with
    the observations staged or already in the slot (K6-written)"""
    from pgmorl_b200 import kernels as K
    d = _dims("mid", H)
    P, N, T, t = 3, 16, 5, 2
    params = _params(d, P, seed=8)
    rng = np.random.RandomState(4)
    x = rng.randn(P, N, d.obs)
    q = rng.exponential(size=(1, N, d.act))
    obs_buf = torch.zeros(P, (T + 1) * N, d.obs, device="cuda")
    if not staged:
        obs_buf[:, t * N:(t + 1) * N] = dev(x)
    value_buf = torch.zeros(P, (T + 1) * N, d.obj, device="cuda")
    action_buf = torch.zeros(P, T * N, 1, device="cuda")
    logp_buf = torch.zeros(P, T * N, device="cuda")
    act_out = torch.zeros(P, N, 1, device="cuda")
    ctl = torch.tensor([t, 1], dtype=torch.int32, device="cuda")
    K.policy_step(dev(params), ctl, dev(x) if staged else None, dev(q), obs_buf, value_buf, action_buf, logp_buf,
                  act_out, N, d)
    torch.cuda.synchronize()
    rows = slice(t * N, (t + 1) * N)
    below = np.zeros(2, dtype=np.int64)
    for p in range(P):
        net = _net(d, dev(params[p]).cpu().numpy())
        xx = dev(x[p]).cpu().numpy().astype(np.float64)
        v, a, _, margin = dref.rollout(net, np.stack([xx, xx]), dev(q).cpu().numpy().astype(np.float64))
        _, z, _ = dref.forward(net, xx)
        assert rel_err(value_buf[p, rows].cpu().numpy(), v[0]) < 2e-5
        ga = action_buf[p, rows, 0].cpu().numpy().astype(np.int64)
        below += _check_actions(ga, a[0], margin[0], "step")
        assert rel_err(logp_buf[p, rows].cpu().numpy(), dref.log_softmax(z)[np.arange(N), ga]) < 2e-5
        assert torch.equal(act_out[p], action_buf[p, rows])
        assert rel_err(obs_buf[p, rows].cpu().numpy(), x[p]) < 1e-7
        assert torch.count_nonzero(action_buf[p, :t * N]) == 0        # other slots untouched
    _report_below(below, f"per-step H={H}")


# ------------------------------------------------------------------------------------------------------- K3 gradient
def _grad_inputs(d, P, mb, seed):
    rng = np.random.RandomState(seed)
    S = 4 * mb
    params = _params(d, P, seed)
    cur = params + rng.randn(*params.shape) * 0.02
    obs = rng.randn(P, S, d.obs)
    act = rng.randint(0, d.act, (P, S))
    value, logp = [], []
    for p in range(P):
        v, z, _ = dref.forward(_net(d, params[p]), obs[p])
        value.append(v)
        logp.append(dref.log_softmax(z)[np.arange(S), act[p]])
    value, logp = np.stack(value), np.stack(logp)
    pk = dict(obs=obs, action=act[..., None].astype(np.float64), logp=logp + rng.randn(P, S) * 0.1,
              value=value + rng.randn(P, S, d.obj) * 0.4, returns=value + rng.randn(P, S, d.obj), adv=rng.randn(P, S))
    return cur, pk, rng.permutation(S)[:mb]


GRAD_CASES = [(n, H, c) for H in (32, 64, 128) for n in ("dst", "mid", "wide_head", "wide_obs") if _fits(n, H)
              for c in (2, 4, 8, 16, 0)] + [(n, 64, 0) for n in ("tc_walker", "tc_hopper3", "tcw_humanoid")]


@pytest.mark.parametrize("ecoef", [0.0, 0.01])
@pytest.mark.parametrize("vu", [False, True])
@pytest.mark.parametrize("name,H,cluster", GRAD_CASES)
def test_k3_gradient_per_tensor(name, H, cluster, vu, ecoef):
    from pgmorl_b200 import kernels as K
    d = _dims(name, H)
    P, mb = 2, 256
    cur, pk, idx = _grad_inputs(d, P, mb, seed=41)
    g, losses = K.ppo_grad(dev(cur), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]),
                           dev(pk["returns"]), dev(pk["adv"]), dev(idx, torch.int32), d,
                           hyper=K.PpoHyper(entropy_coef=ecoef), cluster=cluster, clipped_value_loss=not vu)
    torch.cuda.synchronize()
    g, losses = g.cpu().numpy(), losses.cpu().numpy()
    layout, _ = param_layout(d)
    for p in range(P):
        f = lambda a: dev(a[p][idx]).cpu().numpy().astype(np.float64)
        gref, lref = dref.ppo_grad(_net(d, dev(cur[p]).cpu().numpy()), f(pk["obs"]), pk["action"][p][idx, 0].astype(np.int64),
                                   f(pk["logp"]), f(pk["value"]), f(pk["returns"]), f(pk["adv"]), ecoef=ecoef,
                                   clipped_value_loss=not vu)
        assert rel_err(losses[p], np.array(lref)) < 1e-4
        for tname, (off, shape) in layout.items():
            n = int(np.prod(shape))
            assert rel_err(g[p][off:off + n], gref[off:off + n]) < 2e-5, (tname, rel_err(g[p][off:off + n], gref[off:off + n]))


# --------------------------------------------------------------------------------------------------------- K3 update
@pytest.mark.parametrize("name,H,P", [(n, H, P) for n, H in (("dst", 64), ("mid", 32), ("wide_head", 128), ("tc_walker", 64))
                                      for P in (6, 40)])
def test_k3_update_matches_oracle(name, H, P):
    from pgmorl_b200 import kernels as K
    d = _dims(name, H)
    T, N, B = 32, 4, 2
    params = _params(d, P, seed=13)
    traj = {k: v.numpy() for k, v in synthetic.make_trajectories(P, T, N, d, seed=13, p_done=0.05).items()}
    q, perm = synthetic.host_rng_streams(13, T, N, d.act, 2, categorical=True)
    q, perm = q.numpy(), perm.numpy()
    rng = np.random.RandomState(2)
    S = T * N
    pk = {k: [] for k in ("action", "logp", "value", "returns", "adv")}
    for p in range(P):
        value, action, logp, _ = dref.rollout(_net(d, params[p]), traj["obs"][p].astype(np.float64), q)
        ret = dref.orc.gae_returns(traj["rewards"][p].astype(np.float64), value, traj["masks"][p].astype(np.float64),
                                   traj["bad_masks"][p].astype(np.float64), 0.995, 0.95)
        adv = dref.orc.advantages(ret, value, np.full(d.obj, 1.0 / d.obj), np.ones(d.obj))
        for k, v in zip(pk, (action, logp, value, ret, adv)):
            pk[k].append(v)
    pk = {k: np.stack(v) for k, v in pk.items()}
    cur = params + rng.randn(*params.shape) * 0.02
    m0, v0 = rng.randn(P, d.n_par) * 1e-3, rng.rand(P, d.n_par) * 1e-5
    step0 = np.resize(np.array([0, 7, 640], dtype=np.int32), P)
    lr = np.resize(np.array([3e-4, 2.5e-4, 1e-4]), P)
    hy = K.PpoHyper(entropy_coef=0.01)
    gp, gm, gv, gstep = dev(cur), dev(m0), dev(v0), dev(step0, torch.int32)
    losses = K.ppo_update(gp, gm, gv, gstep, dev(lr, torch.float64), dev(traj["obs"]).reshape(P, (T + 1) * N, d.obs),
                          dev(pk["action"].astype(np.float64)).reshape(P, S, 1), dev(pk["logp"]).reshape(P, S),
                          dev(pk["value"]).reshape(P, (T + 1) * N, d.obj), dev(pk["returns"]).reshape(P, S, d.obj),
                          dev(pk["adv"]).reshape(P, S), dev(perm[None], torch.int32), B, d, hyper=hy)
    torch.cuda.synchronize()
    for p in range(P):
        f32 = lambda a: dev(a).cpu().numpy().astype(np.float64)
        flat, m, v = f32(cur[p]), f32(m0[p]), f32(v0[p])
        step, lref = dref.ppo_update(flat, m, v, int(step0[p]), lr[p], d, f32(traj["obs"][p]), pk["action"][p],
                                     f32(pk["logp"][p]), f32(pk["value"][p]), f32(pk["returns"][p]), f32(pk["adv"][p]),
                                     perm, B, ecoef=0.01)
        assert int(gstep[p]) == step
        assert rel_err(gp[p].cpu().numpy(), flat) < 1e-5
        assert rel_err(gm[p].cpu().numpy(), m) < 1e-4
        assert rel_err(gv[p].cpu().numpy(), v) < 1e-4
        assert rel_err(losses[p].cpu().numpy(), np.array(lref)) < 1e-4


# ---------------------------------------------------------------------------------------------------------- refusals
@pytest.mark.parametrize("H", [32, 64, 128])
@pytest.mark.parametrize("cluster", [1, 32, 64, 128])
def test_k3_refuses_gaussian_only_kernels(H, cluster):
    from pgmorl_b200 import kernels as K
    d = _dims("tc_walker", H)
    cur, pk, idx = _grad_inputs(d, 1, 64, seed=5)
    with pytest.raises(PgmError, match="categorical head"):
        K.ppo_grad(dev(cur), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]), dev(pk["returns"]),
                   dev(pk["adv"]), dev(idx, torch.int32), d, cluster=cluster)


def test_more_than_32_categories_are_refused():
    from pgmorl_b200 import kernels as K
    from pgmorl_b200._lib import check, lib, ptr
    from pgmorl_b200.a2c_ppo_acktr.model import Policy
    with pytest.raises(NotImplementedError, match="1 to 32"):
        Policy((4,), synth_envs_discrete(33), base_kwargs={"layernorm": False}, obj_num=2)
    P, rows, O, n, M = 1, 8, 4, 33, 2
    x = torch.zeros(P, rows, O, device="cuda")
    params = torch.zeros(P, 4096 * 4, device="cuda")
    v, a, lp = (torch.empty(P, rows, M, device="cuda"), torch.empty(P, rows, 1, device="cuda"),
                torch.empty(P, rows, device="cuda"))
    with pytest.raises(PgmError, match="1..32 categories"):
        check(lib().pgm_policy_forward_x_f32(ptr(params), ptr(x), None, 0, ptr(a), ptr(v), ptr(lp), None, 1, P, rows, rows,
                                             O, n, M, 64, DIST_CATEGORICAL, K._stream()))
    d = NetDims(O, 32, M, 64, DIST_CATEGORICAL)
    cur, pk, idx = _grad_inputs(d, 1, 64, seed=5)
    ws = K.ppo_workspace(1, 256, d, "cuda")
    wp, wn = K._aligned(ws)
    g, ls = torch.zeros(1, 8192, device="cuda"), torch.empty(1, 3, device="cuda")
    t = {k: dev(v) for k, v in pk.items()}
    with pytest.raises(PgmError, match="1..32 categories"):
        check(lib().pgm_ppo_grad_x_f32(ptr(dev(cur)), ptr(t["obs"]), t["obs"].stride(0), ptr(t["action"]), ptr(t["logp"]),
                                       ptr(t["value"]), t["value"].stride(0), ptr(t["returns"]), ptr(t["adv"]),
                                       ptr(dev(idx, torch.int32)), 64, ctypes.byref(K.PpoHyper()), ptr(g), ptr(ls), wp, wn,
                                       0, 1, 256, O, 33, M, 64, DIST_CATEGORICAL, K._stream()))
    with pytest.raises(PgmError, match="for categorical heads only"):
        check(lib().pgm_policy_forward_x_f32(ptr(params), ptr(x), None, 0, ptr(a), ptr(v), ptr(lp), ptr(lp), 1, P, rows,
                                             rows, O, 6, M, 64, 0, K._stream()))
    torch.cuda.synchronize()


@pytest.mark.parametrize("name,A,rows", [("walker2d", 6, 40 * 4), ("walker2d", 6, 300 * 4), ("humanoid", 17, 150 * 8),
                                         ("ant", 8, 300 * 4)])
def test_x_entry_points_with_gaussian_head_equal_the_h_ones(name, A, rows):
    """the _x entry points with PGM_DIST_GAUSSIAN run what the _h ones run, bit for bit (forward, gradient at every plan
    family, update)"""
    from pgmorl_b200 import kernels as K
    from pgmorl_b200._lib import PpoHyper, check, lib, ptr
    from pgmorl_b200.layout import ENV_SHAPES
    d = ENV_SHAPES[name]
    P = 2
    gp = dev(np.stack([synthetic.init_policy_flat(d, seed=6 + p).numpy() for p in range(P)]))
    obs = torch.randn(P, rows, d.obs, device="cuda")
    eps = torch.randn(1, rows, d.act, device="cuda")
    st = K._stream()
    outs = []
    for x in (False, True):
        value = torch.empty(P, rows, d.obj, device="cuda"); act = torch.empty(P, rows, d.act, device="cuda")
        logp = torch.empty(P, rows, device="cuda")
        a = (ptr(gp), ptr(obs), ptr(eps), 1, ptr(act), ptr(value), ptr(logp))
        b = (0, P, rows, rows, d.obs, d.act, d.obj, 64)
        check(lib().pgm_policy_forward_x_f32(*a, None, *b, 0, st) if x else lib().pgm_policy_forward_h_f32(*a, *b, st))
        outs.append((value, act, logp))
    for u, w in zip(*outs):
        assert torch.equal(u, w)
    mb = 256
    rng = np.random.RandomState(9)
    S = 4 * mb
    t = {k: dev(v) for k, v in dict(obs=rng.randn(P, S, d.obs), action=rng.randn(P, S, d.act), logp=rng.randn(P, S) - 6,
                                    value=rng.randn(P, S, d.obj), returns=rng.randn(P, S, d.obj), adv=rng.randn(P, S)).items()}
    gidx = dev(rng.permutation(S)[:mb], torch.int32)
    for cluster in ((0, 2, 8, 1, 32) if name != "humanoid" else (0, 2, 8, 32)):
        if name == "ant" and cluster == 32:
            continue
        grads = []
        for x in (False, True):
            ws = K.ppo_workspace(P, S, d, "cuda", cluster)
            wp, wn = K._aligned(ws)
            g = torch.zeros(P, d.n_par, device="cuda"); ls = torch.empty(P, 3, device="cuda")
            a = (ptr(gp), ptr(t["obs"]), t["obs"].stride(0), ptr(t["action"]), ptr(t["logp"]), ptr(t["value"]),
                 t["value"].stride(0), ptr(t["returns"]), ptr(t["adv"]), ptr(gidx), mb,
                 ctypes.byref(PpoHyper(entropy_coef=0.01)), ptr(g), ptr(ls), wp, wn, cluster, P, S, d.obs, d.act, d.obj, 64)
            check(lib().pgm_ppo_grad_x_f32(*a, 0, st) if x else lib().pgm_ppo_grad_h_f32(*a, st))
            torch.cuda.synchronize()
            grads.append((g, ls))
        assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1]), cluster


# --------------------------------------------------------------------------------------------------- whole iterations
class _Discrete:
    def __init__(self, n):
        self.n = n


_Discrete.__name__ = "Discrete"


def synth_envs_discrete(n):
    return _Discrete(n)


class DiscreteActions:
    """Wraps a synth_envs environment: a Discrete(n) action space, and stepping that takes int64 category indices of shape
    [N,1] (vectorised) or [1] / [1,1] (evaluation), as the reference's VecPyTorch / gym envs receive them."""

    def __init__(self, env, n, N=None):
        self.env, self.n, self.N = env, n, N
        self.action_space = _Discrete(n)
        self.observation_space = env.observation_space if hasattr(env, "observation_space") else None
        self.taken = []

    def __getattr__(self, k):
        return getattr(self.env, k)

    def check(self, action):
        a = torch.as_tensor(action)
        assert a.dtype == torch.int64 and a.shape[-1] == 1 and int(a.min()) >= 0 and int(a.max()) < self.n, a
        if self.N is not None:
            assert tuple(a.shape) == (self.N, 1)
        self.taken.append(a.clone())
        return a

    def step(self, action):
        self.check(action)
        return self.env.step(action)


class DiscreteEvalEnv(DiscreteActions):
    """ToyEvalEnv with an objective that depends on the chosen category"""

    def __init__(self, dims):
        super().__init__(synth_envs.ToyEvalEnv(dims), dims.act)
        self.dims = dims

    def step(self, action):
        a = int(self.check(action).reshape(-1)[0])
        ob, r, done, info = self.env.step(np.zeros(1))
        f = a / max(self.dims.act - 1, 1)
        info["obj"] = np.array([1.0 + f, 2.0 - f, 1.0][:self.dims.obj])
        return ob, r, done, info


def _task(d, seed, weights, E, B, ecoef=0.0):
    from pgmorl_b200.a2c_ppo_acktr.algo import PPO
    from pgmorl_b200.a2c_ppo_acktr.model import Policy
    from pgmorl_b200.sample import Sample, Task
    from pgmorl_b200.scalarization_methods import WeightedSumScalarization
    torch.manual_seed(seed)
    pol = Policy((d.obs,), _Discrete(d.act), base_kwargs={"layernorm": False, "hidden_size": d.hidden}, obj_num=d.obj)
    agent = PPO(pol, 0.2, E, B, 0.5, ecoef, lr=3e-4, eps=1e-5, max_grad_norm=0.5)
    sample = Sample({"ob_rms": None, "ret_rms": None, "obj_rms": None}, pol, agent, objs=np.zeros(d.obj), optgraph_id=-1)
    return Task(sample, WeightedSumScalarization(num_objs=d.obj, weights=weights))


def test_policy_act_and_evaluate_actions():
    """Policy.act draws exponential_(1) [N,n] from the global generator and returns int64 [N,1]; evaluate_actions returns
    the mean entropy over the rows"""
    d = _dims("mid", 64)
    torch.manual_seed(4)
    pol = _task(d, 4, np.array([0.5, 0.3, 0.2]), 1, 1).sample.actor_critic
    pol.flat.copy_(dev(_params(d, 1, seed=4)[0]))
    x = torch.randn(64, d.obs)
    torch.manual_seed(11)
    value, action, logp, _ = pol.act(x, None, None)
    st = torch.get_rng_state()
    torch.manual_seed(11)
    q = torch.empty(64, d.act, dtype=torch.float64).exponential_(1)
    assert torch.equal(torch.get_rng_state(), st)
    assert action.dtype == torch.int64 and action.shape == (64, 1) and logp.shape == (64, 1)
    net = _net(d, pol.flat.cpu().numpy())
    xx = x.numpy().astype(np.float64)
    _, z, _ = dref.forward(net, xx)
    a, margin = dref.sample(z, q.numpy())
    below = _check_actions(action[:, 0].cpu().numpy(), a, margin, "act")
    v2, lp2, ent, _ = pol.evaluate_actions(x, None, None, action)
    assert torch.equal(lp2, logp) and rel_err(v2.cpu().numpy(), value.cpu().numpy()) == 0
    assert abs(float(ent) - dref.entropy_rows(z).mean()) < 2e-5 * abs(dref.entropy_rows(z).mean())
    _, a_det, _, _ = pol.act(x, None, None, deterministic=True)
    am, mm = dref.mode(z)
    _report_below(below + _check_actions(a_det[:, 0].cpu().numpy(), am, mm, "mode"), "Policy.act")


def test_worker_and_population_update_match_the_torch_port():
    """One MOPG iteration of a Deep-Sea-Treasure-like Categorical policy on replayed trajectories: MOPG_worker against
    the float64 torch port (1e-4), mopg_population_update host-normalised against MOPG_worker (1e-4), and the K6 mode
    against the host-normalised mode (bit for bit)"""
    from pgmorl_b200 import mopg, warm_up
    from pgmorl_b200.sample import Task
    from tests.test_gpu_ppo_options import _replay_args
    from tests.test_gpu_vecnorm import _HostNormalised, _RawEnv
    d = _dims("dst", 64)
    T, N, E, B, P, j = 32, 4, 2, 4, 3, 1
    args = _replay_args(T, N, E, B, True, True)
    traj = {k: v.numpy() for k, v in synthetic.make_trajectories(P, T, N, d, seed=40, p_done=0.08).items()}
    obj_var = np.array([1.3, 0.7])
    wts = [np.array([0.2, 0.8]), np.array([0.5, 0.5]), np.array([0.9, 0.1])]
    init = [_task(d, 1000 + p, wts[p], E, B, 0.01).sample.actor_critic.flat.cpu().numpy().astype(np.float64)
            for p in range(P)]
    # every sampled action of the rollout clears the float64 margin, so FP32 and float64 take the same actions
    q, _ = synthetic.host_rng_streams(j, T, N, d.act, E, categorical=True)
    for p in range(P):
        _, _, _, margin = dref.rollout(_net(d, dev(init[p]).cpu().numpy()), traj["obs"][p].astype(np.float64), q.numpy())
        assert margin.min() >= MARGIN
    envs = []

    def replay_env(**kw):
        e = DiscreteActions(synth_envs.ReplayVecEnv({k: v[cur[0]] for k, v in traj.items()}, d, obj_var), d.act, N)
        envs.append(e)
        return e

    mopg.set_env_hooks(make_vec_envs=replay_env, gym_make=lambda name: DiscreteEvalEnv(d), make_raw_vec_envs=False)
    worker = []
    for p in range(P):
        cur = [p]
        qq, ev = queue.Queue(), threading.Event()
        ev.set()
        mopg.MOPG_worker(args, p, _task(d, 1000 + p, wts[p], E, B, 0.01), torch.device("cuda"), j, 1, 0.0, qq, ev)
        off = qq.get_nowait()["offspring_batch"][0]
        assert off.actor_critic.dims == d
        worker.append(off.actor_critic.flat.cpu().numpy().astype(np.float64))
        pol = dref.PortCatPolicy(init[p], d.obs, d.act, d.obj, 64)
        opt = torch.optim.Adam(pol.ordered(), lr=3e-4, eps=1e-5)
        port = dref.mopg_iteration_port(pol, opt, {k: v[p] for k, v in traj.items()}, j,
                                        synthetic.linear_lr(3e-4, j, 1.0, 10), wts[p], obj_var, ppo_epoch=E,
                                        num_mini_batch=B, ecoef=0.01)
        assert np.array_equal(torch.cat(envs[-1].taken).reshape(T, N).numpy(), port["action"])
        assert rel_err(worker[p], pol.flat()) < 1e-4
    tasks = [_task(d, 1000 + p, wts[p], E, B, 0.01) for p in range(P)]
    order = iter(range(10 ** 6))

    def replay_env_pop(**kw):
        i = next(order) % P
        e = DiscreteActions(synth_envs.ReplayVecEnv({k: v[i] for k, v in traj.items()}, d, obj_var), d.act, N)
        envs.append(e)
        return e

    mopg.set_env_hooks(make_vec_envs=replay_env_pop)
    pop = mopg.mopg_population_update(args, tasks, torch.device("cuda"), j, 1)
    for p in range(P):
        assert rel_err(pop[p][0].actor_critic.flat.cpu().numpy(), worker[p]) < 1e-4
    # host-normalised vs K6 (raw simulators, normalisation on the device)
    args = synth_envs.run_args_2d("unused", T=T, N=N)
    args.entropy_coef = 0.01
    probe = DiscreteEvalEnv(d)
    mopg.set_env_hooks(make_vec_envs=lambda **kw: DiscreteActions(_HostNormalised(_RawEnv(N, d.obs, d.obj), d, args.gamma),
                                                                  d.act, N),
                       gym_make=lambda name: DiscreteEvalEnv(d))
    torch.manual_seed(0)
    elites, scals = warm_up.initialize_warm_up_batch(args, "cuda")
    assert elites[0].actor_critic.dims == d and probe.action_space.n == d.act
    host = mopg.mopg_population_update(args, [Task(e, s) for e, s in zip(elites[:3], scals[:3])], torch.device("cuda"), 0, 2)
    mopg.set_env_hooks(make_raw_vec_envs=lambda **kw: DiscreteActions(_RawEnv(N, d.obs, d.obj), d.act, N))
    try:
        fused = mopg.mopg_population_update(args, [Task(e, s) for e, s in zip(elites[:3], scals[:3])], torch.device("cuda"), 0, 2)
    finally:
        mopg.set_env_hooks(make_raw_vec_envs=False)
    for hs, fs in zip(host, fused):
        for a, b in zip(hs, fs):
            assert torch.equal(a.actor_critic.flat, b.actor_critic.flat)
            assert torch.equal(a.agent.optimizer.exp_avg_sq, b.agent.optimizer.exp_avg_sq)
            assert len(a.agent.optimizer.state_dict()["state"]) == 12


@pytest.mark.parametrize("H", [32, 64])
def test_run_completes_and_saves_a_categorical_head(tmp_path, H):
    """warm-up + 2 generations of morl.run on a discrete replay environment; the archive's policies carry
    dist.linear.weight [n,H] and no logstd"""
    from pgmorl_b200 import mopg, morl
    d = _dims("dst", H)
    args = synth_envs.run_args_2d(str(tmp_path))
    args.hidden_size = H
    mopg.set_env_hooks(
        make_vec_envs=lambda **kw: DiscreteActions(
            synth_envs.SeededReplayVecEnv(d, args.num_steps, args.num_processes, [1.3, 0.7], base_seed=500), d.act,
            args.num_processes),
        gym_make=lambda name: DiscreteEvalEnv(d))
    ep, population, opt_graph, timings = morl.run(args, device="cuda")
    assert len(timings) == 3
    assert all(s.actor_critic.dims == d for s in population.sample_batch)
    final = os.path.join(str(tmp_path), "final")
    pols = [f for f in os.listdir(final) if f.startswith("EP_policy_")]
    assert pols
    for f in pols:
        sd = torch.load(os.path.join(final, f))
        assert tuple(sd["dist.linear.weight"].shape) == (d.act, H) and tuple(sd["dist.linear.bias"].shape) == (d.act,)
        assert not any("logstd" in k or "fc_mean" in k for k in sd)
