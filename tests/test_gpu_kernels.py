"""GPU parity tests of K1 / K2 / K3 against the float64 oracle, through the C ABI.

Tolerance (north_star): FP32 kernels vs the float64 oracle, norm-wise per tensor,
max|a-b| <= tol * max|b| with tol = 1e-4 for parameters / returns (much tighter where
the arithmetic is short). Written beside each assert.
"""
import numpy as np
import pytest
import torch

from oracle import mopg_oracle as orc
from pgmorl_b200 import synthetic
from pgmorl_b200.layout import NetDims
from tests.helpers import rel_err

pytestmark = pytest.mark.gpu

DIMS = {"walker": NetDims(17, 6, 2), "hopper3": NetDims(11, 3, 3), "humanoid": NetDims(376, 17, 2),
        "hopper2": NetDims(11, 3, 2), "ant": NetDims(27, 8, 2), "swimmer": NetDims(8, 2, 2),
        # test-only shapes at the edges of the K3 planner (tests/test_gpu_shapes.py)
        "s16_16_2": NetDims(16, 16, 2), "s48_16_16": NetDims(48, 16, 16), "s45_16_3": NetDims(45, 16, 3),
        "s60_6_2": NetDims(60, 6, 2), "s64_4_4": NetDims(64, 4, 4), "s33_17_2": NetDims(33, 17, 2)}
TC_SHAPES = ("walker", "hopper3", "humanoid")      # shapes with tensor-core K3 kernels (cluster 32 / 64 / 128)


def dev(x, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(x)).to(device="cuda", dtype=dtype).contiguous()


def make_case(d, P, T, N, seed):
    """Random policies + synthetic trajectories + oracle rollout/GAE/adv in float64."""
    rng = np.random.RandomState(seed)
    params = np.stack([synthetic.init_policy_flat(d, seed=seed * 100 + p).numpy() for p in range(P)])
    params[:, -d.act:] = rng.uniform(-0.5, 0.3, (P, d.act))          # non-trivial logstd
    traj = synthetic.make_trajectories(P, T, N, d, seed=seed, p_done=0.05)
    traj = {k: v.numpy() for k, v in traj.items()}
    eps, perm = synthetic.host_rng_streams(seed, T, N, d.act, 2)
    eps = eps.numpy()
    weights = rng.dirichlet(np.ones(d.obj), P)
    obj_var = rng.uniform(0.5, 2.0, (P, d.obj))
    out = []
    for p in range(P):
        net = orc.Net(params[p].copy(), d.obs, d.act, d.obj)
        value, action, logp = orc.rollout(net, traj["obs"][p].astype(np.float64), eps)
        ret = orc.gae_returns(traj["rewards"][p].astype(np.float64), value, traj["masks"][p].astype(np.float64),
                              traj["bad_masks"][p].astype(np.float64), 0.995, 0.95)
        adv = orc.advantages(ret, value, weights[p], obj_var[p])
        out.append(dict(value=value, action=action, logp=logp, returns=ret, adv=adv))
    return params, traj, eps, perm.numpy(), weights, obj_var, out


@pytest.mark.parametrize("name,P,T,N", [("walker", 3, 50, 4), ("hopper3", 2, 33, 2), ("walker", 1, 1, 4),
                                         ("humanoid", 2, 21, 8),
                                         # >= 1024 rows: the tensor-core forward (csrc/k1_tc.cuh), ragged last tile
                                         ("walker", 2, 301, 4), ("hopper3", 3, 613, 2),
                                         # Humanoid, >= 1024 rows: the wide tensor-core forward (csrc/k1_tcw.cuh)
                                         ("humanoid", 2, 150, 8), ("humanoid", 20, 140, 8),
                                         # shapes without a tensor-core forward at >= 1024 rows: the FFMA kernel, several
                                         # chunks per CTA (8 x 2049 x 4 rows at Ant dims), ragged last chunk
                                         ("ant", 8, 2048, 4), ("hopper2", 2, 300, 4), ("swimmer", 3, 613, 2),
                                         ("s48_16_16", 2, 260, 4)])
@pytest.mark.parametrize("shared_eps", [True, False])
def test_k1_rollout_matches_oracle(name, P, T, N, shared_eps):
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    params, traj, eps, _, _, _, ref = make_case(d, P, T, N, seed=3)
    obs = dev(traj["obs"]).reshape(P, (T + 1) * N, d.obs)
    e = dev(eps).reshape(1, T * N, d.act)
    if not shared_eps:
        e = e.expand(P, -1, -1).contiguous()
    value, action, logp = K.policy_forward(dev(params), obs, d, eps=e, rows_a=T * N)
    torch.cuda.synchronize()
    for p in range(P):
        # FP32 forward of a 3-layer MLP: 2e-5 norm-wise
        assert rel_err(value[p].cpu().numpy().reshape(T + 1, N, -1), ref[p]["value"]) < 2e-5
        assert rel_err(action[p].cpu().numpy().reshape(T, N, -1), ref[p]["action"]) < 2e-5
        assert rel_err(logp[p].cpu().numpy().reshape(T, N), ref[p]["logp"]) < 2e-5


@pytest.mark.parametrize("name,T", [("walker", 40), ("walker", 300), ("humanoid", 300),    # 300 x 4 rows: tensor-core forwards
                                    ("ant", 300), ("swimmer", 40)])
def test_k1_modes(name, T):
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    P, N = 2, 4
    params, traj, eps, _, _, _, ref = make_case(d, P, T, N, seed=5)
    obs = dev(traj["obs"]).reshape(P, (T + 1) * N, d.obs)
    gp = dev(params)
    # deterministic: action == mean, logp = log N(mean | mean, std)
    value, action, logp = K.policy_forward(gp, obs, d, mode=K.ACT_DETERMINISTIC)
    for p in range(P):
        net = orc.Net(params[p].copy(), d.obs, d.act, d.obj)
        v, mean, _ = orc.forward(net, traj["obs"][p].reshape(-1, d.obs).astype(np.float64))
        assert rel_err(action[p].cpu().numpy(), mean) < 2e-5
        assert rel_err(logp[p].cpu().numpy(), orc.log_prob(net, mean, mean)) < 2e-5
        assert rel_err(value[p].cpu().numpy(), v) < 2e-5
    # evaluate: log-prob of given actions (a2c/model.py:75-82)
    given = dev(np.stack([r["action"].reshape(T * N, d.act) for r in ref]))
    value2, a2, logp2 = K.policy_forward(gp, obs, d, action=given, mode=K.ACT_EVALUATE, rows_a=T * N)
    assert a2.data_ptr() == given.data_ptr()
    for p in range(P):
        assert rel_err(logp2[p].cpu().numpy().reshape(T, N), ref[p]["logp"]) < 2e-5
    # get_value only
    v3, _, _ = K.policy_forward(gp, obs, d, rows_a=0, mode=K.ACT_DETERMINISTIC)
    assert torch.equal(v3, value)


@pytest.mark.parametrize("name", ["walker", "humanoid"])
def test_tensor_core_paths_with_unnormalised_observations(name):
    """The tensor-core kernels hold observations as UNSCALED fp16 pairs (range +-65 504, 22 significant bits) and parameters
    as pairs scaled by 2^8 (|w| < 255.9). Observations far outside VecNormalize's +-10 (ob_rms off, raw simulator output)
    still meet the FP32 tolerances on the tensor-core forward and update; a value BEYOND fp16's range does not get clamped
    silently: it turns that task's outputs into inf / NaN (csrc/tc_pair.cuh, pack_h2_ovf) and leaves other tasks alone."""
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    P, T, N = 2, 300 if name == "walker" else 150, 4 if name == "walker" else 8      # >= 1024 rows: tensor-core forward
    params, traj, eps, perm, _, _, _ = make_case(d, P, T, N, seed=23)
    params = params * 0.05                                      # small weights: tanh not saturated by inputs of size 300
    big = traj["obs"].astype(np.float64) * 300.0 + 40.0
    obs = dev(big).reshape(P, (T + 1) * N, d.obs)
    value, action, logp = K.policy_forward(dev(params), obs, d, mode=K.ACT_DETERMINISTIC)
    torch.cuda.synchronize()
    for p in range(P):
        net = orc.Net(dev(params[p]).cpu().numpy().astype(np.float64), d.obs, d.act, d.obj)
        v, mean, _ = orc.forward(net, obs[p].cpu().numpy().astype(np.float64))
        assert rel_err(value[p].cpu().numpy(), v) < 2e-5 and rel_err(action[p].cpu().numpy(), mean) < 2e-5
    # one PPO gradient on the tensor-core update kernel (cluster 32) with the same large observations
    S = T * N
    rng = np.random.RandomState(3)
    act = rng.randn(P, S, d.act); lp = rng.randn(P, S) * 0.1 - 5.0
    vold = value.cpu().numpy().astype(np.float64) + rng.randn(P, (T + 1) * N, d.obj) * 0.05
    ret = rng.randn(P, S, d.obj); adv = rng.randn(P, S)
    idx = rng.permutation(S)[:256 if name == "walker" else 512]
    g, _ = K.ppo_grad(dev(params), obs, dev(act), dev(lp), dev(vold), dev(ret), dev(adv), dev(idx, torch.int32), d, cluster=32)
    torch.cuda.synchronize()
    for p in range(P):
        net = orc.Net(dev(params[p]).cpu().numpy().astype(np.float64), d.obs, d.act, d.obj)
        f64 = lambda t: dev(t).cpu().numpy().astype(np.float64)
        gref, _ = orc.ppo_grad(net, obs[p].cpu().numpy().astype(np.float64)[:S][idx], f64(act[p])[idx], f64(lp[p])[idx],
                               f64(vold[p])[:S][idx], f64(ret[p])[idx], f64(adv[p])[idx])
        assert rel_err(g[p].cpu().numpy(), gref) < 5e-5
    # beyond fp16's range: loud, and confined to the task that holds the value
    bad = obs.clone()
    bad[1, 5, 3] = 1.0e5
    value, action, logp = K.policy_forward(dev(params), bad, d, mode=K.ACT_DETERMINISTIC)
    torch.cuda.synchronize()
    assert not torch.isfinite(value[1, 5]).all() or not torch.isfinite(action[1, 5]).all()
    assert torch.isfinite(value[0]).all() and torch.isfinite(action[0]).all()


@pytest.mark.parametrize("name,P,T,N", [("walker", 3, 64, 4), ("hopper3", 2, 45, 2), ("walker", 2, 2048, 4),
                                         ("walker", 1, 7, 1), ("humanoid", 2, 100, 8),
                                         # long rollouts of small populations: the segmented kernel (32 / N segments of the
                                         # time axis per env column), incl. a ragged last segment and N that does not divide 32
                                         ("humanoid", 2, 2048, 8), ("hopper3", 2, 1030, 3), ("walker", 6, 2048, 4),
                                         ("walker", 70, 700, 4)])      # > 64 tasks: one warp per column again
def test_k2_gae_adv_matches_oracle(name, P, T, N):
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    rng = np.random.RandomState(T)
    traj = {k: v.numpy() for k, v in synthetic.make_trajectories(P, T, N, d, seed=T, p_done=0.03).items()}
    value = rng.randn(P, T + 1, N, d.obj) * 3
    weights = rng.dirichlet(np.ones(d.obj), P)
    obj_var = rng.uniform(0.5, 2.0, (P, d.obj))
    ret, adv = K.gae_adv(dev(traj["rewards"]), dev(value), dev(traj["masks"]), dev(traj["bad_masks"]), 0.995, 0.95,
                         weights=dev(weights), obj_var=dev(obj_var))
    ret_only, none = K.gae_adv(dev(traj["rewards"]), dev(value), dev(traj["masks"]), dev(traj["bad_masks"]),
                               0.995, 0.95)
    torch.cuda.synchronize()
    assert none is None and torch.equal(ret_only, ret)
    v32 = dev(value).cpu().numpy().astype(np.float64)     # the kernel saw the float32-rounded values
    for p in range(P):
        r = orc.gae_returns(traj["rewards"][p].astype(np.float64), v32[p], traj["masks"][p].astype(np.float64),
                            traj["bad_masks"][p].astype(np.float64), 0.995, 0.95)
        a = orc.advantages(r, v32[p], weights[p], obj_var[p])
        assert rel_err(ret[p].cpu().numpy(), r) < 1e-5        # returns: 1e-5 (gate 1e-4)
        assert rel_err(adv[p].cpu().numpy(), a) < 1e-4        # normalised advantage: 1e-4


def _ppo_inputs(d, P, T, N, seed):
    params, traj, eps, perm, weights, obj_var, ref = make_case(d, P, T, N, seed)
    rng = np.random.RandomState(seed + 1)
    # evaluate at perturbed parameters so ratios leave 1 and the value clip is exercised
    cur = params + rng.randn(*params.shape) * 0.02
    S = T * N
    obs = traj["obs"].reshape(P, (T + 1) * N, d.obs)
    pack = dict(
        obs=obs, action=np.stack([r["action"].reshape(S, d.act) for r in ref]),
        logp=np.stack([r["logp"].reshape(S) for r in ref]),
        value=np.stack([r["value"].reshape((T + 1) * N, d.obj) for r in ref]),
        returns=np.stack([r["returns"].reshape(S, d.obj) for r in ref]),
        adv=np.stack([r["adv"].reshape(S) for r in ref]))
    return cur, pack, perm


# 32 / 64 / 128 = tensor-core paths (tcgen05): 2 / 4 / 8 CTAs per task; csrc/k3_tc.cuh (Walker2d, Hopper-v3 shapes),
# csrc/k3_tcw.cuh (Humanoid: layer 1 streamed in 64-feature blocks)
@pytest.mark.parametrize("cluster", [1, 2, 4, 8, 16, 32, 64, 128, 0])
@pytest.mark.parametrize("name,P,T,N,mb", [("walker", 2, 64, 4, 256), ("walker", 1, 30, 4, 100),
                                            ("hopper3", 2, 48, 2, 64), ("humanoid", 1, 32, 8, 96),
                                            ("humanoid", 2, 64, 8, 512), ("humanoid", 1, 40, 8, 300),
                                            ("hopper2", 2, 64, 4, 256), ("ant", 2, 64, 4, 256), ("swimmer", 2, 64, 4, 256),
                                            ("s16_16_2", 2, 64, 4, 256), ("s48_16_16", 2, 64, 4, 256),
                                            ("s45_16_3", 2, 64, 4, 256), ("s60_6_2", 2, 64, 4, 256),
                                            ("s64_4_4", 2, 64, 4, 256), ("s33_17_2", 2, 64, 4, 256)])
def test_k3_gradient_matches_oracle(name, P, T, N, mb, cluster):
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    if name == "humanoid" and cluster == 1:
        pytest.skip("wide networks need cluster >= 2 (both halves do not fit one CTA's shared memory)")
    if name != "humanoid" and cluster == 128:
        pytest.skip("8 CTAs per task exist on the wide-observation tensor-core path only")
    if name == "humanoid" and cluster == 16:
        pytest.skip("16-CTA clusters are a plan of the small-network FFMA kernel only")
    if name not in TC_SHAPES and cluster in (32, 64):
        pytest.skip("the tensor-core kernels are instantiated for the Walker2d, Hopper-v3 and Humanoid shapes only")
    cur, pk, perm = _ppo_inputs(d, P, T, N, seed=11)
    S = T * N
    idx = np.random.RandomState(0).permutation(S)[:mb]
    hyper = K.PpoHyper(entropy_coef=0.01)
    g, losses = K.ppo_grad(dev(cur), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]),
                           dev(pk["returns"]), dev(pk["adv"]), dev(idx, torch.int32), d, hyper=hyper,
                           cluster=cluster)
    torch.cuda.synchronize()
    for p in range(P):
        net = orc.Net(cur[p].copy(), d.obs, d.act, d.obj)
        gref, lref = orc.ppo_grad(net, pk["obs"][p][:S][idx].astype(np.float64), pk["action"][p][idx],
                                  pk["logp"][p][idx], pk["value"][p][:S][idx], pk["returns"][p][idx],
                                  pk["adv"][p][idx], ecoef=0.01)
        # FP32 gradient of a mean over <=256 rows: 5e-5 norm-wise per tensor group (whole vector)
        assert rel_err(g[p].cpu().numpy(), gref) < 5e-5
        assert rel_err(losses[p].cpu().numpy(), np.array(lref)) < 2e-5


@pytest.mark.parametrize("cluster", [0, 1, 2, 4, 8, 16, 32, 64])
@pytest.mark.parametrize("name,P,T,N,B", [("walker", 3, 64, 4, 4), ("hopper3", 2, 48, 2, 3), ("walker", 2, 160, 4, 2),
                                          ("hopper2", 2, 64, 4, 2), ("ant", 3, 64, 4, 2), ("swimmer", 2, 64, 4, 2),
                                          ("s16_16_2", 2, 64, 4, 2), ("s45_16_3", 2, 128, 4, 2), ("s60_6_2", 2, 64, 4, 2),
                                          ("s33_17_2", 2, 64, 4, 2),
                                          # 40 tasks: the auto plan keeps two CTAs per task (Ant: TM = 2 fallback)
                                          ("ant", 40, 32, 4, 1)])
def test_k3_update_matches_oracle(name, P, T, N, B, cluster):
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    if name not in TC_SHAPES and cluster in (32, 64):
        pytest.skip("the tensor-core kernels are instantiated for the Walker2d, Hopper-v3 and Humanoid shapes only")
    if P > 3 and cluster != 0:
        pytest.skip("the large population runs the auto plan only")
    cur, pk, perm = _ppo_inputs(d, P, T, N, seed=13)
    S = T * N
    rng = np.random.RandomState(2)
    m0 = rng.randn(P, d.n_par) * 1e-3
    v0 = rng.rand(P, d.n_par) * 1e-5
    step0 = np.resize(np.array([0, 7, 640], dtype=np.int32), P)
    lr = np.resize(np.array([3e-4, 2.5e-4, 1e-4]), P)
    gp, gm, gv = dev(cur), dev(m0), dev(v0)
    gstep = dev(step0, torch.int32)
    losses = K.ppo_update(gp, gm, gv, gstep, dev(lr, torch.float64), dev(pk["obs"]), dev(pk["action"]),
                          dev(pk["logp"]), dev(pk["value"]), dev(pk["returns"]), dev(pk["adv"]),
                          dev(perm[None], torch.int32), B, d, cluster=cluster)
    torch.cuda.synchronize()
    for p in range(P):
        flat = dev(cur[p]).cpu().numpy().astype(np.float64)
        m = dev(m0[p]).cpu().numpy().astype(np.float64)
        v = dev(v0[p]).cpu().numpy().astype(np.float64)
        obs3 = pk["obs"][p].reshape(T + 1, N, d.obs).astype(np.float64)
        step, lref = orc.ppo_update(flat, m, v, int(step0[p]), lr[p], (d.obs, d.act, d.obj), obs3,
                                    pk["action"][p].reshape(T, N, -1), pk["logp"][p].reshape(T, N),
                                    pk["value"][p].reshape(T + 1, N, -1), pk["returns"][p].reshape(T, N, -1),
                                    pk["adv"][p].reshape(T, N), perm, B)
        assert int(gstep[p]) == step
        assert rel_err(gp[p].cpu().numpy(), flat) < 1e-5       # parameters (gate 1e-4)
        assert rel_err(gm[p].cpu().numpy(), m) < 1e-4          # Adam first moment
        assert rel_err(gv[p].cpu().numpy(), v) < 1e-4          # Adam second moment
        assert rel_err(losses[p].cpu().numpy(), np.array(lref)) < 1e-4


# flags OR-ed into `cluster`: alternative step tails of the FFMA cluster kernel (csrc/k3_fast.cuh)
@pytest.mark.parametrize("P,expect_waves", [(160, True), (74, False), (37, False), (75, True)])
def test_k3_update_large_populations_auto_plan(P, expect_waves):
    """Populations larger than one wave of clusters (the auto plan's tensor-core kernel with 2 CTAs per task: 148 SMs hold
    74 tasks at once; P = 160 runs three waves) and the plan boundaries P = 37 (last size with 4 CTAs per task... first with
    2) and 74 / 75 (last single wave / first with a second wave): parameters, moments and step of tasks at the wave
    boundaries against the float64 oracle, same tolerances as the small-population tests."""
    from pgmorl_b200 import kernels as K
    d = DIMS["walker"]
    T, N, B = 32, 4, 1                                     # one minibatch of 128 rows (one row tile), E epochs
    cur1, pk1, perm = _ppo_inputs(d, 4, T, N, seed=19)     # 4 distinct tasks, tiled to P with per-task parameter offsets
    rng = np.random.RandomState(5)
    reps = (P + 3) // 4
    cur = np.tile(cur1, (reps, 1))[:P] + rng.randn(P, d.n_par) * 1e-3
    pk = {k: np.tile(v, (reps,) + (1,) * (v.ndim - 1))[:P] for k, v in pk1.items()}
    S = T * N
    lr = np.full(P, 3e-4)
    gp, gm, gv = dev(cur), torch.zeros(P, d.n_par, device="cuda"), torch.zeros(P, d.n_par, device="cuda")
    gstep = torch.zeros(P, dtype=torch.int32, device="cuda")
    K.ppo_update(gp, gm, gv, gstep, dev(lr, torch.float64), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]),
                 dev(pk["value"]), dev(pk["returns"]), dev(pk["adv"]), dev(perm[None], torch.int32), B, d, cluster=0)
    torch.cuda.synchronize()
    assert torch.isfinite(gp).all()
    check = sorted({0, 1, 36, 37, 73, 74, 75, 147, 148, P - 1} & set(range(P)))
    for p in check:
        flat = dev(cur[p]).cpu().numpy().astype(np.float64)
        m, v = np.zeros_like(flat), np.zeros_like(flat)
        obs3 = pk["obs"][p].reshape(T + 1, N, d.obs).astype(np.float64)
        step, _ = orc.ppo_update(flat, m, v, 0, lr[p], (d.obs, d.act, d.obj), obs3, pk["action"][p].reshape(T, N, -1),
                                 pk["logp"][p].reshape(T, N), pk["value"][p].reshape(T + 1, N, -1),
                                 pk["returns"][p].reshape(T, N, -1), pk["adv"][p].reshape(T, N), perm, B)
        assert int(gstep[p]) == step
        assert rel_err(gp[p].cpu().numpy(), flat) < 1e-5, p
        assert rel_err(gm[p].cpu().numpy(), m) < 1e-4, p
        assert rel_err(gv[p].cpu().numpy(), v) < 1e-4, p


TAIL2 = 0x100     # two-barrier tail: tiles pushed to the slice owner, whole-half Adam in every CTA
TAILMC = 0x200    # parameter broadcast through the TMA (cp.async.bulk with cluster multicast) instead of DSMEM stores
TAILGL = 0x400    # TAILMC + gradient exchange through L2 scratch slots instead of distributed shared memory
TAIL0 = 0x800     # the plain three-barrier DSMEM tail
TAILBP = 0x1000   # TAILMC + gradient reduce-scatter pushed by cp.async.bulk (shared::cta -> shared::cluster), one barrier left
TAILNB = 0x2000   # TAILBP + norm partials by st.async with mbarrier completion: no cluster barrier inside the step
TAILEP = 0x4000   # TAILNB + the W2-only gradient slices are pushed right after the {dW2, dz1} phase


@pytest.mark.parametrize("cluster", [4, 8, 16])
@pytest.mark.parametrize("name,P,T,N,B", [("walker", 3, 64, 4, 4), ("hopper3", 2, 48, 2, 3), ("walker", 2, 512, 4, 8),
                                          # phase-C plans of the fast kernel the named shapes above do not reach
                                          ("hopper2", 2, 64, 4, 1), ("ant", 2, 64, 4, 1), ("swimmer", 2, 64, 4, 1),
                                          ("s16_16_2", 2, 64, 4, 1), ("s48_16_16", 2, 64, 4, 1)])
def test_k3_step_tails_bit_identical(name, P, T, N, B, cluster):
    """The alternative step tails (two-barrier tail with whole-half Adam in every CTA; TMA multicast parameter broadcast)
    perform the same operations in the same order as the three-barrier sliced tail: parameters, moments and losses are
    equal bit for bit, and so is the raw gradient."""
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    cur, pk, perm = _ppo_inputs(d, P, T, N, seed=17)
    hyper = K.PpoHyper(entropy_coef=0.01)
    lr = dev(np.array([3e-4, 2.5e-4, 1e-4][:P]), torch.float64)
    out = []
    for cl in (cluster, cluster | TAIL0, cluster | TAIL2, cluster | TAILMC, cluster | TAILGL, cluster | TAILBP, cluster | TAILNB, cluster | TAILEP):
        gp, gm, gv = dev(cur), torch.zeros(P, d.n_par, device="cuda"), torch.zeros(P, d.n_par, device="cuda")
        gstep = torch.zeros(P, dtype=torch.int32, device="cuda")
        losses = K.ppo_update(gp, gm, gv, gstep, lr, dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]),
                              dev(pk["returns"]), dev(pk["adv"]), dev(perm[None], torch.int32), B, d, hyper=hyper, cluster=cl)
        idx = np.random.RandomState(0).permutation(T * N)[:max(T * N // B, 1)]
        g, gl = K.ppo_grad(dev(cur), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]),
                           dev(pk["returns"]), dev(pk["adv"]), dev(idx, torch.int32), d, hyper=hyper, cluster=cl)
        torch.cuda.synchronize()
        out.append((gp, gm, gv, gstep, losses, g, gl))
    for other in out[1:]:
        for x, y in zip(out[0], other):
            assert torch.equal(x, y)
    assert int(out[0][3][0]) == perm.shape[0] * B


@pytest.mark.parametrize("cluster", [0, 8, 32, 64, 128])
@pytest.mark.parametrize("T,N,B", [(48, 8, 1), (48, 8, 3), (64, 8, 1)])       # minibatches of 384 (3 row tiles), 128, 512 rows
def test_k3_update_matches_oracle_humanoid(T, N, B, cluster):
    """the update on Humanoid dims: generic FFMA path (cluster 8) and the wide tensor-core kernel with 1 / 2 / 4 CTAs
    per network half (32 / 64 / 128; 0 = auto), same tolerances as the other shapes"""
    from pgmorl_b200 import kernels as K
    d, P = DIMS["humanoid"], 2
    cur, pk, perm = _ppo_inputs(d, P, T, N, seed=19)
    rng = np.random.RandomState(3)
    m0, v0 = rng.randn(P, d.n_par) * 1e-3, rng.rand(P, d.n_par) * 1e-5
    step0, lr = np.array([0, 7], dtype=np.int32), np.array([3e-4, 2.5e-4])
    gp, gm, gv, gstep = dev(cur), dev(m0), dev(v0), dev(step0, torch.int32)
    losses = K.ppo_update(gp, gm, gv, gstep, dev(lr, torch.float64), dev(pk["obs"]), dev(pk["action"]),
                          dev(pk["logp"]), dev(pk["value"]), dev(pk["returns"]), dev(pk["adv"]),
                          dev(perm[None], torch.int32), B, d, cluster=cluster)
    torch.cuda.synchronize()
    for p in range(P):
        flat, m, v = (dev(t[p]).cpu().numpy().astype(np.float64) for t in (cur, m0, v0))
        step, lref = orc.ppo_update(flat, m, v, int(step0[p]), lr[p], (d.obs, d.act, d.obj),
                                    pk["obs"][p].reshape(T + 1, N, d.obs).astype(np.float64),
                                    pk["action"][p].reshape(T, N, -1), pk["logp"][p].reshape(T, N),
                                    pk["value"][p].reshape(T + 1, N, -1), pk["returns"][p].reshape(T, N, -1),
                                    pk["adv"][p].reshape(T, N), perm, B)
        assert int(gstep[p]) == step
        assert rel_err(gp[p].cpu().numpy(), flat) < 1e-5
        assert rel_err(gm[p].cpu().numpy(), m) < 1e-4 and rel_err(gv[p].cpu().numpy(), v) < 1e-4
        assert rel_err(losses[p].cpu().numpy(), np.array(lref)) < 1e-4


@pytest.mark.parametrize("cluster", [0, 8, 32, 64])
def test_full_size_c2_iteration_matches_reference_golden(cluster):
    """BASELINE.json configs[1] at full size (2 of the 6 tasks: T=2048, N=4, 10 epochs x 32 minibatches = 320 Adam
    steps) through the population API, against the UNMODIFIED reference's outputs (mopg_halfcheetah_full.npz).
    Gate: 1e-4 norm-wise on parameters and returns (north_star), Adam moments 1e-3."""
    from pgmorl_b200.population_state import PopulationMOPG
    from tests.helpers import load_mopg_case
    z, meta = load_mopg_case("mopg_halfcheetah_full.npz")
    d, P, T, N = meta["dims"], meta["n_tasks"], meta["T"], meta["N"]
    j = meta["iters"][0]
    pop = PopulationMOPG(d, P, T, N, ppo_epoch=meta["E"], num_mini_batch=meta["B"], gamma=meta["gamma"],
                         gae_lambda=meta["lam"], cluster=cluster)
    for p in range(P):
        pop.load_task(p, z[f"t{p}_init"], weights=z[f"t{p}_weights"], obj_var=z[f"t{p}_obj_var"])
    pop.set_lr(synthetic.linear_lr(3e-4, j, 1.0, meta["total_num_updates"]))
    traj = synthetic.make_trajectories(P, T, N, d, seed=meta["traj_seed"] + j)
    eps, perm = synthetic.host_rng_streams(j, T, N, d.act, meta["E"])
    losses = pop.step_from_host(traj["obs"], traj["rewards"], traj["masks"], traj["bad_masks"],
                                eps.to(torch.float32), perm.to(torch.int32))
    for p in range(P):
        pre = f"t{p}_i0_"
        flat, m, v, step = pop.task_state(p)
        assert step == int(z[pre + "adam_step"]) == 320
        assert rel_err(pop.returns[p].cpu().numpy(), z[pre + "returns"]) < 1e-4
        assert rel_err(pop.adv[p].cpu().numpy(), z[pre + "adv"]) < 1e-4
        assert rel_err(flat, z[pre + "params"]) < 1e-4
        assert rel_err(m, z[pre + "adam_m"]) < 1e-3 and rel_err(v, z[pre + "adam_v"]) < 1e-3
        assert rel_err(losses[p], z[pre + "losses"]) < 1e-3


@pytest.mark.parametrize("name", ["mopg_humanoid_small.npz", "mopg_hopper3_small.npz", "mopg_walker_small.npz"])
def test_population_iterations_match_reference_goldens(name):
    """Whole MOPG iterations (K1 -> K2 -> K3) for every task and every recorded iteration of the small goldens,
    state carried across iterations, through PopulationMOPG. Humanoid dims (O = 376) take the split-half K1 and the
    generic K3 path. Gate 1e-4 norm-wise (north_star); moments 1e-3."""
    from pgmorl_b200.population_state import PopulationMOPG
    from tests.helpers import load_mopg_case
    z, meta = load_mopg_case(name)
    d, P, T, N = meta["dims"], meta["n_tasks"], meta["T"], meta["N"]
    pop = PopulationMOPG(d, P, T, N, ppo_epoch=meta["E"], num_mini_batch=meta["B"], gamma=meta["gamma"],
                         gae_lambda=meta["lam"])
    for p in range(P):
        pop.load_task(p, z[f"t{p}_init"], weights=z[f"t{p}_weights"], obj_var=z[f"t{p}_obj_var"])
    for k, j in enumerate(meta["iters"]):
        pop.set_lr(synthetic.linear_lr(3e-4, j, 1.0, meta["total_num_updates"]))
        traj = synthetic.make_trajectories(P, T, N, d, seed=meta["traj_seed"] + j)
        eps, perm = synthetic.host_rng_streams(j, T, N, d.act, meta["E"])
        losses = pop.step_from_host(traj["obs"], traj["rewards"], traj["masks"], traj["bad_masks"],
                                    eps.to(torch.float32), perm.to(torch.int32))
        for p in range(P):
            pre = f"t{p}_i{k}_"
            flat, m, v, step = pop.task_state(p)
            assert step == int(z[pre + "adam_step"])
            assert rel_err(pop.value[p].cpu().numpy().reshape(T + 1, N, -1), z[pre + "value"]) < 1e-4
            assert rel_err(pop.action[p].cpu().numpy().reshape(T, N, -1), z[pre + "action"]) < 1e-4
            assert rel_err(pop.returns[p].cpu().numpy(), z[pre + "returns"]) < 1e-4
            assert rel_err(pop.adv[p].cpu().numpy(), z[pre + "adv"]) < 1e-4
            assert rel_err(flat, z[pre + "params"]) < 1e-4
            assert rel_err(m, z[pre + "adam_m"]) < 1e-3 and rel_err(v, z[pre + "adam_v"]) < 1e-3
            assert rel_err(losses[p], z[pre + "losses"]) < 1e-3


@pytest.mark.parametrize("name,cluster", [pytest.param("walker", c, id=str(c)) for c in (8, 32, 64)] +
                         [("ant", 2), ("ant", 16), ("s45_16_3", 8), ("s33_17_2", 4), ("swimmer", 1)])
def test_k3_per_task_permutations_equal_shared(name, cluster):
    """perm given per task ([P,E,S]) with identical rows must reproduce the shared-permutation ([1,E,S]) result bit for bit
    (the reference seeds every worker alike, mopg.py:96, but the C ABI accepts per-task streams)."""
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    P, T, N, B = 3, 96, 4, 2                       # mb = 192: two row tiles on the tensor-core path, the second one ragged
    cur, pk, perm = _ppo_inputs(d, P, T, N, seed=17)
    res = []
    for shared in (True, False):
        gp, gm, gv = dev(cur), torch.zeros(P, d.n_par, device="cuda"), torch.zeros(P, d.n_par, device="cuda")
        gstep = torch.zeros(P, dtype=torch.int32, device="cuda")
        pm = dev(perm[None], torch.int32)
        if not shared:
            pm = pm.expand(P, -1, -1).contiguous()
        K.ppo_update(gp, gm, gv, gstep, dev(np.full(P, 3e-4), torch.float64), dev(pk["obs"]), dev(pk["action"]),
                     dev(pk["logp"]), dev(pk["value"]), dev(pk["returns"]), dev(pk["adv"]), pm, B, d, cluster=cluster)
        torch.cuda.synchronize()
        res.append((gp.clone(), gm.clone(), gv.clone()))
    for a, b in zip(*res):
        assert torch.equal(a, b)
