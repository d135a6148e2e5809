"""Categorical heads (Discrete(n) actions) on the CPU: the two float64 restatements of tests/discrete_ref.py (numpy with a
hand-derived backward, torch.distributions.Categorical with autograd) agree, torch's Categorical sampling is the argmax
of probs over Exponential(1) draws with the same generator consumption, the initialisation follows the reference's
construction order, and the C ABI's parameter layout follows layout.param_layout.

No reference golden exists for Categorical heads; the agreement of the two restatements here is the pin of the GPU
tests in tests/test_gpu_discrete.py."""
import ctypes

import numpy as np
import pytest
import torch

import discrete_ref as dref
from pgmorl_b200 import synthetic
from pgmorl_b200.layout import DIST_CATEGORICAL, NetDims, param_layout
from tests.helpers import rel_err

# (O, n, M): Deep-Sea-Treasure-like, a mid shape, a wide head (n > 16), O > 64, and the three (O, n, M) that equal
# Gaussian shapes with tensor-core instantiations
SHAPES = {"dst": (2, 4, 2), "mid": (11, 9, 3), "wide_head": (33, 18, 2), "wide_obs": (70, 5, 2),
          "tc_walker": (17, 6, 2), "tc_hopper3": (11, 3, 3), "tcw_humanoid": (376, 17, 2)}


def cat_dims(O, n, M, H=64):
    return NetDims(O, n, M, H, DIST_CATEGORICAL)


@pytest.mark.parametrize("H", [32, 64, 128])
@pytest.mark.parametrize("shape", ["dst", "mid", "wide_head"])
@pytest.mark.parametrize("ecoef", [0.0, 0.01])
def test_forward_and_gradient_numpy_equals_torch(shape, H, ecoef):
    d = cat_dims(*SHAPES[shape], H)
    rng = np.random.RandomState(3)
    flat = synthetic.init_policy_flat(d, seed=7).numpy()
    lay, _ = param_layout(d)
    off, shp = lay["dist.linear.weight"]
    flat[off:off + d.act * H] = rng.randn(d.act * H) * 0.3           # logits of order one, not the 0.01-gain init
    mb = 48
    x = rng.randn(mb, d.obs)
    action = rng.randint(0, d.act, mb)
    net = dref.net_of(flat.copy(), d)
    value, z, _ = dref.forward(net, x)
    pol = dref.PortCatPolicy(flat, d.obs, d.act, d.obj, H)
    xt = torch.as_tensor(x)
    with torch.no_grad():
        v_t, ha = pol.base(xt)
        dist = pol.dist(ha)
    assert rel_err(value, v_t.numpy()) < 1e-12 and rel_err(z, pol.linear(ha).detach().numpy()) < 1e-12
    lsm = dref.log_softmax(z)
    assert rel_err(lsm[np.arange(mb), action], dist.log_prob(torch.as_tensor(action)).numpy()) < 1e-12
    assert rel_err(dref.entropy_rows(z), dist.entropy().numpy()) < 1e-12
    logp_old, adv = lsm[np.arange(mb), action] + rng.randn(mb) * 0.2, rng.randn(mb)
    v_old, ret = value + rng.randn(mb, d.obj) * 0.4, value + rng.randn(mb, d.obj)
    for clipped in (True, False):
        g, losses = dref.ppo_grad(net, x, action, logp_old, v_old, ret, adv, ecoef=ecoef, clipped_value_loss=clipped)
        gt, lt = dref.port_grad(pol, x, action, logp_old, v_old, ret, adv, ecoef=ecoef, clipped_value_loss=clipped)
        assert g.size == d.n_par
        assert rel_err(g, gt) < 1e-12
        assert rel_err(np.array(losses), np.array(lt)) < 1e-12


@pytest.mark.parametrize("H", [32, 64, 128])
@pytest.mark.parametrize("shape", ["dst", "mid", "wide_head"])
def test_iteration_numpy_equals_torch_port(shape, H):
    """one whole MOPG iteration: per-step sampling from the global generator, GAE, advantage, E x B Adam steps"""
    d = cat_dims(*SHAPES[shape], H)
    T, N, E, B, j = 24, 4, 2, 3, 5
    flat0 = synthetic.init_policy_flat(d, seed=13).numpy()
    traj = {k: v[0].numpy() for k, v in synthetic.make_trajectories(1, T, N, d, seed=9, p_done=0.1).items()}
    weights = np.full(d.obj, 1.0 / d.obj)
    obj_var = np.linspace(0.6, 1.4, d.obj)
    q, perm = synthetic.host_rng_streams(j, T, N, d.act, E, categorical=True)
    flat, m, v = flat0.copy(), np.zeros_like(flat0), np.zeros_like(flat0)
    out = dref.mopg_iteration(flat, m, v, 0, 3e-4, d, traj, q.numpy(), perm.numpy(), weights, obj_var,
                              num_mini_batch=B, ecoef=0.01)
    pol = dref.PortCatPolicy(flat0, d.obs, d.act, d.obj, H)
    opt = torch.optim.Adam(pol.ordered(), lr=3e-4, eps=1e-5)
    port = dref.mopg_iteration_port(pol, opt, traj, j, 3e-4, weights, obj_var, ppo_epoch=E, num_mini_batch=B,
                                    ecoef=0.01)
    assert np.array_equal(out["action"], port["action"])
    assert rel_err(out["logp"], port["logp"]) < 1e-12
    assert rel_err(out["returns"], port["returns"]) < 1e-12
    assert rel_err(out["adv"], port["adv"]) < 1e-12
    assert rel_err(out["losses"], port["losses"]) < 1e-9
    assert rel_err(flat, pol.flat()) < 1e-9
    assert out["step"] == E * B and rel_err(flat, flat0) > 1e-6


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_sample_is_argmax_over_exponential_draws(dtype):
    """Categorical(logits).sample() after manual_seed(j) == first argmax of probs / exponential_(1), drawn as float64
    [N,n], and leaves the generator where that draw leaves it"""
    for j in range(200):
        g = torch.Generator().manual_seed(10_000 + j)
        n, N = 2 + j % 30, 1 + j % 7
        logits = torch.randn(N, n, generator=g, dtype=dtype) * (0.1 + j % 5)
        torch.manual_seed(j)
        a = torch.distributions.Categorical(logits=logits).sample()
        after_sample = torch.get_rng_state()
        torch.manual_seed(j)
        q = torch.empty(N, n, dtype=torch.float64).exponential_(1)
        assert torch.equal(torch.get_rng_state(), after_sample)
        probs = torch.distributions.Categorical(logits=logits).probs
        assert torch.equal(a, (probs / q.to(dtype)).argmax(-1))


def test_host_rng_streams_categorical():
    q, perm = synthetic.host_rng_streams(3, 5, 4, 6, 2, categorical=True)
    torch.manual_seed(3)
    want = torch.stack([torch.empty(4, 6, dtype=torch.float64).exponential_(1) for _ in range(5)])
    assert torch.equal(q, want) and torch.equal(perm[0], torch.randperm(20)) and torch.equal(perm[1], torch.randperm(20))


@pytest.mark.parametrize("H", [32, 64, 128])
def test_init_equals_reference_construction(H):
    """base in the reference's order, then dist.linear = nn.Linear(H, n) with orthogonal_(gain 0.01) and zero bias"""
    d = cat_dims(*SHAPES["mid"], H)
    got = synthetic.init_policy_flat(d, seed=21).numpy()
    torch.manual_seed(21)
    g2 = float(np.sqrt(2))
    mods = []
    for i, o, gain in ((d.obs, H, g2), (H, H, g2), (d.obs, H, g2), (H, H, g2), (H, 1, g2), (H, d.obj, g2),
                       (H, d.act, 0.01)):
        lin = torch.nn.Linear(i, o, dtype=torch.float64)
        torch.nn.init.orthogonal_(lin.weight.data, gain=gain)
        torch.nn.init.constant_(lin.bias.data, 0)
        mods.append(lin)
    pol = dref.PortCatPolicy(None, d.obs, d.act, d.obj, H)
    a0, a2, c0, c2, _, cl, lin = mods
    for dst, src in zip(pol.ordered(), (a0.weight, a0.bias, a2.weight, a2.bias, c0.weight, c0.bias, c2.weight, c2.bias,
                                        cl.weight, cl.bias, lin.weight, lin.bias)):
        dst.data.copy_(src.data)
    assert got.shape == (d.n_par,) and np.array_equal(got, pol.flat())
    layout, _ = param_layout(d)
    assert list(layout)[-2:] == ["dist.linear.weight", "dist.linear.bias"] and len(layout) == 12
    assert layout["dist.linear.weight"][1] == (d.act, H)


def test_c_abi_layout_follows_param_layout():
    from pgmorl_b200._lib import lib
    L = lib()
    for O, n, M in SHAPES.values():
        for H in (32, 64, 128):
            d = cat_dims(O, n, M, H)
            layout, npar = param_layout(d)
            assert L.pgm_n_par_x(O, n, M, H, DIST_CATEGORICAL) == npar
            out = (ctypes.c_int * 13)(*([-7] * 13))
            assert L.pgm_param_offsets_x(O, n, M, H, DIST_CATEGORICAL, out) == 0
            assert list(out)[:12] == [off for off, _ in layout.values()] and out[12] == -7
            g = NetDims(O, n, M, H)
            og, oh = (ctypes.c_int * 13)(), (ctypes.c_int * 13)()
            assert L.pgm_param_offsets_x(O, n, M, H, 0, og) == 0 and L.pgm_param_offsets_h(O, n, M, H, oh) == 0
            assert list(og) == list(oh) == [off for off, _ in param_layout(g)[0].values()]
            assert L.pgm_n_par_x(O, n, M, H, 0) == L.pgm_n_par_h(O, n, M, H) == g.n_par
    assert L.pgm_n_par_x(2, 33, 2, 64, DIST_CATEGORICAL) == -1 and b"1..32 categories" in L.pgm_last_error()
    assert L.pgm_n_par_x(2, 4, 2, 64, 7) == -1 and b"unknown action head" in L.pgm_last_error()
    assert L.pgm_ppo_workspace_bytes_x(2, 64, 2, 4, 2, 0, 64, 7) == 0
    assert L.pgm_ppo_workspace_bytes_x(2, 64, 17, 6, 2, 0, 64, 0) == L.pgm_ppo_workspace_bytes_h(2, 64, 17, 6, 2, 0, 64)


def test_policy_and_storage_accept_discrete():
    from pgmorl_b200.a2c_ppo_acktr.algo.ppo import DeviceAdam
    from pgmorl_b200.a2c_ppo_acktr.model import Policy
    from pgmorl_b200.a2c_ppo_acktr.storage import RolloutStorage

    class Discrete:
        def __init__(self, n):
            self.n = n

    pol = Policy((2,), Discrete(4), base_kwargs={"layernorm": False}, obj_num=2, device="cpu")
    assert pol.dims == cat_dims(2, 4, 2)
    sd = pol.state_dict()
    assert sd["dist.linear.weight"].shape == (4, 64) and sd["dist.linear.bias"].shape == (4,)
    assert not any("logstd" in k or "fc_mean" in k for k in sd)
    pol2 = Policy((2,), Discrete(4), base_kwargs={"layernorm": False}, obj_num=2, device="cpu")
    pol2.load_state_dict(sd)
    assert torch.equal(pol2.flat, pol.flat)
    opt = DeviceAdam(pol, 3e-4, 1e-5)
    assert opt.param_groups[0]["params"] == list(range(12))
    st = RolloutStorage(5, 3, (2,), Discrete(4), 1, obj_num=2, device="cpu")
    assert st.actions.shape == (5, 3, 1) and st.actions.dtype == torch.int64
    with pytest.raises(NotImplementedError, match="1 to 32"):
        Policy((2,), Discrete(33), base_kwargs={"layernorm": False}, obj_num=2, device="cpu")
