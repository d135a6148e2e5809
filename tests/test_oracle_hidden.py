"""Hidden widths 32 and 128 on the CPU: the two float64 restatements (numpy with a hand-derived backward, torch nn.Linear
with autograd) agree at these widths, the initialisation follows the reference's construction order, the C ABI's
parameter layout follows layout.param_layout, and Policy refuses a width the kernels are not built for.

No reference golden exists at a width other than 64; the two oracles are pinned to the goldens at 64
(tests/test_oracle_mopg.py) and take the width as a parameter, so their agreement here is the pin of the GPU tests in
tests/test_gpu_hidden.py."""
import numpy as np
import pytest
import torch

import hidden_ref
from oracle import mopg_oracle as orc
from oracle.mopg_torch_port import PortPolicy, mopg_iteration_port
from pgmorl_b200 import synthetic
from pgmorl_b200.layout import ENV_SHAPES, NetDims, param_layout
from tests.helpers import rel_err

WIDTHS = (32, 128)
SHAPES = {"walker": (17, 6, 2), "hopper3": (11, 3, 3), "ant": (27, 8, 2)}


def _dims(shape, H):
    return NetDims(*SHAPES[shape], hidden=H)


@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("shape", SHAPES)
def test_forward_and_gradient_numpy_equals_torch(shape, H):
    d = _dims(shape, H)
    rng = np.random.RandomState(3)
    flat = synthetic.init_policy_flat(d, seed=7).numpy()
    flat[-d.act:] = rng.uniform(-0.5, 0.3, d.act)
    mb = 48
    x, action = rng.randn(mb, d.obs), rng.randn(mb, d.act)
    net = orc.Net(flat.copy(), d.obs, d.act, d.obj, H)
    value, mean, _ = orc.forward(net, x)
    pol = PortPolicy(flat, d.obs, d.act, d.obj, H)
    xt = torch.as_tensor(x)
    with torch.no_grad():
        v_t, ha = pol.base(xt)
        mean_t = pol.fm(ha)
    assert rel_err(value, v_t.numpy()) < 1e-12 and rel_err(mean, mean_t.numpy()) < 1e-12
    logp_old, adv = rng.randn(mb) * 0.3 - 6.0, rng.randn(mb)
    v_old = value + rng.randn(mb, d.obj) * 0.4
    ret = value + rng.randn(mb, d.obj)
    g, losses = orc.ppo_grad(net, x, action, logp_old, v_old, ret, adv, ecoef=0.01)
    values, logp, ent = pol.evaluate_actions(xt, torch.as_tensor(action))
    ratio = torch.exp(logp - torch.as_tensor(logp_old)[:, None])
    at = torch.as_tensor(adv)[:, None]
    action_loss = -torch.min(ratio * at, torch.clamp(ratio, 0.8, 1.2) * at).mean()
    vo, rt = torch.as_tensor(v_old), torch.as_tensor(ret)
    vclip = vo + (values - vo).clamp(-0.2, 0.2)
    value_loss = 0.5 * torch.max((values - rt).pow(2), (vclip - rt).pow(2)).mean()
    pol.zero_grad()
    (value_loss * 0.5 + action_loss - ent * 0.01).backward()
    gt = torch.cat([p.grad.reshape(-1) for p in pol.ordered()]).numpy()
    assert g.size == d.n_par
    assert rel_err(g, gt) < 1e-12
    assert rel_err(np.array(losses), np.array([value_loss.item(), action_loss.item(), ent.item()])) < 1e-12


@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("shape", SHAPES)
def test_iteration_numpy_equals_torch_port(shape, H):
    """one whole MOPG iteration (rollout, GAE, advantage, E x B dependent Adam steps)"""
    d = _dims(shape, H)
    T, N, E, B, j = 24, 4, 2, 3, 5
    flat0 = synthetic.init_policy_flat(d, seed=13).numpy()
    traj = {k: v[0].numpy() for k, v in synthetic.make_trajectories(1, T, N, d, seed=9, p_done=0.1).items()}
    weights = np.full(d.obj, 1.0 / d.obj)
    obj_var = np.linspace(0.6, 1.4, d.obj)
    eps, perm = synthetic.host_rng_streams(j, T, N, d.act, E)
    flat, m, v = flat0.copy(), np.zeros_like(flat0), np.zeros_like(flat0)
    out = hidden_ref.mopg_iteration(flat, m, v, 0, 3e-4, d, traj, eps.numpy(), perm.numpy(), weights, obj_var,
                                    num_mini_batch=B)
    pol = PortPolicy(flat0, d.obs, d.act, d.obj, H)
    opt = torch.optim.Adam(pol.ordered(), lr=3e-4, eps=1e-5)
    port = mopg_iteration_port(pol, opt, traj, j, 3e-4, weights, obj_var, ppo_epoch=E, num_mini_batch=B)
    assert rel_err(out["returns"], port["returns"]) < 1e-12
    assert rel_err(out["adv"], port["adv"]) < 1e-12
    assert rel_err(out["losses"], port["losses"]) < 1e-9
    assert rel_err(flat, pol.flat()) < 1e-9
    assert out["step"] == E * B and rel_err(flat, flat0) > 1e-6


@pytest.mark.parametrize("H", WIDTHS)
def test_init_equals_nn_linear_construction(H):
    """init_policy_flat at width H draws from torch's generator in the reference's order: actor.0, actor.2, critic.0,
    critic.2, MLPBase.critic_linear (replaced), MOMLPBase.critic_linear, fc_mean; each nn.Linear default init, then
    orthogonal_ with the reference's gain and zero bias"""
    d = _dims("walker", H)
    got = synthetic.init_policy_flat(d, seed=21).numpy()
    torch.manual_seed(21)
    g2 = float(np.sqrt(2))
    mods = []
    for i, o, gain in ((d.obs, H, g2), (H, H, g2), (d.obs, H, g2), (H, H, g2), (H, 1, g2), (H, d.obj, g2),
                       (H, d.act, 1.0)):
        lin = torch.nn.Linear(i, o, dtype=torch.float64)
        torch.nn.init.orthogonal_(lin.weight.data, gain=gain)
        torch.nn.init.constant_(lin.bias.data, 0)
        mods.append(lin)
    a0, a2, c0, c2, _, cl, fm = mods
    want = torch.cat([t.detach().reshape(-1) for t in (a0.weight, a0.bias, a2.weight, a2.bias, c0.weight, c0.bias,
                                                       c2.weight, c2.bias, cl.weight, cl.bias, fm.weight, fm.bias)]
                     + [torch.zeros(d.act, dtype=torch.float64)]).numpy()
    assert got.shape == (d.n_par,) and np.array_equal(got, want)
    layout, _ = param_layout(d)
    assert layout["base.actor.0.weight"][1] == (H, d.obs) and layout["base.actor.2.weight"][1] == (H, H)


def test_c_abi_layout_follows_param_layout():
    import ctypes
    from pgmorl_b200._lib import lib
    L = lib()
    for d in ENV_SHAPES.values():
        for H in (32, 64, 128):
            dh = NetDims(d.obs, d.act, d.obj, H)
            layout, n = param_layout(dh)
            assert L.pgm_n_par_h(d.obs, d.act, d.obj, H) == n
            out = (ctypes.c_int * 13)()
            assert L.pgm_param_offsets_h(d.obs, d.act, d.obj, H, out) == 0
            assert list(out) == [off for off, _ in layout.values()]
        old = (ctypes.c_int * 13)()
        new = (ctypes.c_int * 13)()
        assert L.pgm_param_offsets(d.obs, d.act, d.obj, old) == 0
        assert L.pgm_param_offsets_h(d.obs, d.act, d.obj, 64, new) == 0
        assert list(old) == list(new) and L.pgm_n_par(d.obs, d.act, d.obj) == L.pgm_n_par_h(d.obs, d.act, d.obj, 64)
    assert L.pgm_n_par_h(17, 6, 2, 48) == -1 and b"{32, 64, 128}" in L.pgm_last_error()
    out = (ctypes.c_int * 13)()
    assert L.pgm_param_offsets_h(17, 6, 2, 256, out) == 1 and b"{32, 64, 128}" in L.pgm_last_error()
    assert L.pgm_ppo_workspace_bytes_h(2, 64, 17, 6, 2, 0, 48) == 0


@pytest.mark.parametrize("H", [16, 48, 256])
def test_policy_refuses_unsupported_width(H):
    from pgmorl_b200.a2c_ppo_acktr.model import Policy
    from synth_envs import _Box
    with pytest.raises(NotImplementedError, match=r"\{32, 64, 128\}"):
        Policy((17,), _Box(6), base_kwargs={"layernorm": False, "hidden_size": H}, obj_num=2, device="cpu")


@pytest.mark.parametrize("H", [32, 64, 128])
def test_policy_state_dict_shapes_follow_width(H):
    from pgmorl_b200.a2c_ppo_acktr.model import Policy
    from synth_envs import _Box
    kw = {"layernorm": False} if H == 64 else {"layernorm": False, "hidden_size": H}
    pol = Policy((17,), _Box(6), base_kwargs=kw, obj_num=2, device="cpu")
    assert pol.dims == NetDims(17, 6, 2, H)
    sd = pol.state_dict()
    assert sd["base.actor.0.weight"].shape == (H, 17) and sd["base.critic.2.weight"].shape == (H, H)
    assert sd["dist.fc_mean.weight"].shape == (6, H) and sd["base.critic_linear.weight"].shape == (2, H)
    pol2 = Policy((17,), _Box(6), base_kwargs=kw, obj_num=2, device="cpu")
    pol2.load_state_dict(sd)
    assert torch.equal(pol2.flat, pol.flat)
