"""The two float64 restatements of the non-default PPO options (tests/ppo_options_ref.py) against each other: the n-step
and plain-GAE return branches of compute_returns and the unclipped value loss, on masks / bad masks with zeros (also in
the bootstrap slot T). The numpy side is literal loops and a hand-derived gradient, the torch side the reference's tensor
code and autograd. Also the argument checks of the K2 entry points, which run before any CUDA call."""
import numpy as np
import pytest
import torch

import ppo_options_ref as ref
from oracle import mopg_oracle as orc
from oracle.mopg_torch_port import PortPolicy
from pgmorl_b200 import synthetic
from pgmorl_b200.layout import NetDims
from tests.helpers import rel_err


def _rollout_arrays(T, N, M, seed):
    rng = np.random.RandomState(seed)
    rewards = rng.randn(T, N, M)
    value = rng.randn(T + 1, N, M) * 2
    masks = (rng.uniform(size=(T + 1, N)) > 0.15).astype(np.float64)
    bad = (rng.uniform(size=(T + 1, N)) > 0.15).astype(np.float64)
    masks[T, 0] = 0.0; bad[T, 1] = 0.0                 # zeros in the bootstrap slot too
    return rewards, value, masks, bad, rng.randn(N, M)


@pytest.mark.parametrize("use_gae,use_ptl", ref.BRANCHES)
def test_return_branches_numpy_equals_torch(use_gae, use_ptl):
    T, N, M = 37, 3, 3
    rewards, value, masks, bad, nv = _rollout_arrays(T, N, M, seed=4)
    assert masks.min() == 0 and bad.min() == 0
    got = ref.returns_np(rewards, value, masks, bad, 0.99, 0.9, use_gae, use_ptl, next_value=None if use_gae else nv)
    t = lambda a: torch.as_tensor(a)
    vp = t(value.copy())
    want = ref.returns_torch(t(rewards), vp, t(masks)[..., None], t(bad)[..., None], t(value[-1] if use_gae else nv),
                             0.99, 0.9, use_gae, use_ptl)
    assert rel_err(got, want[:-1].numpy()) < 1e-12
    if not use_gae:          # the n-step branches leave value_preds alone and put the bootstrap in returns[-1]
        assert np.array_equal(vp.numpy(), value) and np.array_equal(want[-1].numpy(), nv)
    if use_gae and use_ptl:  # branch A is the oracle's gae_returns (pinned against the reference's goldens)
        assert rel_err(got, orc.gae_returns(rewards, value, masks, bad, 0.99, 0.9)) < 1e-12


def test_without_time_limit_cuts_the_branches_coincide():
    """bad_masks == 1: GAE with and without proper time limits are the same numbers, and so are the two n-step branches"""
    T, N, M = 29, 2, 2
    rewards, value, masks, _, nv = _rollout_arrays(T, N, M, seed=8)
    ones = np.ones_like(masks)
    r = {b: ref.returns_np(rewards, value, masks, ones, 0.995, 0.95, *b, next_value=nv if not b[0] else None)
         for b in ref.BRANCHES}
    assert np.array_equal(r[(True, True)], r[(True, False)])
    assert np.array_equal(r[(False, True)], r[(False, False)])
    assert not np.allclose(r[(True, True)], r[(False, True)])


@pytest.mark.parametrize("dims", [NetDims(17, 6, 2), NetDims(11, 3, 3)])
def test_unclipped_value_loss_gradient_equals_autograd(dims):
    d = dims
    rng = np.random.RandomState(2)
    flat = synthetic.init_policy_flat(d, seed=5).numpy().astype(np.float64)
    flat[-d.act:] = rng.uniform(-0.5, 0.3, d.act)
    mb = 64
    x, action = rng.randn(mb, d.obs), rng.randn(mb, d.act)
    logp_old, adv = rng.randn(mb) * 0.3 - 6.0, rng.randn(mb)
    value, _, _ = orc.forward(orc.Net(flat.copy(), d.obs, d.act, d.obj), x)
    v_old = value + rng.randn(mb, d.obj) * 0.4
    ret = value + rng.randn(mb, d.obj)
    assert (np.abs(value - v_old) > 0.2).mean() > 0.2       # the clip is active: the two losses differ
    pol = PortPolicy(flat, d.obs, d.act, d.obj)
    for clipped in (True, False):
        g, losses = ref.ppo_grad_np(orc.Net(flat.copy(), d.obs, d.act, d.obj), x, action, logp_old, v_old, ret, adv,
                                    ecoef=0.01, clipped_value_loss=clipped)
        gt, lt = ref.ppo_grad_torch(pol, x, action, logp_old, v_old, ret, adv, ecoef=0.01, clipped_value_loss=clipped)
        assert rel_err(g, gt) < 1e-12 and rel_err(np.array(losses), np.array(lt)) < 1e-12
        if clipped:
            g_clipped = g
    assert rel_err(g, g_clipped) > 1e-3


@pytest.mark.parametrize("use_gae,use_ptl,clipped", [(False, True, True), (True, False, True), (False, False, True),
                                                     (True, True, False), (False, False, False)])
def test_iteration_numpy_equals_torch_port(use_gae, use_ptl, clipped):
    """one whole MOPG iteration (rollout, returns, advantage, E x B Adam steps) of the two restatements"""
    d = NetDims(17, 6, 2)
    T, N, E, B, j = 24, 4, 2, 3, 3
    flat0 = synthetic.init_policy_flat(d, seed=11).numpy().astype(np.float64)
    traj = {k: v[0].numpy() for k, v in synthetic.make_trajectories(1, T, N, d, seed=6, p_done=0.1).items()}
    traj["bad_masks"][T, 0] = 0.0
    weights, obj_var = np.array([0.3, 0.7]), np.array([1.4, 0.6])
    eps, perm = synthetic.host_rng_streams(j, T, N, d.act, E)
    flat, m, v = flat0.copy(), np.zeros_like(flat0), np.zeros_like(flat0)
    out = ref.mopg_iteration_np(flat, m, v, 0, 3e-4, (d.obs, d.act, d.obj), traj, eps.numpy(), perm.numpy(), weights,
                                obj_var, num_mini_batch=B, use_gae=use_gae, use_proper_time_limits=use_ptl,
                                clipped_value_loss=clipped)
    pol = PortPolicy(flat0, d.obs, d.act, d.obj)
    opt = torch.optim.Adam(pol.ordered(), lr=3e-4, eps=1e-5)
    port = ref.mopg_iteration_torch(pol, opt, traj, j, 3e-4, weights, obj_var, ppo_epoch=E, num_mini_batch=B,
                                    use_gae=use_gae, use_proper_time_limits=use_ptl, clipped_value_loss=clipped)
    assert rel_err(out["returns"], port["returns"]) < 1e-12
    assert rel_err(out["adv"], port["adv"]) < 1e-12
    # E x B dependent Adam steps: the same gate as the oracle-vs-reference tests (tests/test_oracle_mopg.py)
    assert rel_err(out["losses"], port["losses"]) < 1e-9
    assert rel_err(flat, pol.flat()) < 1e-9


def test_returns_entry_point_checks_its_arguments_without_a_gpu():
    """pgm_returns_adv_f32 refuses unknown mode bits and null buffers before any CUDA call; pgm_gae_adv_f32 keeps its own
    messages"""
    import ctypes
    from pgmorl_b200._lib import lib
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    rc = lib().pgm_returns_adv_f32(p, p, None, p, p, None, None, 0.99, 0.95, 4, p, None, 1, 2, 2, 2, None)
    assert rc == 1 and b"pgm_returns_adv_f32: unknown mode bits 0x4" in lib().pgm_last_error()
    rc = lib().pgm_returns_adv_f32(None, p, None, p, p, None, None, 0.99, 0.95, 0, p, None, 1, 2, 2, 2, None)
    assert rc == 1 and b"pgm_returns_adv_f32: null pointer" in lib().pgm_last_error()
    rc = lib().pgm_gae_adv_f32(p, p, p, p, None, None, 0.99, 0.95, p, None, 1, 2, 33, 2, None)
    assert rc == 1 and b"pgm_gae_adv_f32: need 1 <= N <= 32" in lib().pgm_last_error()
