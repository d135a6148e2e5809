"""Float64 restatement of one MOPG iteration at any hidden width, on the numpy oracle's building blocks.

oracle/mopg_oracle.mopg_iteration / ppo_update build their `Net` at the default width 64. Everything they call
(rollout, gae_returns, advantages, ppo_grad, clip_and_adam) works on a `Net` of any width, so this helper repeats their
loop with `Net(flat, O, A, M, H)`; nothing else differs. Pinned against the torch port (nn.Linear + autograd) in
tests/test_oracle_hidden.py."""
import numpy as np

from oracle import mopg_oracle as orc


def ppo_update(flat, m, v, step, lr, dims, obs, action, logp, value, returns, adv, perm, num_mini_batch, **kw):
    """orc.ppo_update with a network of width dims.hidden; in place on flat / m / v. Returns (step, mean losses)."""
    O, A, M, H = dims.obs, dims.act, dims.obj, dims.hidden
    clip, vcoef, ecoef = kw.get("clip", 0.2), kw.get("vcoef", 0.5), kw.get("ecoef", 0.0)
    net = orc.Net(flat, O, A, M, H)
    T, N = action.shape[0], action.shape[1]
    X, ACT, LP = obs[:-1].reshape(T * N, O), action.reshape(T * N, A), logp.reshape(T * N)
    VO, RET, ADV = value[:-1].reshape(T * N, M), returns.reshape(T * N, M), adv.reshape(T * N)
    mb = (T * N) // num_mini_batch
    sums = np.zeros(3)
    for e in range(perm.shape[0]):
        for b in range(num_mini_batch):
            idx = perm[e, b * mb:(b + 1) * mb]
            g, losses = orc.ppo_grad(net, X[idx], ACT[idx], LP[idx], VO[idx], RET[idx], ADV[idx], clip, vcoef, ecoef)
            step = orc.clip_and_adam(flat, g, m, v, step, lr, kw.get("max_grad_norm", 0.5))
            sums += losses
    return step, tuple(sums / (perm.shape[0] * num_mini_batch))


def mopg_iteration(flat, m, v, step, lr, dims, traj, eps, perm, weights, obj_var, gamma=0.995, lam=0.95,
                   num_mini_batch=32, **kw):
    """orc.mopg_iteration with a network of width dims.hidden. In place on flat / m / v."""
    net = orc.Net(flat, dims.obs, dims.act, dims.obj, dims.hidden)
    obs = traj["obs"].astype(np.float64)
    value, action, logp = orc.rollout(net, obs, eps)
    ret = orc.gae_returns(traj["rewards"].astype(np.float64), value, traj["masks"].astype(np.float64),
                          traj["bad_masks"].astype(np.float64), gamma, lam)
    adv = orc.advantages(ret, value, weights, obj_var)
    step, losses = ppo_update(flat, m, v, step, lr, dims, obs, action, logp, value, ret, adv, perm, num_mini_batch, **kw)
    return {"value": value, "action": action, "logp": logp, "returns": ret, "adv": adv, "losses": np.array(losses),
            "step": step}
