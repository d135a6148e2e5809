"""Test infrastructure (not product code): float64 restatements of the PPO options beyond PG-MORL's defaults, i.e. the
return branches of RolloutStorage.compute_returns other than GAE with proper time limits (a2c/storage.py:77-116) and the
unclipped value loss of PPO.update (a2c/algo/ppo.py:86-94, use_clipped_value_loss=False).

Two independent restatements, as for the default options in oracle/:
  - numpy: literal loops of the reference's branches and a hand-derived gradient of the unclipped loss, on top of
    oracle/mopg_oracle.py (forward, advantage, clip + Adam are shared);
  - torch: the same branches on the reference's tensor shapes, and the loss differentiated by autograd, on top of
    oracle/mopg_torch_port.py's policy.
No golden of the unmodified reference exists for these options (the goldens were made with PG-MORL's run.py settings),
so the two restatements are checked against each other (tests/test_oracle_ppo_options.py) and the kernels against them."""
import numpy as np
import torch
import torch.nn as nn

from oracle import mopg_oracle as orc

BRANCHES = [(True, True), (False, True), (True, False), (False, False)]      # (use_gae, use_proper_time_limits): A, B, C, D


# ---------------------------------------------------------------------------------------------------------------------
# numpy
# ---------------------------------------------------------------------------------------------------------------------
def returns_np(rewards, value, masks, bad_masks, gamma, lam, use_gae, use_proper_time_limits, next_value=None):
    """storage.py:77-116. rewards [T,N,M], value [T+1,N,M] (row T = next_value in the GAE branches), masks / bad_masks
    [T+1,N]; next_value [N,M] = returns[-1] of the n-step branches (default value[T]). -> returns [T,N,M]"""
    T = rewards.shape[0]
    value = value.copy()
    returns = np.zeros((T + 1,) + rewards.shape[1:])
    mk, bd = masks[:, :, None], bad_masks[:, :, None]
    nv = value[-1] if next_value is None else next_value
    if use_proper_time_limits:
        if use_gae:
            value[-1] = nv
            gae = 0
            for s in reversed(range(T)):
                delta = rewards[s] + gamma * value[s + 1] * mk[s + 1] - value[s]
                gae = delta + gamma * lam * mk[s + 1] * gae
                gae = gae * bd[s + 1]
                returns[s] = gae + value[s]
        else:
            returns[-1] = nv
            for s in reversed(range(T)):
                returns[s] = (returns[s + 1] * gamma * mk[s + 1] + rewards[s]) * bd[s + 1] + (1 - bd[s + 1]) * value[s]
    else:
        if use_gae:
            value[-1] = nv
            gae = 0
            for s in reversed(range(T)):
                delta = rewards[s] + gamma * value[s + 1] * mk[s + 1] - value[s]
                gae = delta + gamma * lam * mk[s + 1] * gae
                returns[s] = gae + value[s]
        else:
            returns[-1] = nv
            for s in reversed(range(T)):
                returns[s] = returns[s + 1] * gamma * mk[s + 1] + rewards[s]
    return returns[:-1]


def ppo_grad_np(net, x, action, logp_old, v_old, ret, adv, clip=0.2, vcoef=0.5, ecoef=0.0, clipped_value_loss=True):
    """orc.ppo_grad, plus the unclipped value loss 0.5 * mean((V - R)^2) (mean over mb x M) and its gradient
    d loss / d V = vcoef * (V - R) / (mb * M) backpropagated through the critic."""
    if clipped_value_loss:
        return orc.ppo_grad(net, x, action, logp_old, v_old, ret, adv, clip, vcoef, ecoef)
    g, (_, action_loss, ent) = orc.ppo_grad(net, x, action, logp_old, v_old, ret, adv, clip, 0.0, ecoef)   # actor part
    mb, M = x.shape[0], net.M
    value, _, (c1, c2, _, _) = orc.forward(net, x)
    value_loss = 0.5 * ((value - ret) ** 2).mean()
    dV = vcoef * (value - ret) / (mb * M)
    G = orc.Net(g, net.O, net.A, net.M, net.H)
    G.Wv[:] = dV.T @ c2
    G.bv[:] = dV.sum(0)
    dy2 = (dV @ net.Wv) * (1 - c2 ** 2)
    G.W2c[:] = dy2.T @ c1
    G.b2c[:] = dy2.sum(0)
    dy1 = (dy2 @ net.W2c) * (1 - c1 ** 2)
    G.W1c[:] = dy1.T @ x
    G.b1c[:] = dy1.sum(0)
    return g, (value_loss, action_loss, ent)


def ppo_update_np(flat, m, v, step, lr, dims, obs, action, logp, value, returns, adv, perm, num_mini_batch,
                  clipped_value_loss=True, clip=0.2, vcoef=0.5, ecoef=0.0, max_grad_norm=0.5, adam_eps=1e-5):
    """orc.ppo_update with the choice of value loss. In place on flat / m / v; returns (step, mean losses)."""
    O, A, M = dims
    net = orc.Net(flat, O, A, M)
    T, N = action.shape[0], action.shape[1]
    X, ACT, LP = obs[:-1].reshape(T * N, O), action.reshape(T * N, A), logp.reshape(T * N)
    VO, RET, ADV = value[:-1].reshape(T * N, M), returns.reshape(T * N, M), adv.reshape(T * N)
    mb = (T * N) // num_mini_batch
    sums = np.zeros(3)
    for e in range(perm.shape[0]):
        for b in range(num_mini_batch):
            idx = perm[e, b * mb:(b + 1) * mb]
            g, losses = ppo_grad_np(net, X[idx], ACT[idx], LP[idx], VO[idx], RET[idx], ADV[idx], clip, vcoef, ecoef,
                                    clipped_value_loss)
            step = orc.clip_and_adam(flat, g, m, v, step, lr, max_grad_norm, eps=adam_eps)
            sums += losses
    return step, tuple(sums / (perm.shape[0] * num_mini_batch))


def mopg_iteration_np(flat, m, v, step, lr, dims, traj, eps, perm, weights, obj_var, gamma=0.995, lam=0.95,
                      num_mini_batch=32, use_gae=True, use_proper_time_limits=True, clipped_value_loss=True):
    """orc.mopg_iteration with the return branch and the value loss chosen; the bootstrap of the n-step branches is the
    value of the last observation (next_value, mopg.py:132-135)."""
    O, A, M = dims
    net = orc.Net(flat, O, A, M)
    obs = traj["obs"].astype(np.float64)
    value, action, logp = orc.rollout(net, obs, eps)
    ret = returns_np(traj["rewards"].astype(np.float64), value, traj["masks"].astype(np.float64),
                     traj["bad_masks"].astype(np.float64), gamma, lam, use_gae, use_proper_time_limits)
    adv = orc.advantages(ret, value, weights, obj_var)           # (returns - value[:-1]) scaled, scalarised, normalised
    step, losses = ppo_update_np(flat, m, v, step, lr, dims, obs, action, logp, value, ret, adv, perm, num_mini_batch,
                                 clipped_value_loss)
    return {"value": value, "returns": ret, "adv": adv, "losses": np.array(losses), "step": step}


# ---------------------------------------------------------------------------------------------------------------------
# torch (autograd)
# ---------------------------------------------------------------------------------------------------------------------
def returns_torch(rewards, value_preds, masks, bad_masks, next_value, gamma, lam, use_gae, use_proper_time_limits):
    """storage.py:77-116 on the reference's shapes: rewards [T,N,M], value_preds [T+1,N,M], masks [T+1,N,1]. Returns the
    [T+1,N,M] returns buffer; value_preds is written (row T) by the GAE branches only, as in the reference."""
    T = rewards.shape[0]
    returns = torch.zeros_like(value_preds)
    if use_proper_time_limits:
        if use_gae:
            value_preds[-1] = next_value
            gae = 0
            for step in reversed(range(T)):
                delta = rewards[step] + gamma * value_preds[step + 1] * masks[step + 1] - value_preds[step]
                gae = delta + gamma * lam * masks[step + 1] * gae
                gae = gae * bad_masks[step + 1]
                returns[step] = gae + value_preds[step]
        else:
            returns[-1] = next_value
            for step in reversed(range(T)):
                returns[step] = (returns[step + 1] * gamma * masks[step + 1] + rewards[step]) * bad_masks[step + 1] \
                    + (1 - bad_masks[step + 1]) * value_preds[step]
    else:
        if use_gae:
            value_preds[-1] = next_value
            gae = 0
            for step in reversed(range(T)):
                delta = rewards[step] + gamma * value_preds[step + 1] * masks[step + 1] - value_preds[step]
                gae = delta + gamma * lam * masks[step + 1] * gae
                returns[step] = gae + value_preds[step]
        else:
            returns[-1] = next_value
            for step in reversed(range(T)):
                returns[step] = returns[step + 1] * gamma * masks[step + 1] + rewards[step]
    return returns


def ppo_losses_torch(policy, x, action, logp_old, v_old, ret, adv, clip=0.2, clipped_value_loss=True):
    """(value_loss, action_loss, entropy) of ppo.py:76-100 as autograd graphs."""
    values, logp, ent = policy.evaluate_actions(x, action)
    ratio = torch.exp(logp - logp_old)
    surr1 = ratio * adv
    surr2 = torch.clamp(ratio, 1.0 - clip, 1.0 + clip) * adv
    action_loss = -torch.min(surr1, surr2).mean()
    if clipped_value_loss:
        vclip = v_old + (values - v_old).clamp(-clip, clip)
        value_loss = 0.5 * torch.max((values - ret).pow(2), (vclip - ret).pow(2)).mean()
    else:
        value_loss = 0.5 * (ret - values).pow(2).mean()
    return value_loss, action_loss, ent


def ppo_grad_torch(policy, x, action, logp_old, v_old, ret, adv, clip=0.2, vcoef=0.5, ecoef=0.0, clipped_value_loss=True):
    """Flat gradient (reference parameter order) of value_loss * vcoef + action_loss - ecoef * entropy, by autograd."""
    f = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float64)
    vl, al, ent = ppo_losses_torch(policy, f(x), f(action), f(logp_old).view(-1, 1), f(v_old), f(ret), f(adv).view(-1, 1),
                                   clip, clipped_value_loss)
    for p in policy.ordered():
        p.grad = None
    (vl * vcoef + al - ent * ecoef).backward()
    g = torch.cat([p.grad.reshape(-1) for p in policy.ordered()]).numpy().copy()
    return g, (vl.item(), al.item(), ent.item())


def mopg_iteration_torch(policy, optimizer, traj, j, lr, weights, obj_var, gamma=0.995, lam=0.95, ppo_epoch=10,
                         num_mini_batch=32, clip=0.2, vcoef=0.5, ecoef=0.0, max_grad_norm=0.5, use_gae=True,
                         use_proper_time_limits=True, clipped_value_loss=True):
    """oracle/mopg_torch_port.mopg_iteration_port with the return branch and the value loss chosen."""
    obs_all = torch.as_tensor(traj["obs"])
    T, N = obs_all.shape[0] - 1, obs_all.shape[1]
    M = traj["rewards"].shape[-1]
    A = policy.fm.out_features
    f64 = torch.float64
    obs = torch.zeros(T + 1, N, obs_all.shape[2], dtype=f64)
    rewards = torch.zeros(T, N, M, dtype=f64)
    value_preds = torch.zeros(T + 1, N, M, dtype=f64)
    logps = torch.zeros(T, N, 1, dtype=f64)
    actions = torch.zeros(T, N, A, dtype=f64)
    masks = torch.ones(T + 1, N, 1, dtype=f64)
    bad_masks = torch.ones(T + 1, N, 1, dtype=f64)
    obs[0].copy_(obs_all[0])
    torch.manual_seed(j)
    for g in optimizer.param_groups:
        g["lr"] = lr
    tm, tb, tr = torch.as_tensor(traj["masks"]), torch.as_tensor(traj["bad_masks"]), torch.as_tensor(traj["rewards"])
    for step in range(T):
        with torch.no_grad():
            value, action, logp = policy.act(obs[step])
        obs[step + 1].copy_(obs_all[step + 1])
        actions[step].copy_(action); logps[step].copy_(logp); value_preds[step].copy_(value)
        rewards[step].copy_(tr[step])
        masks[step + 1].copy_(tm[step + 1].unsqueeze(-1)); bad_masks[step + 1].copy_(tb[step + 1].unsqueeze(-1))
    with torch.no_grad():
        next_value = policy.base(obs[-1])[0]
    returns = returns_torch(rewards, value_preds, masks, bad_masks, next_value, gamma, lam, use_gae, use_proper_time_limits)
    w = torch.as_tensor(weights, dtype=f64)
    sc = torch.as_tensor(np.sqrt(obj_var + 1e-8), dtype=f64)
    adv = ((returns * sc)[:-1] * w).sum(-1) - ((value_preds * sc)[:-1] * w).sum(-1)
    adv = (adv - adv.mean()) / (adv.std() + 1e-5)
    S = T * N
    mb = S // num_mini_batch
    sums = np.zeros(3)
    X = obs[:-1].view(S, -1); ACT = actions.view(S, -1); VO = value_preds[:-1].view(S, -1)
    RET = returns[:-1].view(S, -1); LP = logps.view(S, 1); ADV = adv.view(S, 1)
    params = list(policy.parameters())
    for _ in range(ppo_epoch):
        perm = torch.randperm(S)
        for b in range(num_mini_batch):
            idx = perm[b * mb:(b + 1) * mb]
            value_loss, action_loss, ent = ppo_losses_torch(policy, X[idx], ACT[idx], LP[idx], VO[idx], RET[idx], ADV[idx],
                                                            clip, clipped_value_loss)
            optimizer.zero_grad()
            (value_loss * vcoef + action_loss - ent * ecoef).backward()
            nn.utils.clip_grad_norm_(params, max_grad_norm)
            optimizer.step()
            sums += (value_loss.item(), action_loss.item(), ent.item())
    return {"returns": returns[:-1].numpy(), "adv": adv.numpy(), "losses": sums / (ppo_epoch * num_mini_batch)}
