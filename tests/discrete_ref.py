"""Float64 restatements of one MOPG iteration for a Categorical head (Discrete(n) actions), in two independent forms.

* numpy, hand-derived backward (`CatNet`, `forward`, `ppo_grad`, `mopg_iteration`), on the numpy oracle's GAE, advantage,
  clip and Adam (oracle/mopg_oracle.py);
* torch, `torch.distributions.Categorical` + autograd + torch.optim.Adam with the reference's per-step `act` loop
  (`PortCatPolicy`, `mopg_iteration_port`), drawing the action noise from torch's global CPU generator as
  `dist.sample()` does.

No golden of the unmodified reference exists for Categorical heads; tests/test_oracle_discrete.py pins the two forms to
each other, and the sampling identity `Categorical.sample() == argmax(probs / exponential_)` to torch itself.

Head semantics (FixedCategorical of a2c/distributions.py): logits z = W h2 + b; log-prob z_a - logsumexp(z); entropy
-sum_j p_j log p_j per row, averaged over the minibatch by evaluate_actions; sample = first argmax of p_j / q_j with
q ~ Exponential(1) (torch.multinomial's single-sample path in torch 2.11); mode = first argmax of the probabilities.
"""
import numpy as np
import torch
import torch.nn as nn

from oracle import mopg_oracle as orc


class CatNet:
    """Views into one flat float64 vector of the 12-tensor Categorical layout (pgmorl_b200/layout.py)."""

    def __init__(self, flat, O, n, M, H=64):
        self.O, self.A, self.M, self.H = O, n, M, H
        self.flat = flat
        off = 0

        def take(*shape):
            nonlocal off
            k = int(np.prod(shape))
            v = flat[off:off + k].reshape(shape)
            off += k
            return v

        self.W1a, self.b1a = take(H, O), take(H)
        self.W2a, self.b2a = take(H, H), take(H)
        self.W1c, self.b1c = take(H, O), take(H)
        self.W2c, self.b2c = take(H, H), take(H)
        self.Wv, self.bv = take(M, H), take(M)
        self.Wz, self.bz = take(n, H), take(n)
        assert off == flat.size, (off, flat.size)


def net_of(flat, dims):
    return CatNet(flat, dims.obs, dims.act, dims.obj, dims.hidden)


def forward(net, x):
    """-> value [R,M], logits [R,n], caches."""
    c1 = np.tanh(x @ net.W1c.T + net.b1c)
    c2 = np.tanh(c1 @ net.W2c.T + net.b2c)
    value = c2 @ net.Wv.T + net.bv
    h1 = np.tanh(x @ net.W1a.T + net.b1a)
    h2 = np.tanh(h1 @ net.W2a.T + net.b2a)
    z = h2 @ net.Wz.T + net.bz
    return value, z, (c1, c2, h1, h2)


def log_softmax(z):
    mx = z.max(-1, keepdims=True)
    return z - (mx + np.log(np.exp(z - mx).sum(-1, keepdims=True)))


def entropy_rows(z):
    lp = log_softmax(z)
    return -(np.exp(lp) * lp).sum(-1)


def sample(z, q):
    """First argmax of p_j / q_j, and the float64 top-two margin (r1 - r2) / r1 of each row."""
    r = np.exp(log_softmax(z)) / q
    srt = np.sort(r, -1)
    return r.argmax(-1), (srt[..., -1] - srt[..., -2]) / srt[..., -1]


def mode(z):
    """First argmax of the logits, and the top-two probability margin (p1 - p2) / p1 of each row."""
    p = np.exp(log_softmax(z))
    srt = np.sort(p, -1)
    return z.argmax(-1), (srt[..., -1] - srt[..., -2]) / srt[..., -1]


def rollout(net, obs, q):
    """obs [T+1,N,O], q [T,N,n] Exponential(1) draws -> value [T+1,N,M], action int [T,N], logp [T,N], margin [T,N]."""
    T = q.shape[0]
    value, z, _ = forward(net, obs.reshape(-1, obs.shape[-1]))
    value = value.reshape(obs.shape[0], obs.shape[1], -1)
    z = z.reshape(obs.shape[0], obs.shape[1], -1)[:T]
    action, margin = sample(z, q)
    logp = np.take_along_axis(log_softmax(z), action[..., None], -1)[..., 0]
    return value, action, logp, margin


def ppo_grad(net, x, action, logp_old, v_old, ret, adv, clip=0.2, vcoef=0.5, ecoef=0.0, clipped_value_loss=True):
    """Loss of algo/ppo.py:76-100 for a Categorical head and its gradient, flat float64 (hand-derived backward).
    action: int [mb]. Returns (grad, (value_loss, action_loss, mean entropy))."""
    mb, M = x.shape[0], net.M
    value, z, (c1, c2, h1, h2) = forward(net, x)
    lsm = log_softmax(z)
    p = np.exp(lsm)
    H = -(p * lsm).sum(-1)
    logp = lsm[np.arange(mb), action]
    ratio = np.exp(logp - logp_old)
    surr1 = ratio * adv
    surr2 = np.clip(ratio, 1.0 - clip, 1.0 + clip) * adv
    action_loss = -np.minimum(surr1, surr2).mean()
    d = value - v_old
    v_clip = v_old + np.clip(d, -clip, clip)
    la = (value - ret) ** 2
    lb = (v_clip - ret) ** 2 if clipped_value_loss else np.full_like(la, -1.0)
    value_loss = 0.5 * np.maximum(la, lb).mean()

    in_rng = ((ratio >= 1.0 - clip) & (ratio <= 1.0 + clip)).astype(np.float64)
    w1 = np.where(surr1 < surr2, 1.0, np.where(surr1 == surr2, 0.5, 0.0))
    dlogp = -(1.0 / mb) * (w1 * adv + (1.0 - w1) * adv * in_rng) * ratio
    onehot = np.zeros_like(z)
    onehot[np.arange(mb), action] = 1.0
    # d logp_i / dz_ij = [j = a_i] - p_ij ; d(-c * mean_i H_i) / dz_ij = c / mb * p_ij (log p_ij + H_i)
    dz = dlogp[:, None] * (onehot - p) + (ecoef / mb) * p * (lsm + H[:, None])
    pas = ((d >= -clip) & (d <= clip)).astype(np.float64)
    wa = np.where(la > lb, 1.0, np.where(la == lb, 0.5, 0.0))
    dV = vcoef * 0.5 / (mb * M) * (wa * 2 * (value - ret) + (1.0 - wa) * 2 * (v_clip - ret) * pas)

    g = np.zeros_like(net.flat)
    G = CatNet(g, net.O, net.A, net.M, net.H)
    G.Wz[:] = dz.T @ h2
    G.bz[:] = dz.sum(0)
    dz2 = (dz @ net.Wz) * (1 - h2 ** 2)
    G.W2a[:] = dz2.T @ h1
    G.b2a[:] = dz2.sum(0)
    dz1 = (dz2 @ net.W2a) * (1 - h1 ** 2)
    G.W1a[:] = dz1.T @ x
    G.b1a[:] = dz1.sum(0)
    G.Wv[:] = dV.T @ c2
    G.bv[:] = dV.sum(0)
    dy2 = (dV @ net.Wv) * (1 - c2 ** 2)
    G.W2c[:] = dy2.T @ c1
    G.b2c[:] = dy2.sum(0)
    dy1 = (dy2 @ net.W2c) * (1 - c1 ** 2)
    G.W1c[:] = dy1.T @ x
    G.b1c[:] = dy1.sum(0)
    return g, (value_loss, action_loss, float(H.mean()))


def ppo_update(flat, m, v, step, lr, dims, obs, action, logp, value, returns, adv, perm, num_mini_batch, clip=0.2,
               vcoef=0.5, ecoef=0.0, max_grad_norm=0.5, clipped_value_loss=True):
    """algo/ppo.py:62-115 for a Categorical head; in place on flat / m / v. action int [T,N].
    Returns (step, mean (value_loss, action_loss, entropy))."""
    net = net_of(flat, dims)
    T, N = action.shape
    O, M = dims.obs, dims.obj
    X, ACT, LP = obs[:-1].reshape(T * N, O), action.reshape(T * N), logp.reshape(T * N)
    VO, RET, ADV = value[:-1].reshape(T * N, M), returns.reshape(T * N, M), adv.reshape(T * N)
    mb = (T * N) // num_mini_batch
    sums = np.zeros(3)
    for e in range(perm.shape[0]):
        for b in range(num_mini_batch):
            idx = perm[e, b * mb:(b + 1) * mb]
            g, losses = ppo_grad(net, X[idx], ACT[idx], LP[idx], VO[idx], RET[idx], ADV[idx], clip, vcoef, ecoef,
                                 clipped_value_loss)
            step = orc.clip_and_adam(flat, g, m, v, step, lr, max_grad_norm)
            sums += losses
    return step, tuple(sums / (perm.shape[0] * num_mini_batch))


def mopg_iteration(flat, m, v, step, lr, dims, traj, q, perm, weights, obj_var, gamma=0.995, lam=0.95,
                   num_mini_batch=32, **kw):
    """mopg.py:96-144 for one task with a Categorical head on given observations / rewards / masks; q [T,N,n] the
    Exponential(1) draws of the rollout. In place on flat / m / v."""
    net = net_of(flat, dims)
    obs = traj["obs"].astype(np.float64)
    value, action, logp, margin = rollout(net, obs, q)
    ret = orc.gae_returns(traj["rewards"].astype(np.float64), value, traj["masks"].astype(np.float64),
                          traj["bad_masks"].astype(np.float64), gamma, lam)
    adv = orc.advantages(ret, value, weights, obj_var)
    step, losses = ppo_update(flat, m, v, step, lr, dims, obs, action, logp, value, ret, adv, perm, num_mini_batch, **kw)
    return {"value": value, "action": action, "logp": logp, "margin": margin, "returns": ret, "adv": adv,
            "losses": np.array(losses), "step": step}


# ------------------------------------------------------------------------------------------------------------------
# torch port: the reference's modules and loop
# ------------------------------------------------------------------------------------------------------------------
class PortCatPolicy(nn.Module):
    """The reference Policy with MOMLPBase and the Categorical head: base first, then dist.linear."""

    def __init__(self, flat, O, n, M, H=64):
        super().__init__()
        f64 = torch.float64
        self.a0, self.a2 = nn.Linear(O, H, dtype=f64), nn.Linear(H, H, dtype=f64)
        self.c0, self.c2 = nn.Linear(O, H, dtype=f64), nn.Linear(H, H, dtype=f64)
        self.cl = nn.Linear(H, M, dtype=f64)
        self.linear = nn.Linear(H, n, dtype=f64)
        if flat is not None:
            self.load_flat(flat)

    def ordered(self):
        return [self.a0.weight, self.a0.bias, self.a2.weight, self.a2.bias, self.c0.weight, self.c0.bias,
                self.c2.weight, self.c2.bias, self.cl.weight, self.cl.bias, self.linear.weight, self.linear.bias]

    def load_flat(self, flat):
        flat = torch.as_tensor(np.asarray(flat), dtype=torch.float64)
        off = 0
        with torch.no_grad():
            for p in self.ordered():
                p.copy_(flat[off:off + p.numel()].view_as(p))
                off += p.numel()

    def flat(self):
        return torch.cat([p.detach().reshape(-1) for p in self.ordered()]).numpy().copy()

    def base(self, x):
        hc = torch.tanh(self.c2(torch.tanh(self.c0(x))))
        ha = torch.tanh(self.a2(torch.tanh(self.a0(x))))
        return self.cl(hc), ha

    def dist(self, ha):
        return torch.distributions.Categorical(logits=self.linear(ha))

    def act(self, x, deterministic=False):
        value, ha = self.base(x)
        d = self.dist(ha)
        action = d.probs.argmax(-1, keepdim=True) if deterministic else d.sample().unsqueeze(-1)
        return value, action, d.log_prob(action.squeeze(-1)).view(action.size(0), -1).sum(-1).unsqueeze(-1)

    def evaluate_actions(self, x, action):
        value, ha = self.base(x)
        d = self.dist(ha)
        logp = d.log_prob(action.squeeze(-1)).view(action.size(0), -1).sum(-1).unsqueeze(-1)
        return value, logp, d.entropy().mean()


def port_grad(policy, x, action, logp_old, v_old, ret, adv, clip=0.2, vcoef=0.5, ecoef=0.0, clipped_value_loss=True):
    """Autograd gradient (flat float64) and losses of one minibatch; action int64 [mb]."""
    t = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float64)
    values, logp, ent = policy.evaluate_actions(t(x), torch.as_tensor(np.asarray(action), dtype=torch.int64)[:, None])
    ratio = torch.exp(logp - t(logp_old)[:, None])
    A = t(adv)[:, None]
    action_loss = -torch.min(ratio * A, torch.clamp(ratio, 1.0 - clip, 1.0 + clip) * A).mean()
    VO, R = t(v_old), t(ret)
    if clipped_value_loss:
        vclip = VO + (values - VO).clamp(-clip, clip)
        value_loss = 0.5 * torch.max((values - R).pow(2), (vclip - R).pow(2)).mean()
    else:
        value_loss = 0.5 * (R - values).pow(2).mean()
    policy.zero_grad()
    (value_loss * vcoef + action_loss - ent * ecoef).backward()
    g = torch.cat([p.grad.reshape(-1) for p in policy.ordered()]).numpy().copy()
    return g, (value_loss.item(), action_loss.item(), ent.item())


def mopg_iteration_port(policy, optimizer, traj, j, lr, weights, obj_var, gamma=0.995, lam=0.95, ppo_epoch=10,
                        num_mini_batch=32, clip=0.2, vcoef=0.5, ecoef=0.0, max_grad_norm=0.5):
    """The loop body of morl/mopg.py:96-144 with a Categorical policy (env replaced by `traj`): torch.manual_seed(j),
    T per-step act calls drawing from the global generator, GAE, advantage, E x B autograd minibatch steps."""
    obs_all = torch.as_tensor(traj["obs"])
    T, N = obs_all.shape[0] - 1, obs_all.shape[1]
    M = traj["rewards"].shape[-1]
    f64 = torch.float64
    obs = torch.zeros(T + 1, N, obs_all.shape[2], dtype=f64)
    value_preds = torch.zeros(T + 1, N, M, dtype=f64)
    returns = torch.zeros(T + 1, N, M, dtype=f64)
    logps = torch.zeros(T, N, 1, dtype=f64)
    actions = torch.zeros(T, N, 1, dtype=torch.int64)
    obs[0].copy_(obs_all[0])
    torch.manual_seed(j)
    for g in optimizer.param_groups:
        g["lr"] = lr
    masks = torch.ones(T + 1, N, 1, dtype=f64)
    bad_masks = torch.ones(T + 1, N, 1, dtype=f64)
    masks[1:, :, 0] = torch.as_tensor(traj["masks"][1:], dtype=f64)
    bad_masks[1:, :, 0] = torch.as_tensor(traj["bad_masks"][1:], dtype=f64)
    rewards = torch.as_tensor(traj["rewards"], dtype=f64)
    for step in range(T):
        with torch.no_grad():
            value, action, logp = policy.act(obs[step])
        obs[step + 1].copy_(obs_all[step + 1])
        actions[step].copy_(action); logps[step].copy_(logp); value_preds[step].copy_(value)
    with torch.no_grad():
        value_preds[-1] = policy.base(obs[-1])[0]
    gae = 0
    for step in reversed(range(T)):
        delta = rewards[step] + gamma * value_preds[step + 1] * masks[step + 1] - value_preds[step]
        gae = delta + gamma * lam * masks[step + 1] * gae
        gae = gae * bad_masks[step + 1]
        returns[step] = gae + value_preds[step]
    w = torch.as_tensor(weights, dtype=f64)
    sc = torch.as_tensor(np.sqrt(obj_var + 1e-8), dtype=f64)
    adv = ((returns * sc)[:-1] * w).sum(-1) - ((value_preds * sc)[:-1] * w).sum(-1)
    adv = (adv - adv.mean()) / (adv.std() + 1e-5)
    S = T * N
    mb = S // num_mini_batch
    sums = np.zeros(3)
    X, ACT, VO = obs[:-1].view(S, -1), actions.view(S, 1), value_preds[:-1].view(S, -1)
    RET, LP, ADV = returns[:-1].view(S, -1), logps.view(S, 1), adv.view(S, 1)
    params = policy.ordered()
    for _ in range(ppo_epoch):
        perm = torch.randperm(S)
        for b in range(num_mini_batch):
            idx = perm[b * mb:(b + 1) * mb]
            values, logp, ent = policy.evaluate_actions(X[idx], ACT[idx])
            ratio = torch.exp(logp - LP[idx])
            surr1 = ratio * ADV[idx]
            surr2 = torch.clamp(ratio, 1.0 - clip, 1.0 + clip) * ADV[idx]
            action_loss = -torch.min(surr1, surr2).mean()
            vclip = VO[idx] + (values - VO[idx]).clamp(-clip, clip)
            value_loss = 0.5 * torch.max((values - RET[idx]).pow(2), (vclip - RET[idx]).pow(2)).mean()
            optimizer.zero_grad()
            (value_loss * vcoef + action_loss - ent * ecoef).backward()
            nn.utils.clip_grad_norm_(params, max_grad_norm)
            optimizer.step()
            sums += (value_loss.item(), action_loss.item(), ent.item())
    return {"value": value_preds.numpy(), "action": actions[..., 0].numpy(), "logp": logps[..., 0].numpy(),
            "returns": returns[:-1].numpy(), "adv": adv.numpy(), "losses": sums / (ppo_epoch * num_mini_batch)}
