"""ORACLE (test infrastructure, NOT product code) -- float64 numpy restatement of the
reference's per-task MOPG iteration: rollout inference, vector GAE, scalarised +
normalised advantage, and the PPO minibatch loop with hand-derived backward,
grad-norm clipping and Adam.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this package. The product path (pgmorl_b200/) never does.

Parity pin: tests/golden/mopg_*.npz hold outputs of the UNMODIFIED reference
(imported in-process from /root/reference by tests/golden/make_golden.py) on the
same seeded inputs; tests/test_oracle_mopg.py checks this file against them.

Reference anchors (paths relative to /root/reference):
  forward        externals/pytorch-a2c-ppo-acktr-gail/a2c_ppo_acktr/model.py:57-82,237-246
  DiagGaussian   .../a2c_ppo_acktr/distributions.py:30-40,71-90 ; utils.py:32-43 (AddBias)
  GAE            .../a2c_ppo_acktr/storage.py:83-94
  advantage      .../a2c_ppo_acktr/algo/ppo.py:40-56 ; morl/scalarization_methods.py:28-29
  sampler        .../a2c_ppo_acktr/storage.py:118-154
  PPO loss       .../a2c_ppo_acktr/algo/ppo.py:62-107
  clip / Adam    torch/nn/utils/clip_grad.py ; torch/optim/adam.py (_single_tensor_adam)
  LR schedule    .../a2c_ppo_acktr/utils.py:46-50 ; morl/mopg.py:96-101
"""
import math

import numpy as np

HALF_LOG_2PI = math.log(math.sqrt(2 * math.pi))


class Net:
    """Views into one flat float64 parameter vector (order: pgmorl_b200/layout.py)."""

    def __init__(self, flat, O, A, M, H=64):
        self.O, self.A, self.M, self.H = O, A, M, H
        self.flat = flat
        off = 0

        def take(*shape):
            nonlocal off
            n = int(np.prod(shape))
            v = flat[off:off + n].reshape(shape)
            off += n
            return v

        self.W1a, self.b1a = take(H, O), take(H)
        self.W2a, self.b2a = take(H, H), take(H)
        self.W1c, self.b1c = take(H, O), take(H)
        self.W2c, self.b2c = take(H, H), take(H)
        self.Wv, self.bv = take(M, H), take(M)
        self.Wmu, self.bmu = take(A, H), take(A)
        self.logstd = take(A)
        assert off == flat.size, (off, flat.size)


def n_par(O, A, M, H=64):
    return 2 * (H * O + H + H * H + H) + M * H + M + A * H + A + A


def forward(net, x):
    """model.py:237-246 (MLPBase.forward) + distributions.py:81-90 (mean only)."""
    c1 = np.tanh(x @ net.W1c.T + net.b1c)
    c2 = np.tanh(c1 @ net.W2c.T + net.b2c)
    value = c2 @ net.Wv.T + net.bv
    h1 = np.tanh(x @ net.W1a.T + net.b1a)
    h2 = np.tanh(h1 @ net.W2a.T + net.b2a)
    mean = h2 @ net.Wmu.T + net.bmu
    return value, mean, (c1, c2, h1, h2)


def log_prob(net, mean, action):
    """distributions.py:33-36: Normal.log_prob summed over the action dim (keepdim dropped)."""
    std = np.exp(net.logstd)
    var = std ** 2
    log_scale = np.log(std)
    return (-((action - mean) ** 2) / (2 * var) - log_scale - HALF_LOG_2PI).sum(-1)


def entropy(net):
    """distributions.py:38-39: sum_a (0.5 + 0.5*log(2pi) + log(std_a)); batch-mean of a constant."""
    return float((0.5 + HALF_LOG_2PI + np.log(np.exp(net.logstd))).sum())


def act(net, obs, eps):
    """model.py:57-69 with deterministic=False: action = mean + std*eps
    (torch.normal(mean, std) == normal_(0,1)*std + mean, bit-exact on the CPU generator)."""
    value, mean, _ = forward(net, obs)
    action = eps * np.exp(net.logstd) + mean
    return value, action, log_prob(net, mean, action)


def rollout(net, obs, eps):
    """mopg.py:103-135 with the env replaced by given observations.
    obs [T+1,N,O], eps [T,N,A] -> value [T+1,N,M], action [T,N,A], logp [T,N]."""
    T = eps.shape[0]
    value, mean, _ = forward(net, obs.reshape(-1, obs.shape[-1]))
    value = value.reshape(obs.shape[0], obs.shape[1], -1)
    mean = mean.reshape(obs.shape[0], obs.shape[1], -1)[:T]
    action = eps * np.exp(net.logstd) + mean
    return value, action, log_prob(net, mean, action)


def gae_returns(rewards, value, masks, bad_masks, gamma, lam):
    """storage.py:83-94 (use_gae and use_proper_time_limits).
    rewards [T,N,M], value [T+1,N,M], masks/bad_masks [T+1,N] -> returns [T,N,M]."""
    T = rewards.shape[0]
    ret = np.zeros_like(rewards)
    gae = np.zeros_like(rewards[0])
    for t in reversed(range(T)):
        m = masks[t + 1][:, None]
        delta = rewards[t] + gamma * value[t + 1] * m - value[t]
        gae = delta + gamma * lam * m * gae
        gae = gae * bad_masks[t + 1][:, None]
        ret[t] = gae + value[t]
    return ret


def advantages(returns, value, weights, obj_var):
    """algo/ppo.py:43-56: un-normalise by sqrt(obj_var+1e-8), weighted sum, then
    (adv - mean) / (unbiased std + 1e-5) over all T*N samples."""
    scale = np.sqrt(obj_var + 1e-8) if obj_var is not None else 1.0
    adv = ((returns * scale) * weights).sum(-1) - ((value[:-1] * scale) * weights).sum(-1)
    return (adv - adv.mean()) / (adv.std(ddof=1) + 1e-5)


def ppo_grad(net, x, action, logp_old, v_old, ret, adv, clip=0.2, vcoef=0.5, ecoef=0.0):
    """Loss of algo/ppo.py:76-100 and its gradient (what autograd produces), flat float64.
    Tie semantics of torch.min / torch.max (gradient split 1/2-1/2 on exact ties) and
    torch.clamp (gradient passes on the closed interval) are restated exactly."""
    mb = x.shape[0]
    M = net.M
    value, mean, (c1, c2, h1, h2) = forward(net, x)
    std = np.exp(net.logstd)
    var = std ** 2
    logp = log_prob(net, mean, action)
    ratio = np.exp(logp - logp_old)
    surr1 = ratio * adv
    rc = np.clip(ratio, 1.0 - clip, 1.0 + clip)
    surr2 = rc * adv
    action_loss = -np.minimum(surr1, surr2).mean()

    d = value - v_old
    v_clip = v_old + np.clip(d, -clip, clip)
    la = (value - ret) ** 2
    lb = (v_clip - ret) ** 2
    value_loss = 0.5 * np.maximum(la, lb).mean()
    ent = entropy(net)

    # d loss / d logp
    in_rng = ((ratio >= 1.0 - clip) & (ratio <= 1.0 + clip)).astype(np.float64)
    w1 = np.where(surr1 < surr2, 1.0, np.where(surr1 == surr2, 0.5, 0.0))
    w2 = 1.0 - w1
    dmin_dr = w1 * adv + w2 * adv * in_rng
    dlogp = -(1.0 / mb) * dmin_dr * ratio
    # d loss / d value
    pas = ((d >= -clip) & (d <= clip)).astype(np.float64)
    wa = np.where(la > lb, 1.0, np.where(la == lb, 0.5, 0.0))
    wb = 1.0 - wa
    dV = vcoef * 0.5 / (mb * M) * (wa * 2 * (value - ret) + wb * 2 * (v_clip - ret) * pas)

    g = np.zeros_like(net.flat)
    G = Net(g, net.O, net.A, net.M, net.H)
    # actor
    diff = action - mean
    dmean = dlogp[:, None] * diff / var
    G.logstd[:] = (dlogp[:, None] * (diff ** 2 / var - 1.0)).sum(0) - ecoef
    G.Wmu[:] = dmean.T @ h2
    G.bmu[:] = dmean.sum(0)
    dz2 = (dmean @ net.Wmu) * (1 - h2 ** 2)
    G.W2a[:] = dz2.T @ h1
    G.b2a[:] = dz2.sum(0)
    dz1 = (dz2 @ net.W2a) * (1 - h1 ** 2)
    G.W1a[:] = dz1.T @ x
    G.b1a[:] = dz1.sum(0)
    # critic
    G.Wv[:] = dV.T @ c2
    G.bv[:] = dV.sum(0)
    dy2 = (dV @ net.Wv) * (1 - c2 ** 2)
    G.W2c[:] = dy2.T @ c1
    G.b2c[:] = dy2.sum(0)
    dy1 = (dy2 @ net.W2c) * (1 - c1 ** 2)
    G.W1c[:] = dy1.T @ x
    G.b1c[:] = dy1.sum(0)
    return g, (value_loss, action_loss, ent)


def clip_and_adam(p, g, m, v, step, lr, max_grad_norm=0.5, beta1=0.9, beta2=0.999, eps=1e-5, norms=None):
    """clip_grad_norm_ (coef = min(1, max/(norm+1e-6)), always multiplied) then one Adam
    step in torch's _single_tensor_adam arithmetic. In place on p, m, v; returns step+1.
    `norms`, if a list, receives the gradient norm before clipping."""
    total = math.sqrt(float((g * g).sum()))
    if norms is not None:
        norms.append(total)
    coef = min(1.0, max_grad_norm / (total + 1e-6))
    g = g * coef
    step += 1
    m += (g - m) * (1 - beta1)
    v *= beta2
    v += (1 - beta2) * g * g
    bc1 = 1 - beta1 ** step
    bc2 = 1 - beta2 ** step
    denom = np.sqrt(v) / math.sqrt(bc2) + eps
    p -= (lr / bc1) * (m / denom)
    return step


def ppo_update(flat, m, v, step, lr, dims, obs, action, logp, value, returns, adv, perm,
               num_mini_batch, clip=0.2, vcoef=0.5, ecoef=0.0, max_grad_norm=0.5,
               adam_eps=1e-5, beta1=0.9, beta2=0.999, norms=None):
    """algo/ppo.py:62-115. obs [T+1,N,O] etc.; perm int [E, T*N]. In place on flat/m/v.
    Returns (step, (value_loss, action_loss, entropy) averaged over E*B updates).
    `norms`, if a list, receives each step's gradient norm before clipping."""
    O, A, M = dims
    net = Net(flat, O, A, M)
    T, N = action.shape[0], action.shape[1]
    X = obs[:-1].reshape(T * N, O)
    ACT = action.reshape(T * N, A)
    LP = logp.reshape(T * N)
    VO = value[:-1].reshape(T * N, M)
    RET = returns.reshape(T * N, M)
    ADV = adv.reshape(T * N)
    mb = (T * N) // num_mini_batch
    sums = np.zeros(3)
    for e in range(perm.shape[0]):
        for b in range(num_mini_batch):          # drop_last=True
            idx = perm[e, b * mb:(b + 1) * mb]
            g, losses = ppo_grad(net, X[idx], ACT[idx], LP[idx], VO[idx], RET[idx], ADV[idx],
                                 clip, vcoef, ecoef)
            step = clip_and_adam(flat, g, m, v, step, lr, max_grad_norm, beta1, beta2, adam_eps, norms)
            sums += losses
    return step, tuple(sums / (perm.shape[0] * num_mini_batch))


def mopg_iteration(flat, m, v, step, lr, dims, traj, eps, perm, weights, obj_var,
                   gamma=0.995, lam=0.95, num_mini_batch=32, **ppo_kw):
    """One pass of mopg.py:96-144 for one task on given observations / rewards / masks.
    In place on flat/m/v. Returns dict of every intermediate the parity tests compare."""
    O, A, M = dims
    net = Net(flat, O, A, M)
    obs = traj["obs"].astype(np.float64)
    value, action, logp = rollout(net, obs, eps)
    ret = gae_returns(traj["rewards"].astype(np.float64), value,
                      traj["masks"].astype(np.float64), traj["bad_masks"].astype(np.float64),
                      gamma, lam)
    adv = advantages(ret, value, weights, obj_var)
    step, losses = ppo_update(flat, m, v, step, lr, dims, obs, action, logp, value, ret, adv,
                              perm, num_mini_batch, **ppo_kw)
    return {"value": value, "action": action, "logp": logp, "returns": ret, "adv": adv,
            "losses": np.array(losses), "step": step}
