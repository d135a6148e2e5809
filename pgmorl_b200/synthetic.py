"""Policy initialisation, the host RNG contract, and seeded synthetic trajectories of the named environment shapes.

MuJoCo stepping is out of scope (BASELINE.json north_star), so parity tests and
bench.py feed the path synthetic trajectories. Everything here is generated on
the host with torch's CPU generator so that the oracle and the CUDA path see
identical bytes (SURVEY.md section 8(d), configs C1-C5). Replay / toy environments
and synthetic selection histories are test infrastructure: tests/synth_envs.py.
"""
import numpy as np
import torch

from .layout import NetDims, param_layout


def init_policy_flat(dims: NetDims, seed=None):
    """Random-init parameters, drawing from torch's global CPU generator in the same
    order as the reference's ``Policy(obs_shape, Box(A), base_kwargs={'layernorm':
    False}, obj_num=M).double()`` (warm_up.py:34-40): each ``nn.Linear`` first runs its
    default init, then ``orthogonal_`` with the reference's gain
    (model.py:208-216,252-254; distributions.py:75-78). Returns float64 [n_par].
    A Categorical head (``Policy(obs_shape, Discrete(n))``) is built after the base in the same way: ``dist.linear =
    nn.Linear(H, n)``, orthogonal with gain 0.01, bias 0 (the Categorical module of distributions.py), and has no logstd.
    """
    if seed is not None:
        torch.manual_seed(seed)
    O, A, M, H = dims.obs, dims.act, dims.obj, dims.hidden
    f64 = torch.float64
    g2 = float(np.sqrt(2))

    def lin(i, o, gain):
        m = torch.nn.Linear(i, o, dtype=f64)
        torch.nn.init.orthogonal_(m.weight.data, gain=gain)
        torch.nn.init.constant_(m.bias.data, 0)
        return m

    a0 = lin(O, H, g2); a2 = lin(H, H, g2)
    c0 = lin(O, H, g2); c2 = lin(H, H, g2)
    lin(H, 1, g2)                      # MLPBase.critic_linear, replaced by MOMLPBase
    cl = lin(H, M, g2)
    fm = lin(H, A, 0.01 if dims.categorical else 1.0)
    tensors = [a0.weight, a0.bias, a2.weight, a2.bias, c0.weight, c0.bias, c2.weight, c2.bias,
               cl.weight, cl.bias, fm.weight, fm.bias] + ([] if dims.categorical else [torch.zeros(A, 1, dtype=f64)])
    flat = torch.cat([t.detach().reshape(-1) for t in tensors])
    assert flat.numel() == param_layout(dims)[1]
    return flat


def simplex_weights(obj_num, delta):
    """Evenly spaced scalarisation weights (utils.py:67-78 generate_weights_batch_dfs with
    min 0 / max 1), same float accumulation ``w += delta``."""
    out = []

    def dfs(i, weight):
        if i == obj_num - 1:
            out.append(weight + [1.0 - float(np.sum(weight[0:i]))])
            return
        w = 0.0
        while w < 1.0 + 0.5 * delta and np.sum(weight[0:i]) + w < 1.0 + 0.5 * delta:
            dfs(i + 1, weight[0:i] + [w])
            w += delta

    dfs(0, [])
    return np.array(out, dtype=np.float64)


def make_trajectories(P, T, N, dims: NetDims, seed=1, p_done=0.002):
    """Synthetic rollout inputs for P tasks (SURVEY.md section 8(d) C2).

    obs      f32 [P,T+1,N,O]  clip(N(0,1), +-10)  (reference obs pass through float32 once)
    rewards  f32 [P,T,N,M]    U[0,1)              (normalised objective vectors)
    masks    f32 [P,T+1,N]    0 where an episode ended at the previous step
    bad_masks f32 [P,T+1,N]   0 on half of those ends (time-limit truncations)
    """
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(P, T + 1, N, dims.obs, generator=g, dtype=torch.float32).clamp_(-10, 10)
    rewards = torch.rand(P, T, N, dims.obj, generator=g, dtype=torch.float32)
    done = torch.rand(P, T + 1, N, generator=g, dtype=torch.float32) < p_done
    trunc = done & (torch.rand(P, T + 1, N, generator=g, dtype=torch.float32) < 0.5)
    masks = (~done).to(torch.float32)
    bad_masks = (~trunc).to(torch.float32)
    masks[:, 0] = 1.0
    bad_masks[:, 0] = 1.0
    return {"obs": obs, "rewards": rewards, "masks": masks, "bad_masks": bad_masks}


def host_rng_streams(j, T, N, A, epochs, eps_dtype=torch.float64, categorical=False):
    """The reference's per-iteration random streams (mopg.py:96 ``torch.manual_seed(j)``):
    T draws of action noise ``[N,A]`` in rollout order (distributions.py:30-40 via
    ``dist.sample()`` == ``mean + std*normal_(0,1)``), then one ``randperm(T*N)`` per PPO
    epoch (storage.py:133-137 ``BatchSampler(SubsetRandomSampler(range(T*N)))``).
    categorical=True (A = n categories): the noise of each step is ``exponential_(1)`` of shape ``[N,n]``, what
    ``Categorical.sample()`` draws in torch 2.11 (``torch.multinomial(probs, 1, True)`` takes ``argmax(probs / q)``
    with ``q = empty_like(probs).exponential_(1)`` for a single sample).
    Returns eps f64 [T,N,A], perm int64 [epochs, T*N].
    """
    torch.manual_seed(j)
    eps = torch.empty(T, N, A, dtype=eps_dtype)
    for t in range(T):
        if categorical:
            eps[t].exponential_(1)
        else:
            eps[t].normal_(0, 1)
    perm = torch.stack([torch.randperm(T * N) for _ in range(epochs)])
    return eps, perm


def linear_lr(lr0, j, lr_decay_ratio, total_num_updates):
    """a2c_ppo_acktr/utils.py:46-50 called as mopg.py:97-101."""
    return lr0 - (lr0 * ((j * lr_decay_ratio) / float(total_num_updates)))
