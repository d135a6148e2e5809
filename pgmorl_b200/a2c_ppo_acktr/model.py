"""Policy with the reference's interface (a2c_ppo_acktr/model.py:15-82) whose parameters live in ONE flat
float32 CUDA vector (order: pgmorl_b200/layout.py) and whose forward passes are K1 launches.

Supported: 1-D observations, MOMLPBase H-H tanh without LayerNorm (H = base_kwargs['hidden_size'], default 64; 32, 64
and 128 run on the device), and the head the action space selects as in the reference: Box -> DiagGaussian with
state-independent logstd (the configuration PG-MORL instantiates, warm_up.py:34-40), Discrete(n) -> Categorical
(1 <= n <= 32). CNN / GRU bases and MultiBinary (Bernoulli) heads are not provided."""
from collections import OrderedDict

import numpy as np
import torch

from .. import kernels as K
from ..layout import CATEGORICAL_MAX, DIST_CATEGORICAL, DIST_GAUSSIAN, NetDims, param_layout
from ..synthetic import init_policy_flat

HIDDEN_SIZES = (32, 64, 128)     # hidden widths the K1 / K3 kernels are built for (include/pgmorl_b200.h)


class Policy:
    def __init__(self, obs_shape, action_space, base=None, base_kwargs=None, obj_num=1, device="cuda", flat=None):
        kind = action_space.__class__.__name__
        if len(obs_shape) != 1 or kind not in ("Box", "Discrete"):
            raise NotImplementedError("Policy: only 1-D observations with Box or Discrete actions")
        if base_kwargs and base_kwargs.get("layernorm", False):
            raise NotImplementedError("Policy: layernorm=True is not part of the PG-MORL configuration (warm_up.py:37)")
        hidden = int((base_kwargs or {}).get("hidden_size", 64))
        if hidden not in HIDDEN_SIZES:
            raise NotImplementedError(f"Policy: hidden_size={hidden} is not supported; the kernels are built for "
                                      f"hidden_size in {{32, 64, 128}}")
        if kind == "Discrete":
            n = int(action_space.n)
            if not 1 <= n <= CATEGORICAL_MAX:
                raise NotImplementedError(f"Policy: Discrete({n}) is not supported; the kernels are built for categorical "
                                          f"heads of 1 to {CATEGORICAL_MAX} actions")
            self.dims = NetDims(int(obs_shape[0]), n, int(obj_num), hidden, DIST_CATEGORICAL)
        else:
            self.dims = NetDims(int(obs_shape[0]), int(action_space.shape[0]), int(obj_num), hidden, DIST_GAUSSIAN)
        self.device = torch.device(device)
        if flat is None:
            flat = init_policy_flat(self.dims)          # draws from torch's global CPU generator like the reference
        self.flat = torch.as_tensor(np.asarray(flat), dtype=torch.float32).to(self.device).contiguous()

    # ---- nn.Module-like surface the reference touches
    is_recurrent = False
    recurrent_hidden_state_size = 1

    def to(self, device):
        self.device = torch.device(device)
        self.flat = self.flat.to(self.device)
        return self

    def double(self):
        return self      # arithmetic is FP32 on the device; state_dict() hands out float64 like the reference

    def parameters(self):
        return [self.flat]

    def state_dict(self):
        layout, _ = param_layout(self.dims)
        host = self.flat.detach().cpu().to(torch.float64)
        return OrderedDict((name, host[off:off + int(np.prod(shape))].reshape(shape).clone())
                           for name, (off, shape) in layout.items())

    def load_state_dict(self, sd):
        layout, n = param_layout(self.dims)
        flat = torch.empty(n, dtype=torch.float64)
        for name, (off, shape) in layout.items():
            flat[off:off + int(np.prod(shape))] = torch.as_tensor(sd[name], dtype=torch.float64).reshape(-1)
        self.flat = flat.to(torch.float32).to(self.device).contiguous()

    def __deepcopy__(self, memo):
        new = Policy.__new__(Policy)
        new.dims, new.device, new.flat = self.dims, self.device, self.flat.clone()
        return new

    # ---- forward passes (K1)
    def _obs(self, inputs):
        return torch.as_tensor(inputs).to(self.device, torch.float32).reshape(1, -1, self.dims.obs).contiguous()

    def act(self, inputs, rnn_hxs, masks, deterministic=False):
        """-> value [N,M], action [N,A], action_log_probs [N,1], rnn_hxs (model.py:57-69). Sampling noise comes from
        torch's global CPU generator, one normal_(0,1) draw of shape [N,A] in float64, exactly the stream
        dist.sample() consumes in the reference. Categorical head: one exponential_(1) draw of shape [N,n] in float64
        (torch.multinomial's single-sample path), and the action is int64 [N,1]."""
        obs = self._obs(inputs)
        n = obs.shape[1]
        if deterministic:
            value, action, logp = K.policy_forward(self.flat[None], obs, self.dims, mode=K.ACT_DETERMINISTIC)
        else:
            eps = torch.empty(n, self.dims.act, dtype=torch.float64)
            eps.exponential_(1) if self.dims.categorical else eps.normal_(0, 1)
            value, action, logp = K.policy_forward(self.flat[None], obs, self.dims,
                                                   eps=eps.to(self.device, torch.float32)[None].contiguous())
        action = action[0].to(torch.int64) if self.dims.categorical else action[0]
        return value[0], action, logp[0].unsqueeze(-1), rnn_hxs

    def get_value(self, inputs, rnn_hxs, masks):
        value, _, _ = K.policy_forward(self.flat[None], self._obs(inputs), self.dims, rows_a=0, mode=K.ACT_DETERMINISTIC)
        return value[0]

    def evaluate_actions(self, inputs, rnn_hxs, masks, action):
        """-> value, action_log_probs [N,1], dist_entropy (scalar), rnn_hxs (model.py:75-82)."""
        obs = self._obs(inputs)
        act = torch.as_tensor(action).to(self.device, torch.float32).reshape(1, -1, self.dims.act_cols).contiguous()
        if self.dims.categorical:        # per-row entropy from K1, mean over the rows (FixedCategorical.entropy().mean())
            ent_rows = torch.empty(1, act.shape[1], device=self.device, dtype=torch.float32)
            value, _, logp = K.policy_forward(self.flat[None], obs, self.dims, action=act, mode=K.ACT_EVALUATE,
                                              entropy=ent_rows)
            return value[0], logp[0].unsqueeze(-1), ent_rows.mean(), rnn_hxs
        value, _, logp = K.policy_forward(self.flat[None], obs, self.dims, action=act, mode=K.ACT_EVALUATE)
        logstd = self.flat[-self.dims.act:]
        entropy = (0.5 + 0.5 * float(np.log(2 * np.pi)) + logstd).sum()
        return value[0], logp[0].unsqueeze(-1), entropy, rnn_hxs
