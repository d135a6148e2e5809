"""PPO agent with the reference's interface (a2c_ppo_acktr/algo/ppo.py:7-115); `update` = one K2 launch for the
scalarised, normalised advantage and one K3 launch for the E x B minibatch steps (loss, backward, clip, Adam).
The optimiser object keeps torch.optim.Adam's state_dict layout so Samples interchange with the reference."""
from copy import deepcopy

import numpy as np
import torch

from ... import kernels as K
from ..._lib import PpoHyper
from ...layout import param_layout


class DeviceAdam:
    """Adam moments as flat float32 CUDA vectors + the scalar step; state_dict()/load_state_dict() speak
    torch.optim.Adam's format (13 parameter tensors in named_parameters() order, 12 for a Categorical head)."""

    def __init__(self, actor_critic, lr, eps):
        self.dims, self.device = actor_critic.dims, actor_critic.flat.device
        self.exp_avg = torch.zeros_like(actor_critic.flat)
        self.exp_avg_sq = torch.zeros_like(actor_critic.flat)
        self.step_count = 0
        self.param_groups = [{"lr": lr, "betas": (0.9, 0.999), "eps": eps, "weight_decay": 0, "amsgrad": False,
                              "params": list(range(len(param_layout(self.dims)[0])))}]

    def state_dict(self):
        layout, _ = param_layout(self.dims)
        m, v = self.exp_avg.cpu().to(torch.float64), self.exp_avg_sq.cpu().to(torch.float64)
        state = {}
        if self.step_count > 0:
            for i, (name, (off, shape)) in enumerate(layout.items()):
                n = int(np.prod(shape))
                state[i] = {"step": torch.tensor(float(self.step_count)), "exp_avg": m[off:off + n].reshape(shape).clone(),
                            "exp_avg_sq": v[off:off + n].reshape(shape).clone()}
        return {"state": state, "param_groups": deepcopy(self.param_groups)}

    def load_state_dict(self, sd):
        layout, n = param_layout(self.dims)
        m, v = torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.float64)
        self.step_count = 0
        for i, (name, (off, shape)) in enumerate(layout.items()):
            if i in sd["state"]:
                st = sd["state"][i]
                k = int(np.prod(shape))
                m[off:off + k] = torch.as_tensor(st["exp_avg"], dtype=torch.float64).reshape(-1)
                v[off:off + k] = torch.as_tensor(st["exp_avg_sq"], dtype=torch.float64).reshape(-1)
                self.step_count = int(float(st["step"]))
        self.exp_avg, self.exp_avg_sq = m.to(torch.float32).to(self.device), v.to(torch.float32).to(self.device)
        for g, src in zip(self.param_groups, sd["param_groups"]):
            g.update({k: src[k] for k in ("lr", "betas", "eps") if k in src})

    def __deepcopy__(self, memo):
        new = DeviceAdam.__new__(DeviceAdam)
        new.dims, new.device, new.step_count = self.dims, self.device, self.step_count
        new.exp_avg, new.exp_avg_sq = self.exp_avg.clone(), self.exp_avg_sq.clone()
        new.param_groups = deepcopy(self.param_groups)
        return new


class PPO():
    def __init__(self, actor_critic, clip_param, ppo_epoch, num_mini_batch, value_loss_coef, entropy_coef, lr=None,
                 eps=None, max_grad_norm=None, use_clipped_value_loss=True, obj_weights=None, scalarization_func=None,
                 cluster=0):
        self.actor_critic = actor_critic
        self.clip_param, self.ppo_epoch, self.num_mini_batch = clip_param, ppo_epoch, num_mini_batch
        self.value_loss_coef, self.entropy_coef, self.max_grad_norm = value_loss_coef, entropy_coef, max_grad_norm
        self.use_clipped_value_loss = use_clipped_value_loss
        self.optimizer = self.make_optimizer(actor_critic, lr=lr, eps=eps)
        self.obj_weights = None if obj_weights is None else torch.Tensor(obj_weights)
        self.scalarization_func = scalarization_func
        self.cluster = cluster

    @staticmethod
    def make_optimizer(actor_critic, lr, eps):
        return DeviceAdam(actor_critic, lr, eps)

    def update(self, rollouts, scalarization=None, obj_var=None):
        """-> (value_loss, action_loss, dist_entropy) averaged over ppo_epoch * num_mini_batch updates.
        Minibatch permutations are drawn with torch.randperm on the global CPU generator, one per epoch, the
        stream SubsetRandomSampler consumes in the reference (storage.py:133-137)."""
        pol, opt = self.actor_critic, self.optimizer
        d, dev = pol.dims, pol.flat.device
        T, N, M = rollouts.rewards.shape
        S = T * N
        scal = scalarization if scalarization is not None else self.scalarization_func
        if scal is None:
            raise NotImplementedError("PPO.update: a scalarization is required (multi-objective path)")
        w = torch.as_tensor(np.asarray(scal.weights, dtype=np.float64), dtype=torch.float32, device=dev)[None]
        ov = None if obj_var is None else torch.as_tensor(np.asarray(obj_var, dtype=np.float64) * np.ones(M),
                                                          dtype=torch.float32, device=dev)[None]
        # advantage from the returns already in storage (ppo.py:43-56): K2 recomputes returns (same branch and bootstrap
        # as compute_returns) and normalises
        ret, adv = K.returns_adv(rollouts.rewards[None], rollouts.value_preds[None], rollouts.masks.view(1, T + 1, N),
                                 rollouts.bad_masks.view(1, T + 1, N), self._gamma(rollouts), self._lam(rollouts),
                                 weights=w, obj_var=ov, **rollouts.return_branch())
        perm = torch.stack([torch.randperm(S) for _ in range(self.ppo_epoch)]).to(torch.int32).to(dev)[None].contiguous()
        step = torch.tensor([opt.step_count], dtype=torch.int32, device=dev)
        lr = torch.tensor([opt.param_groups[0]["lr"]], dtype=torch.float64, device=dev)
        hyper = PpoHyper(self.clip_param, self.value_loss_coef, self.entropy_coef, self.max_grad_norm,
                         opt.param_groups[0]["betas"][0], opt.param_groups[0]["betas"][1], opt.param_groups[0]["eps"])
        params, m, v = pol.flat[None], opt.exp_avg[None], opt.exp_avg_sq[None]
        losses = K.ppo_update(params, m, v, step, lr, rollouts.obs.view(1, (T + 1) * N, d.obs),
                              rollouts.actions.view(1, S, d.act_cols).to(torch.float32), rollouts.action_log_probs.view(1, S),
                              rollouts.value_preds.view(1, (T + 1) * N, M), ret.view(1, S, M), adv.view(1, S), perm,
                              self.num_mini_batch, d, hyper=hyper, cluster=self.cluster,
                              clipped_value_loss=self.use_clipped_value_loss)
        opt.step_count = int(step.item())
        vl, al, ent = losses[0].tolist()
        return vl, al, ent

    # GAE hyper-parameters travel with the storage when the worker sets them (see mopg.py); default = run.py:56-70
    @staticmethod
    def _gamma(rollouts):
        return getattr(rollouts, "gamma", 0.995)

    @staticmethod
    def _lam(rollouts):
        return getattr(rollouts, "gae_lambda", 0.95)
