"""RolloutStorage with the reference's buffers and methods (a2c_ppo_acktr/storage.py:9-154), resident in HBM as
float32. compute_returns (all four branches of storage.py:77-116) is a K2 launch."""
import torch

from .. import kernels as K


class RolloutStorage(object):
    def __init__(self, num_steps, num_processes, obs_shape, action_space, recurrent_hidden_state_size, obj_num=1,
                 device="cuda"):
        kind = action_space.__class__.__name__
        if kind not in ("Box", "Discrete"):
            raise NotImplementedError("RolloutStorage: Box or Discrete action spaces only")
        dv, T, N = torch.device(device), num_steps, num_processes
        z = lambda *s: torch.zeros(*s, device=dv, dtype=torch.float32)
        self.obs = z(T + 1, N, *obs_shape)
        self.recurrent_hidden_states = z(T + 1, N, recurrent_hidden_state_size)
        self.rewards = z(T, N, obj_num)
        self.value_preds = z(T + 1, N, obj_num)
        self.returns = z(T + 1, N, obj_num)
        self.action_log_probs = z(T, N, 1)
        # Discrete: one int64 column per step, as the reference stores the sampled category (RolloutStorage.__init__)
        self.actions = (torch.zeros(T, N, 1, device=dv, dtype=torch.int64) if kind == "Discrete"
                        else z(T, N, action_space.shape[0]))
        self.masks = torch.ones(T + 1, N, 1, device=dv)
        self.bad_masks = torch.ones(T + 1, N, 1, device=dv)
        self.num_steps = num_steps
        self.step = 0

    def to(self, device):
        for k, v in list(self.__dict__.items()):
            if isinstance(v, torch.Tensor):
                setattr(self, k, v.to(device))

    def insert(self, obs, recurrent_hidden_states, actions, action_log_probs, value_preds, rewards, masks, bad_masks):
        dv = self.obs.device
        f = lambda t: torch.as_tensor(t).to(dv, torch.float32)
        self.obs[self.step + 1].copy_(f(obs))
        self.actions[self.step].copy_(torch.as_tensor(actions).to(dv, self.actions.dtype))
        self.action_log_probs[self.step].copy_(f(action_log_probs))
        self.value_preds[self.step].copy_(f(value_preds))
        self.rewards[self.step].copy_(f(rewards))
        self.masks[self.step + 1].copy_(f(masks))
        self.bad_masks[self.step + 1].copy_(f(bad_masks))
        self.step = (self.step + 1) % self.num_steps

    def after_update(self):
        self.obs[0].copy_(self.obs[-1])
        self.masks[0].copy_(self.masks[-1])
        self.bad_masks[0].copy_(self.bad_masks[-1])

    def compute_returns(self, next_value, use_gae, gamma, gae_lambda, use_proper_time_limits=True):
        # PPO.update re-derives the advantage with the same branch and values (return_branch())
        self.gamma, self.gae_lambda = gamma, gae_lambda
        self.use_gae, self.use_proper_time_limits = bool(use_gae), bool(use_proper_time_limits)
        nv = torch.as_tensor(next_value).to(self.obs.device, torch.float32)
        if use_gae:
            self.value_preds[-1].copy_(nv)
        else:
            self.returns[-1].copy_(nv)        # the n-step branches bootstrap from returns[-1]; value_preds[-1] is left alone
        T, N, M = self.rewards.shape
        ret, _ = K.returns_adv(self.rewards[None], self.value_preds[None], self.masks.view(1, T + 1, N),
                               self.bad_masks.view(1, T + 1, N), gamma, gae_lambda, **self.return_branch())
        self.returns[:-1].copy_(ret[0])

    def return_branch(self):
        """Keyword arguments of kernels.returns_adv for the branch the last compute_returns took (default: GAE with
        proper time limits, morl/run.py:56-70)."""
        use_gae = getattr(self, "use_gae", True)
        return dict(use_gae=use_gae, use_proper_time_limits=getattr(self, "use_proper_time_limits", True),
                    boot=None if use_gae else self.returns[-1][None])

    def feed_forward_generator(self, advantages, num_mini_batch=None, mini_batch_size=None):
        """Same minibatches as storage.py:118-154 (torch.randperm on the global CPU generator); the device PPO
        update consumes the permutation directly, this generator is kept for API parity."""
        T, N = self.rewards.shape[0:2]
        batch_size = N * T
        if mini_batch_size is None:
            mini_batch_size = batch_size // num_mini_batch
        perm = torch.randperm(batch_size)
        flat = lambda t, last: t.reshape(-1, last)
        for b in range(batch_size // mini_batch_size):
            idx = perm[b * mini_batch_size:(b + 1) * mini_batch_size].to(self.obs.device)
            yield (flat(self.obs[:-1], self.obs.shape[-1])[idx], flat(self.recurrent_hidden_states[:-1], 1)[idx],
                   flat(self.actions, self.actions.shape[-1])[idx], flat(self.value_preds[:-1], self.value_preds.shape[-1])[idx],
                   flat(self.returns[:-1], self.returns.shape[-1])[idx], flat(self.masks[:-1], 1)[idx],
                   flat(self.action_log_probs, 1)[idx], None if advantages is None else advantages.reshape(-1, 1)[idx])
