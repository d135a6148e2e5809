"""Device-resident population state and the batched MOPG iteration (K1 -> K2 -> K3).

The reference runs one OS process per task (morl/morl.py:84-88), each looping
morl/mopg.py:96-144. Here all P tasks of this GPU's shard live in one
struct-of-arrays state in HBM and advance together, one kernel launch per stage:

    params, adam_m, adam_v  [P, n_par] f32      adam_step [P] i32     lr [P] f64
    weights, obj_var        [P, M]     f32

Rollout buffers are preallocated once (nothing is allocated per iteration), host inputs
arrive through pinned staging buffers, and the three stages run back to back on the
current CUDA stream.
"""
import numpy as np
import torch

from . import kernels as K
from ._nvtx import rng as _nvtx
from ._lib import PpoHyper
from .layout import NetDims


class PopulationMOPG:
    def __init__(self, dims: NetDims, P, T, N, ppo_epoch=10, num_mini_batch=32, gamma=0.995, gae_lambda=0.95,
                 hyper: PpoHyper = None, device="cuda", cluster=0, shared_rng=True, use_gae=True,
                 use_proper_time_limits=True, clipped_value_loss=True):
        self.dims, self.P, self.T, self.N = dims, P, T, N
        self.E, self.B = ppo_epoch, num_mini_batch
        self.gamma, self.lam = gamma, gae_lambda
        # branch of compute_returns (storage.py:77-116; the n-step branches bootstrap from value row T, where K1 puts the
        # value of the last observation) and PPO's use_clipped_value_loss
        self.use_gae, self.use_proper_time_limits = use_gae, use_proper_time_limits
        self.clipped_value_loss = clipped_value_loss
        self.hyper = hyper or PpoHyper()
        self.device = torch.device(device)
        self.cluster = cluster
        self.shared_rng = shared_rng          # all tasks of a generation share eps / perm (mopg.py:96 seeds with j)
        S = self.S = T * N
        O, A, M = dims.obs, dims.act, dims.obj
        dv, f32 = self.device, torch.float32
        z = lambda *s, dtype=f32: torch.zeros(*s, device=dv, dtype=dtype)
        # ---- persistent per-task state
        self.params, self.adam_m, self.adam_v = z(P, dims.n_par), z(P, dims.n_par), z(P, dims.n_par)
        self.adam_step = z(P, dtype=torch.int32)
        self.lr = z(P, dtype=torch.float64)
        self.weights, self.obj_var = z(P, M), z(P, M)
        # ---- rollout buffers
        Pr = 1 if shared_rng else P
        self.obs = z(P, (T + 1) * N, O)
        self.rewards = z(P, T, N, M)
        self.masks, self.bad_masks = z(P, T + 1, N), z(P, T + 1, N)
        self.eps = z(Pr, S, A)
        self.perm = z(Pr, self.E, S, dtype=torch.int32)
        self.value = z(P, (T + 1) * N, M)
        self.action, self.logp = z(P, S, dims.act_cols), z(P, S)      # Categorical: one column, the category index
        self.returns, self.adv = z(P, T, N, M), z(P, T, N)
        self.losses = z(P, 3)
        self.workspace = K.ppo_workspace(P, S, dims, dv, cluster)
        # ---- pinned host staging (end-to-end path)
        pin = lambda t: torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        self._h = {k: pin(getattr(self, k)) for k in ("obs", "rewards", "masks", "bad_masks", "eps", "perm")}
        self._h_losses = pin(self.losses)
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self._h.values())
        self.d2h_bytes = self._h_losses.numel() * self._h_losses.element_size()

    # ------------------------------------------------------------------ state in / out
    def load_task(self, p, flat, adam_m=None, adam_v=None, adam_step=0, weights=None, obj_var=None):
        """Install task p from float64/float32 host vectors (a Sample's policy + Adam state)."""
        as32 = lambda x: torch.as_tensor(np.asarray(x), dtype=torch.float32)
        self.params[p].copy_(as32(flat))
        self.adam_m[p].copy_(as32(adam_m)) if adam_m is not None else self.adam_m[p].zero_()
        self.adam_v[p].copy_(as32(adam_v)) if adam_v is not None else self.adam_v[p].zero_()
        self.adam_step[p] = int(adam_step)
        if weights is not None:
            self.weights[p].copy_(as32(weights))
        if obj_var is not None:
            self.obj_var[p].copy_(as32(obj_var))

    def set_lr(self, lr):
        self.lr.copy_(torch.as_tensor(np.broadcast_to(np.asarray(lr, dtype=np.float64), (self.P,)).copy()))

    def task_state(self, p):
        """-> (flat, adam_m, adam_v) float64 numpy + step (what a Sample snapshot stores)."""
        f = lambda t: t[p].detach().cpu().numpy().astype(np.float64)
        return f(self.params), f(self.adam_m), f(self.adam_v), int(self.adam_step[p])

    # ------------------------------------------------------------------ the hot path
    def step(self):
        """One MOPG iteration for all P tasks on data already resident in HBM
        (rollout inference -> vector GAE + advantage -> PPO update). Asynchronous."""
        T, N, P, d = self.T, self.N, self.P, self.dims
        with _nvtx("mopg.k1_forward"):
            K.policy_forward(self.params, self.obs, d, eps=self.eps, rows_a=self.S,
                             out=(self.value, self.action, self.logp))
        with _nvtx("mopg.k2_gae_adv"):
            self._returns_adv()
        with _nvtx("mopg.k3_ppo_update"):
            self._ppo_update()
        return self.losses

    def _returns_adv(self):
        T, N, P, d = self.T, self.N, self.P, self.dims
        K.returns_adv(self.rewards, self.value.view(P, T + 1, N, d.obj), self.masks, self.bad_masks, self.gamma, self.lam,
                      use_gae=self.use_gae, use_proper_time_limits=self.use_proper_time_limits, weights=self.weights,
                      obj_var=self.obj_var, out=(self.returns, self.adv))

    def _ppo_update(self):
        P, d = self.P, self.dims
        K.ppo_update(self.params, self.adam_m, self.adam_v, self.adam_step, self.lr, self.obs, self.action,
                     self.logp, self.value, self.returns.view(P, self.S, d.obj), self.adv.view(P, self.S),
                     self.perm, self.B, d, hyper=self.hyper, workspace=self.workspace, cluster=self.cluster,
                     losses=self.losses, clipped_value_loss=self.clipped_value_loss)

    GPU_LAUNCHES_PER_STEP = 4   # K1 forward, K2 GAE/adv, K3 record pack, K3 PPO

    # ------------------------------------------------------------------ per-step mode (real environment loops)
    def act_step(self, t, obs_host, eps_t):
        """K1 in per-step mode: obs_host [P,N,O] (host) at time t, eps_t [N,A] float64 shared by all tasks.
        Stores obs/value/action/logp of step t in the rollout buffers; returns actions [P,N,A] (device; [P,N,1] category
        indices as float32 for a Categorical head)."""
        P, N, d = self.P, self.N, self.dims
        if not hasattr(self, "_step_obs"):
            self._step_obs = torch.empty(P, N, d.obs, device=self.device)
            self._step_out = (torch.empty(P, N, d.obj, device=self.device), torch.empty(P, N, d.act_cols, device=self.device),
                              torch.empty(P, N, device=self.device))
        self._step_obs.copy_(obs_host)
        eps = eps_t.to(self.device, torch.float32)[None].contiguous()
        value, action, logp = K.policy_forward(self.params, self._step_obs, d, eps=eps, out=self._step_out)
        rows = slice(t * N, (t + 1) * N)
        self.obs[:, rows].copy_(self._step_obs)
        self.value[:, rows].copy_(value); self.action[:, rows].copy_(action); self.logp[:, rows].copy_(logp)
        return action

    def act_step_resident(self, t, eps_t):
        """K1 in per-step mode on the observation ALREADY in the rollout buffer (written there by K6,
        vec_normalize.DeviceVecNormalize): nothing but the noise travels host -> device. Returns actions [P,N,A]."""
        P, N, d = self.P, self.N, self.dims
        if not hasattr(self, "_step_obs"):
            self._step_obs = torch.empty(P, N, d.obs, device=self.device)
            self._step_out = (torch.empty(P, N, d.obj, device=self.device), torch.empty(P, N, d.act_cols, device=self.device),
                              torch.empty(P, N, device=self.device))
        rows = slice(t * N, (t + 1) * N)
        self._step_obs.copy_(self.obs[:, rows])
        eps = eps_t.to(self.device, torch.float32)[None].contiguous()
        value, action, logp = K.policy_forward(self.params, self._step_obs, d, eps=eps, out=self._step_out)
        self.value[:, rows].copy_(value); self.action[:, rows].copy_(action); self.logp[:, rows].copy_(logp)
        return action

    def finish_rollout_resident(self):
        """Bootstrap value of the observation K6 left in the last slot (mopg.py:132-135)."""
        T, N, d = self.T, self.N, self.dims
        self._step_obs.copy_(self.obs[:, T * N:])
        value, _, _ = K.policy_forward(self.params, self._step_obs, d, rows_a=0, mode=K.ACT_DETERMINISTIC)
        self.value[:, T * N:].copy_(value)

    def store_transition(self, p, t, objs, masks, bad_masks):
        """Reward vector / termination flags task p observed after step t (host values)."""
        self.rewards[p, t].copy_(torch.as_tensor(objs, dtype=torch.float32))
        self.masks[p, t + 1].copy_(torch.as_tensor(masks, dtype=torch.float32))
        self.bad_masks[p, t + 1].copy_(torch.as_tensor(bad_masks, dtype=torch.float32))

    def finish_rollout(self, obs_host):
        """Bootstrap value of the observation after the last step (mopg.py:132-135)."""
        T, N, d = self.T, self.N, self.dims
        self._step_obs.copy_(obs_host)
        value, _, _ = K.policy_forward(self.params, self._step_obs, d, rows_a=0, mode=K.ACT_DETERMINISTIC)
        self.obs[:, T * N:].copy_(self._step_obs)
        self.value[:, T * N:].copy_(value)

    def update_only(self):
        """K2 + K3 on the rollout already in the buffers."""
        self._returns_adv()
        self._ppo_update()
        return self.losses

    def upload(self, obs, rewards, masks, bad_masks, eps, perm):
        """Stage one iteration's host inputs through pinned memory and copy them to HBM (async)."""
        src = dict(obs=obs, rewards=rewards, masks=masks, bad_masks=bad_masks, eps=eps, perm=perm)
        for k, t in src.items():
            h = self._h[k]
            h.copy_(torch.as_tensor(t).reshape(h.shape))
            getattr(self, k).copy_(h, non_blocking=True)

    def upload_staged(self):
        """H2D of whatever already sits in the pinned staging buffers (bench end-to-end leg)."""
        for k, h in self._h.items():
            getattr(self, k).copy_(h, non_blocking=True)

    # ---- pipelined uploads: the next iteration's inputs travel host -> HBM on a copy stream while this one computes ----
    def upload_staged_async(self):
        """H2D of the pinned staging buffers into the ALTERNATE set of input buffers, on a separate stream.
        The caller must have finished (synchronised) the iteration that last read the alternate set."""
        if not hasattr(self, "_alt"):
            self._alt = {k: torch.empty_like(getattr(self, k)) for k in self._h}
            self._copy_stream = torch.cuda.Stream(device=self.device)
            self._copy_done = torch.cuda.Event()
        with torch.cuda.stream(self._copy_stream):
            for k, h in self._h.items():
                self._alt[k].copy_(h, non_blocking=True)
            self._copy_done.record(self._copy_stream)

    def swap_inputs(self):
        """Make the set filled by the last upload_staged_async() current (the compute stream waits for that copy)."""
        torch.cuda.current_stream().wait_event(self._copy_done)
        for k in self._h:
            cur = getattr(self, k)
            setattr(self, k, self._alt[k])
            self._alt[k] = cur

    def step_from_host(self, obs, rewards, masks, bad_masks, eps, perm):
        """End-to-end call: host buffers in, host losses out (H2D + K1..K3 + D2H)."""
        self.upload(obs, rewards, masks, bad_masks, eps, perm)
        self.step()
        self._h_losses.copy_(self.losses, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._h_losses.numpy().copy()

    def staging(self):
        """The pinned host buffers the environment workers fill for the next iteration: obs, rewards, masks, bad_masks,
        eps, perm (shapes of the device buffers)."""
        return self._h

    def step_from_staged(self, snapshot_slot=None):
        """End-to-end call on the inputs sitting in the pinned staging buffers: blocking sequence H2D of THIS iteration's
        inputs -> K1..K3 -> (optional) device snapshot of every task's state -> D2H of the losses -> host wait.
        Nothing of the next iteration overlaps: an on-policy loop cannot have its inputs before this update is done."""
        self.upload_staged()
        self.step()
        if snapshot_slot is not None:
            self.snapshot(snapshot_slot)
        self._h_losses.copy_(self.losses, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._h_losses

    # ---- per-iteration offspring snapshots (what morl/mopg.py:146-149 deep-copies into a Sample), kept on the device ----
    def snapshot(self, slot):
        """Copy params / Adam moments / step of every task into snapshot slot `slot` (ring of `n_slots` slots, allocated on
        first use: one per iteration of a generation)."""
        if not hasattr(self, "_snap"):
            self.alloc_snapshots(20)
        k = slot % self._snap.shape[0]
        self._snap[k, :, 0].copy_(self.params); self._snap[k, :, 1].copy_(self.adam_m); self._snap[k, :, 2].copy_(self.adam_v)
        self._snap_step[k].copy_(self.adam_step)

    def alloc_snapshots(self, n_slots):
        self._snap = torch.empty(n_slots, self.P, 3, self.dims.n_par, device=self.device)
        self._snap_step = torch.empty(n_slots, self.P, dtype=torch.int32, device=self.device)

    def snapshot_state(self, slot, p):
        """-> (params, adam_m, adam_v [n_par] f32 views, step tensor) of task p in snapshot slot `slot`."""
        k = slot % self._snap.shape[0]
        return self._snap[k, p, 0], self._snap[k, p, 1], self._snap[k, p, 2], self._snap_step[k, p]
