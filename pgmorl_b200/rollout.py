"""Per-step rollout pipe for real environment loops (morl/mopg.py:103-135 for a whole population shard).

The reference calls Policy.act once per environment step and task (2048 x P tiny torch calls per iteration) and
inserts the results into RolloutStorage. Here ONE CUDA graph replay per environment step serves all P tasks:

    H2D of one pinned staging block  ->  [K6: normalise the simulators' raw answer into rollout slot t]  ->
    K1 per-step mode: value / action / log-prob of slot t written straight into the rollout buffers  ->
    D2H of the dense action block

The time slot and the mode flags travel inside the staging block (device control word), so the captured graph is the
same for every step of every iteration: per step the host pays one graph launch and one stream synchronise instead of
~25 small copies and launches. Reward vectors / masks of the host-normalised mode are not needed by K1 at all: they
are collected in pinned memory during the rollout and uploaded once before K2.
"""
import ctypes as C

import numpy as np
import torch

from . import kernels as K
from ._lib import check, lib, ptr
from ._nvtx import rng as _nvtx


def _carve(nbytes_by_name):
    """name -> (offset, nbytes), every block 16-byte aligned; returns (layout, total)."""
    off, out = 0, {}
    for name, n in nbytes_by_name:
        out[name] = (off, n)
        off += (n + 15) // 16 * 16
    return out, off


class StepPipe:
    """`vn` = DeviceVecNormalize of the shard (raw-simulator mode, K6 on the device) or None (the environments hand
    over normalised observations / objective vectors, as a2c_ppo_acktr.envs.make_vec_envs does)."""

    def __init__(self, pop, vn=None):
        self.pop, self.vn = pop, vn
        P, N, d = pop.P, pop.N, pop.dims
        O, A, M = d.obs, d.act, d.obj
        self.P, self.N, self.O, self.A, self.M = P, N, O, A, M
        AC = d.act_cols        # noise block [1,N,A] (A = n Exponential(1) draws for a Categorical head), actions [P,N,AC]
        blocks = [("ctl", 16)]
        if vn is not None:
            blocks += [("raw_obs", 8 * P * N * O), ("raw_rew", 8 * P * N), ("raw_obj", 8 * P * N * M),
                       ("bad", 4 * P * N), ("done", P * N)]
        else:
            blocks += [("obs", 4 * P * N * O)]
        blocks += [("eps", 4 * N * A)]
        self.layout, total = _carve(blocks)
        self.h = torch.zeros(total, dtype=torch.uint8, pin_memory=True)
        self.dv = torch.zeros(total, dtype=torch.uint8, device=pop.device)
        self.h_act = torch.zeros(P, N, AC, dtype=torch.float32, pin_memory=True)
        self.d_act = torch.zeros(P, N, AC, dtype=torch.float32, device=pop.device)

        def view(buf, name, dtype, shape):
            o, n = self.layout[name]
            return buf[o:o + n].view(dtype).view(*shape)

        self.h_ctl, self.d_ctl = view(self.h, "ctl", torch.int32, (4,)), view(self.dv, "ctl", torch.int32, (4,))
        self.h_eps, self.d_eps = view(self.h, "eps", torch.float32, (1, N, A)), view(self.dv, "eps", torch.float32, (1, N, A))
        if vn is not None:
            self.h_raw_obs, self.d_raw_obs = (view(b, "raw_obs", torch.float64, (P, N, O)) for b in (self.h, self.dv))
            self.h_raw_rew, self.d_raw_rew = (view(b, "raw_rew", torch.float64, (P, N)) for b in (self.h, self.dv))
            self.h_raw_obj, self.d_raw_obj = (view(b, "raw_obj", torch.float64, (P, N, M)) for b in (self.h, self.dv))
            self.h_bad, self.d_bad = (view(b, "bad", torch.float32, (P, N)) for b in (self.h, self.dv))
            self.h_done, self.d_done = (view(b, "done", torch.uint8, (P, N)) for b in (self.h, self.dv))
            self.h_obs = self.d_obs = None
        else:
            self.h_obs, self.d_obs = (view(b, "obs", torch.float32, (P, N, O)) for b in (self.h, self.dv))
        # numpy views of the pinned blocks: the per-step host work is plain array assignment
        self.np_ctl = self.h_ctl.numpy()
        self.np_eps = self.h_eps.numpy()
        self.np_act = self.h_act.numpy()
        self.graph = None

    # ------------------------------------------------------------------ the device work of one step
    def _launch(self):
        pop, vn = self.pop, self.vn
        self.dv.copy_(self.h, non_blocking=True)
        if vn is not None:
            check(lib().pgm_vecnorm_rollout_step_f64(
                ptr(self.d_ctl), ptr(self.d_raw_obs), ptr(self.d_raw_rew), ptr(self.d_raw_obj), ptr(self.d_done),
                ptr(self.d_bad),
                ptr(vn.ob_mean if vn.has_ob else None), ptr(vn.ob_var if vn.has_ob else None),
                ptr(vn.ob_count if vn.has_ob else None),
                ptr(vn.ret_acc if vn.has_ret else None), ptr(vn.ret_stat if vn.has_ret else None),
                ptr(vn.obj_acc), ptr(vn.obj_started),
                ptr(vn.obj_mean if vn.has_obj else None), ptr(vn.obj_var if vn.has_obj else None),
                ptr(vn.obj_count if vn.has_obj else None),
                ptr(pop.obs), pop.obs.stride(0), ptr(pop.rewards), pop.rewards.stride(0),
                ptr(pop.masks), pop.masks.stride(0), ptr(pop.bad_masks), pop.bad_masks.stride(0),
                vn.gamma, vn.clipob, vn.cliprew, vn.epsilon, int(vn.training), self.P, self.N, self.O, self.M,
                C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        K.policy_step(pop.params, self.d_ctl, self.d_obs, self.d_eps, pop.obs, pop.value, pop.action, pop.logp,
                      self.d_act, self.N, pop.dims)
        self.h_act.copy_(self.d_act, non_blocking=True)

    def _capture(self):
        # warm-up on a side stream (module loading, attribute calls), then capture the three operations once
        side = torch.cuda.Stream(device=self.pop.device)
        side.wait_stream(torch.cuda.current_stream())
        keep = self.np_ctl.copy()
        self.np_ctl[:] = (0, 0, 0, 0)              # t = 0, value only, no normalisation: touches slot 0 harmlessly
        with torch.cuda.stream(side):
            saved = (self.pop.obs[:, :self.N].clone(), self.pop.value[:, :self.N].clone())
            self._launch()
            side.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                self._launch()
            side.synchronize()
            self.pop.obs[:, :self.N].copy_(saved[0]); self.pop.value[:, :self.N].copy_(saved[1])
            side.synchronize()
        torch.cuda.current_stream().wait_stream(side)
        self.np_ctl[:] = keep
        self.graph = g

    # ------------------------------------------------------------------ host API
    def step(self, t, eps_t, sample=True, normalise=False):
        """Run slot t for all tasks on whatever the staging block holds (fill `h_obs` or the raw blocks first).
        eps_t: float64 [N,A] draw of this step (None for the bootstrap). Returns the pinned action block [P,N,A]
        ([P,N,1] float32 category indices for a Categorical head; valid until the next call)."""
        self.np_ctl[0] = t
        self.np_ctl[1] = (1 if sample else 0) | (2 if normalise else 0)
        if eps_t is not None:
            self.np_eps[0] = eps_t.numpy() if hasattr(eps_t, "numpy") else eps_t
        if self.graph is None:
            self._capture()
        with _nvtx("rollout.step"):
            self.graph.replay()
            torch.cuda.current_stream().synchronize()
        return self.h_act
