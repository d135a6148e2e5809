"""Running observation / return / objective normalisation on the device for a whole population shard
(SURVEY 8(f2)): the state machine of VecNormalize (externals/baselines/baselines/common/vec_env/vec_normalize.py:11-66,
a2c/envs.py:197-211) and RunningMeanStd (baselines/common/running_mean_std.py:4-31), P tasks x N environments at once.

The host environment workers hand over RAW simulator output; kernel K6 (`pgm_vecnorm_step_f64`) updates the FP64
running moments and writes the normalised float32 observation, reward vector and mask straight into the slots of the
rollout buffers that K1 / K2 read (`PopulationMOPG.obs / rewards / masks`). Moments are bit-identical to the
reference's, so `Sample.env_params` snapshots (`ob_rms`, `ret_rms`, `obj_rms`) interchange with its pickles.
"""
import ctypes as C

import numpy as np
import torch

from ._lib import check, lib, ptr


class RunningMeanStd:
    """Host snapshot with the reference's attribute names (running_mean_std.py:4-9)."""

    def __init__(self, epsilon=1e-4, shape=()):
        self.mean, self.var, self.count = np.zeros(shape, 'float64'), np.ones(shape, 'float64'), epsilon


def _rms_class():
    """The class snapshots are made of: the reference's own `baselines.common.running_mean_std.RunningMeanStd` when that
    package is importable, so that final/EP_env_params_*.pkl (morl/morl.py:228) resolves for the reference's tooling
    without this package; the local stand-in (same attributes) otherwise."""
    try:
        from baselines.common.running_mean_std import RunningMeanStd as Ref
        return Ref
    except Exception:
        return RunningMeanStd


class DeviceVecNormalize:
    def __init__(self, P, N, obs_dim, obj_num, ob=True, ret=True, obj_rms=False, clipob=10., cliprew=10., gamma=0.99,
                 epsilon=1e-8, device="cuda"):
        self.P, self.N, self.O, self.M = P, N, obs_dim, obj_num
        self.clipob, self.cliprew, self.gamma, self.epsilon = clipob, cliprew, gamma, epsilon
        self.device = dev = torch.device(device)
        self.training = True                                   # a2c/envs.py:200, train() / eval()
        f64 = dict(device=dev, dtype=torch.float64)
        self.has_ob, self.has_ret, self.has_obj = bool(ob), bool(ret), bool(ret and obj_rms)
        self.ob_mean, self.ob_var = torch.zeros(P, obs_dim, **f64), torch.ones(P, obs_dim, **f64)
        self.ob_count = torch.full((P,), 1e-4, **f64)
        self.ret_acc = torch.zeros(P, N, **f64)
        self.ret_stat = torch.tensor([[0.0, 1.0, 1e-4]] * P, **f64)
        self.obj_acc = torch.zeros(P, N, obj_num, **f64)
        self.obj_started = torch.zeros(P, device=dev, dtype=torch.int32)
        self.obj_mean, self.obj_var = torch.zeros(P, obj_num, **f64), torch.ones(P, obj_num, **f64)
        self.obj_count = torch.full((P,), 1e-4, **f64)
        self._obj_scalar = [True] * P                          # obj_rms keeps shape () until its first update
        pin = lambda *s, dtype=torch.float64: torch.empty(*s, dtype=dtype, pin_memory=True)
        self._h = {"obs": pin(P, N, obs_dim), "rew": pin(P, N), "obj": pin(P, N, obj_num), "done": pin(P, N, dtype=torch.uint8)}
        self._d = {k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in self._h.items()}

    def reset_state(self):
        """Back to the state of a freshly constructed object (the shard's normaliser is reused by every generation)."""
        self.ob_mean.zero_(); self.ob_var.fill_(1.0); self.ob_count.fill_(1e-4)
        self.ret_acc.zero_()
        self.ret_stat.copy_(torch.tensor([[0.0, 1.0, 1e-4]] * self.P, dtype=torch.float64))
        self.obj_acc.zero_(); self.obj_started.zero_()
        self.obj_mean.zero_(); self.obj_var.fill_(1.0); self.obj_count.fill_(1e-4)
        self._obj_scalar = [True] * self.P
        self.training = True

    def mark_stepped(self):
        """Steps were run through the rollout-slot entry point (rollout.StepPipe): obj_rms now has its vector shape."""
        if self.has_obj:
            self._obj_scalar = [False] * self.P

    def train(self):
        self.training = True

    def eval(self):
        self.training = False

    # ------------------------------------------------------------------ Sample.env_params <-> device state
    def load_task(self, p, env_params):
        """Install the running moments a Sample carries (mopg.py:70-75)."""
        as64 = lambda x, n: torch.as_tensor(np.broadcast_to(np.asarray(x, dtype=np.float64), (n,)).copy())
        rms = env_params.get('ob_rms')
        if rms is not None:
            self.ob_mean[p].copy_(as64(rms.mean, self.O)); self.ob_var[p].copy_(as64(rms.var, self.O))
            self.ob_count[p] = float(rms.count)
        rms = env_params.get('ret_rms')
        if rms is not None:
            self.ret_stat[p].copy_(torch.tensor([float(rms.mean), float(rms.var), float(rms.count)], dtype=torch.float64))
        rms = env_params.get('obj_rms')
        if rms is not None:
            self._obj_scalar[p] = np.ndim(rms.mean) == 0
            self.obj_mean[p].copy_(as64(rms.mean, self.M)); self.obj_var[p].copy_(as64(rms.var, self.M))
            self.obj_count[p] = float(rms.count)

    def snapshot(self, p):
        """-> {'ob_rms', 'ret_rms', 'obj_rms'} host copies for Sample.env_params (mopg.py:146-149)."""
        out = {'ob_rms': None, 'ret_rms': None, 'obj_rms': None}
        RunningMeanStd = _rms_class()
        if self.has_ob:
            r = RunningMeanStd(shape=(self.O,))
            r.mean, r.var, r.count = self.ob_mean[p].cpu().numpy(), self.ob_var[p].cpu().numpy(), float(self.ob_count[p])
            out['ob_rms'] = r
        if self.has_ret:
            r, st = RunningMeanStd(), self.ret_stat[p].cpu().numpy()
            r.mean, r.var, r.count = np.float64(st[0]), np.float64(st[1]), float(st[2])
            out['ret_rms'] = r
        if self.has_obj:
            r = RunningMeanStd()
            if self._obj_scalar[p]:                            # as loaded: shape () until the first update
                r.mean, r.var = self.obj_mean[p, 0].cpu().numpy(), self.obj_var[p, 0].cpu().numpy()
            else:
                r.mean, r.var = self.obj_mean[p].cpu().numpy(), self.obj_var[p].cpu().numpy()
            r.count = float(self.obj_count[p])
            out['obj_rms'] = r
        return out

    def obj_var_host(self, p):
        return self.obj_var[p].cpu().numpy()

    # ------------------------------------------------------------------ the per-step call
    def _launch(self, raw_obs, raw_rew, raw_obj, done, obs_out, obj_out, mask_out, reset):
        P, N, O, M = self.P, self.N, self.O, self.M
        for t, name in ((obs_out, "obs_out"), (obj_out, "obj_out"), (mask_out, "mask_out")):
            if t is not None and not (t.is_cuda and t.dtype == torch.float32 and t.stride(-1) == 1):
                raise ValueError(f"{name}: expected a float32 CUDA view with unit inner stride")
        st = lambda t: 0 if t is None else t.stride(0)
        check(lib().pgm_vecnorm_step_f64(
            ptr(raw_obs), ptr(raw_rew), ptr(raw_obj), ptr(done),
            ptr(self.ob_mean if self.has_ob else None), ptr(self.ob_var if self.has_ob else None),
            ptr(self.ob_count if self.has_ob else None),
            ptr(self.ret_acc if self.has_ret else None), ptr(self.ret_stat if self.has_ret else None),
            ptr(self.obj_acc), ptr(self.obj_started),
            ptr(self.obj_mean if self.has_obj else None), ptr(self.obj_var if self.has_obj else None),
            ptr(self.obj_count if self.has_obj else None),
            ptr(obs_out), st(obs_out), ptr(obj_out), st(obj_out), ptr(mask_out), st(mask_out),
            self.gamma, self.clipob, self.cliprew, self.epsilon, int(self.training), int(reset), P, N, O, M,
            C.c_void_p(torch.cuda.current_stream().cuda_stream)))

    def _up(self, key, value):
        h, d = self._h[key], self._d[key]
        h.copy_(torch.as_tensor(np.ascontiguousarray(value)).reshape(h.shape))
        d.copy_(h, non_blocking=True)
        return d

    def reset(self, raw_obs, obs_out):
        """VecNormalize.reset on every task: raw_obs [P,N,O] (host) -> obs_out[p] = normalised [N,O] rows (device view)."""
        self._launch(self._up("obs", raw_obs), None, None, None, obs_out, None, None, True)

    def step(self, raw_obs, raw_rew, raw_obj, done, obs_out, obj_out, mask_out):
        """VecNormalize.step_wait on every task. Host inputs: raw_obs [P,N,O], raw_rew [P,N] (or None), raw_obj [P,N,M],
        done [P,N] bool. Device views written: obs_out[p] [N,O], obj_out[p] [N,M], mask_out[p] [N] (1 - done)."""
        rew = self._up("rew", raw_rew) if raw_rew is not None else None
        self._launch(self._up("obs", raw_obs), rew, self._up("obj", raw_obj),
                     self._up("done", np.asarray(done, dtype=np.uint8)), obs_out, obj_out, mask_out, False)
        if self.has_obj:
            self._obj_scalar = [False] * self.P
