"""CPU restatement of the running normalisation K6 replaces -- TEST INFRASTRUCTURE ONLY (imported by tests/ and
__graft_entry__.smoke(); never by pgmorl_b200/).

Follows externals/baselines/baselines/common/vec_env/vec_normalize.py:29-66 (step_wait / _obfilt / reset) and
externals/baselines/baselines/common/running_mean_std.py:10-31, with numpy's reductions written out element by
element so the evaluation order the CUDA kernel must reproduce is explicit. Pinned bit for bit by
tests/golden/vecnorm.npz (outputs of the unmodified reference files, tests/golden/make_golden_vecnorm.py).
"""
import numpy as np


def _sum_rows(x):
    """np.add.reduce(x, axis=0) of a C-contiguous [N, ...] array: rows are added one after the other."""
    s = x[0].copy()
    for n in range(1, x.shape[0]):
        s = s + x[n]
    return s


def _pairwise(a):
    """numpy's pairwise summation of a contiguous 1-D block of <= 128 doubles."""
    n = len(a)
    if n < 8:
        res = np.float64(0.0)
        for v in a:
            res = res + v
        return res
    r = [np.float64(a[j]) for j in range(8)]
    i = 8
    while i < n - (n % 8):
        for j in range(8):
            r[j] = r[j] + a[i + j]
        i += 8
    res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
    while i < n:
        res = res + a[i]
        i += 1
    return res


def _sum_1d(a):
    """np.add.reduce of a contiguous 1-D array = the pairwise sum (probe: 2000 random vectors per length 3..20)."""
    return _pairwise(a)


def batch_moments(x):
    """(np.mean(x, axis=0), np.var(x, axis=0)) as RunningMeanStd.update computes them (running_mean_std.py:16-18)."""
    n = np.float64(x.shape[0])
    if x.ndim == 2 and x.shape[1] == 1:
        # numpy collapses a C-contiguous [N, 1] block into one contiguous 1-D reduction: pairwise, not row by row
        mean, var = batch_moments(x[:, 0])
        return np.array([mean]), np.array([var])
    if x.ndim == 1:
        mean = _sum_1d(x) / n
        d = x - mean
        return mean, _sum_1d(d * d) / n
    mean = _sum_rows(x) / n
    d = x - mean
    return mean, _sum_rows(d * d) / n


class RunningMeanStd:
    """running_mean_std.py:4-31"""

    def __init__(self, epsilon=1e-4, shape=()):
        self.mean, self.var, self.count = np.zeros(shape, "float64"), np.ones(shape, "float64"), epsilon

    def update(self, x):
        bmean, bvar = batch_moments(np.asarray(x, dtype=np.float64))
        bcount = x.shape[0]
        delta = bmean - self.mean
        tot = self.count + bcount
        new_mean = self.mean + delta * bcount / tot
        m2 = self.var * self.count + bvar * bcount + np.square(delta) * self.count * bcount / tot
        self.mean, self.var, self.count = new_mean, m2 / tot, tot


class VecNormalizeOracle:
    """One task's VecNormalize state machine on raw arrays (vec_normalize.py:11-66, a2c/envs.py:197-211)."""

    def __init__(self, N, O, ob=True, ret=True, obj_rms=False, clipob=10.0, cliprew=10.0, gamma=0.99, epsilon=1e-8):
        self.ob_rms = RunningMeanStd(shape=(O,)) if ob else None
        self.ret_rms = RunningMeanStd(shape=()) if ret else None
        self.obj_rms = RunningMeanStd(shape=()) if ret and obj_rms else None
        self.clipob, self.cliprew, self.gamma, self.epsilon = clipob, cliprew, gamma, epsilon
        self.ret, self.obj = np.zeros(N), None

    def _obfilt(self, obs, update=True):
        if self.ob_rms is None:
            return obs
        if update:
            self.ob_rms.update(obs)
        return np.clip((obs - self.ob_rms.mean) / np.sqrt(self.ob_rms.var + self.epsilon), -self.clipob, self.clipob)

    def reset(self, raw_obs):
        self.ret = np.zeros(len(self.ret))
        return self._obfilt(raw_obs)

    def step(self, raw_obs, raw_rew, raw_obj, done, update=True):
        """-> (normalised obs, normalised scalar reward, normalised objective vectors [N,M])"""
        self.ret = self.ret * self.gamma + raw_rew
        self.obj = self.obj * self.gamma + raw_obj if self.obj is not None else raw_obj.copy()
        obs = self._obfilt(raw_obs, update)
        rew, obj = raw_rew, raw_obj
        if self.ret_rms is not None:
            self.ret_rms.update(self.ret)
            rew = np.clip(raw_rew / np.sqrt(self.ret_rms.var + self.epsilon), -self.cliprew, self.cliprew)
        if self.obj_rms is not None:
            self.obj_rms.update(self.obj)
            obj = np.clip(raw_obj / np.sqrt(self.obj_rms.var + self.epsilon), -self.cliprew, self.cliprew)
        self.ret[done] = 0.0
        self.obj[done] = 0.0
        return obs, rew, obj
