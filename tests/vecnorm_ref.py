"""Literal numpy restatement of the running normalisation K6 replaces -- test reference only.

RunningMeanStd is externals/baselines/baselines/common/running_mean_std.py:4-31 as written there: np.mean / np.var over
axis 0, then update_mean_var_count_from_moments. VecNormalize is the state machine of vec_env/vec_normalize.py:11-66 with
the a2c override of _obfilt (a2c_ppo_acktr/envs.py:197-211): the return and objective accumulators, train() / eval()
gating only the observation moments, reset restarting the returns, np.clip and np.sqrt(var + epsilon).

Nothing here sums element by element: numpy chooses every reduction order, so this file carries no assumption about
that order (oracle/vecnorm_oracle.py writes the order out; this file is what it and K6 are checked against).
"""
import numpy as np


class RunningMeanStd:
    """running_mean_std.py:4-31"""

    def __init__(self, epsilon=1e-4, shape=()):
        self.mean = np.zeros(shape, 'float64')
        self.var = np.ones(shape, 'float64')
        self.count = epsilon

    def update(self, x):
        batch_mean, batch_var, batch_count = np.mean(x, axis=0), np.var(x, axis=0), x.shape[0]
        delta = batch_mean - self.mean
        tot = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot
        m2 = self.var * self.count + batch_var * batch_count + np.square(delta) * self.count * batch_count / tot
        self.mean, self.var, self.count = new_mean, m2 / tot, tot


class VecNormalize:
    """One task's VecNormalize on raw [N, ...] arrays: step() returns (obs, rew, obj) as the wrapper hands them on."""

    def __init__(self, N, O, ob=True, ret=True, obj_rms=False, clipob=10., cliprew=10., gamma=0.99, epsilon=1e-8):
        self.ob_rms = RunningMeanStd(shape=(O,)) if ob else None
        self.ret_rms = RunningMeanStd(shape=()) if ret else None
        self.obj_rms = RunningMeanStd(shape=()) if ret and obj_rms else None
        self.clipob, self.cliprew, self.gamma, self.epsilon = clipob, cliprew, gamma, epsilon
        self.ret = np.zeros(N)
        self.obj = None
        self.training = True

    def train(self):
        self.training = True

    def eval(self):
        self.training = False

    def _obfilt(self, obs, update=True):
        if self.ob_rms is None:
            return obs
        if self.training and update:
            self.ob_rms.update(obs)
        return np.clip((obs - self.ob_rms.mean) / np.sqrt(self.ob_rms.var + self.epsilon), -self.clipob, self.clipob)

    def reset(self, obs):
        self.ret = np.zeros(len(self.ret))
        return self._obfilt(obs)

    def step(self, obs, rews, objs, news):
        self.ret = self.ret * self.gamma + rews
        self.obj = objs.copy() if self.obj is None else self.obj * self.gamma + objs
        obs = self._obfilt(obs)
        if self.ret_rms is not None:
            self.ret_rms.update(self.ret)
            rews = np.clip(rews / np.sqrt(self.ret_rms.var + self.epsilon), -self.cliprew, self.cliprew)
        if self.obj_rms is not None:
            self.obj_rms.update(self.obj)
            objs = np.clip(objs / np.sqrt(self.obj_rms.var + self.epsilon), -self.cliprew, self.cliprew)
        self.ret[news] = 0.
        self.obj[news] = 0.
        return obs, rews, objs
