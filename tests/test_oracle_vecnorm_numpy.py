"""tests/vecnorm_ref.py (numpy choosing every reduction order) against the golden vectors of the unmodified reference,
and oracle/vecnorm_oracle.py's written-out reductions against numpy itself at every batch size K6 accepts (N <= 128)."""
import os

import numpy as np
import pytest

import vecnorm_ref
from oracle.vecnorm_oracle import batch_moments

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vecnorm.npz"))


@pytest.mark.parametrize("case", ["n4", "n9", "n1"])
def test_numpy_reference_matches_golden_bit_for_bit(case):
    N, O, M, steps = (int(v) for v in G[case + "_dims"])
    env = vecnorm_ref.VecNormalize(N, O, ob=True, ret=True, obj_rms=True, gamma=float(G[case + "_gamma"]))
    assert np.array_equal(env.reset(G[case + "_reset_obs"]).astype(np.float32), G[case + "_reset_out"])
    for t in range(steps):
        obs, _, obj = env.step(G[case + "_raw_obs"][t], G[case + "_raw_rew"][t], G[case + "_raw_obj"][t],
                               G[case + "_raw_done"][t])
        assert np.array_equal(obs.astype(np.float32), G[case + "_obs_out"][t]), t
        assert np.array_equal(obj, G[case + "_obj_out"][t]), t
    for name, rms in (("ob", env.ob_rms), ("ret", env.ret_rms), ("obj", env.obj_rms)):
        assert np.array_equal(rms.mean, G[case + "_" + name + "_mean"]), name
        assert np.array_equal(rms.var, G[case + "_" + name + "_var"]), name
        assert rms.count == float(G[case + "_" + name + "_count"])
    assert np.array_equal(env.ret, G[case + "_ret_acc"]) and np.array_equal(env.obj, G[case + "_obj_acc"])


@pytest.mark.parametrize("width", [None, 1, 2, 3, 17, 376])
def test_batch_moments_equal_numpy_at_every_batch_size(width):
    """np.mean / np.var over axis 0 of a C-contiguous block: rows one after the other at width >= 2, but a width-1
    block is reduced by numpy as one contiguous 1-D array (pairwise from N = 8 on), like a 1-D vector (width None)."""
    rng = np.random.RandomState(5 if width is None else width)
    for N in range(1, 129):
        for k in range(4):
            shape = (N,) if width is None else (N, width)
            x = rng.standard_normal(shape) * 10.0 ** rng.uniform(-3, 3) + rng.uniform(-50, 50)
            mean, var = batch_moments(x)
            assert mean.shape == np.mean(x, axis=0).shape
            assert np.array_equal(mean, np.mean(x, axis=0)), (N, k)
            assert np.array_equal(var, np.var(x, axis=0)), (N, k)
