"""K6 against tests/vecnorm_ref.py, the literal numpy VecNormalize / RunningMeanStd in which numpy itself decides every
reduction order, at the shapes, settings and values pgm_vecnorm_step_f64 / pgm_vecnorm_rollout_step_f64 accept.

Every comparison is bit for bit: float32 observations and objective vectors, masks, every FP64 running moment and
count, and the return / objective accumulators (signed zeros included; NaN equals NaN only in the NaN / inf case).
Covered: batch sizes on both sides of the pairwise sum's 8-lane blocks (N = 1 ... 128), widths 1 (numpy reduces an
[N, 1] column pairwise, wider blocks row by row) up to Humanoid's 376, every on / off combination of the three
normalisers with non-default gamma / clip / epsilon, loaded and snapshotted moments, clipping, constant features,
magnitudes from 1e-150 to 1e150, NaN / inf from a simulator, the rollout-slot entry point, and a whole MOPG iteration
at one observation feature with K1 / K3 checked there against the float64 oracle."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

import vecnorm_ref
from oracle import mopg_oracle as orc
from pgmorl_b200.layout import NetDims
from tests.helpers import rel_err
from tests.test_gpu_kernels import _ppo_inputs, dev, make_case

pytestmark = pytest.mark.gpu

SENT = -777.25           # sentinel in output buffers: cells K6 must not write keep it


def _same(got, want, nan=False):
    """Bit-for-bit equality of `got` with `want` converted to got's dtype (float32 outputs: numpy's own rounding of the
    float64 result); signed zeros must agree; NaN equals NaN only when `nan` is set."""
    got = np.asarray(got)
    want = np.broadcast_to(np.asarray(want).astype(got.dtype), got.shape)
    if not np.array_equal(got, want, equal_nan=nan):
        return False
    num = ~np.isnan(want)
    return np.array_equal(np.signbit(got[num]), np.signbit(want[num]))


def _state(env, p):
    """Device state of task p as host arrays, keyed like the reference's attributes."""
    h = lambda t: t[p].cpu().numpy()
    return dict(ob_mean=h(env.ob_mean), ob_var=h(env.ob_var), ob_count=h(env.ob_count), ret_acc=h(env.ret_acc),
                ret_stat=h(env.ret_stat), obj_acc=h(env.obj_acc), obj_mean=h(env.obj_mean), obj_var=h(env.obj_var),
                obj_count=h(env.obj_count))


def _check_state(env, refs, nan=False, where=""):
    for p, r in enumerate(refs):
        s = _state(env, p)
        if r.ob_rms is not None:
            for k, want in (("ob_mean", r.ob_rms.mean), ("ob_var", r.ob_rms.var), ("ob_count", r.ob_rms.count)):
                assert _same(s[k], want, nan), (where, p, k)
        if r.ret_rms is not None:
            assert _same(s["ret_stat"], [r.ret_rms.mean, r.ret_rms.var, r.ret_rms.count], nan), (where, p, "ret_stat")
            assert _same(s["ret_acc"], r.ret, nan), (where, p, "ret_acc")
        if r.obj_rms is not None:
            for k, want in (("obj_mean", r.obj_rms.mean), ("obj_var", r.obj_rms.var), ("obj_count", r.obj_rms.count)):
                assert _same(s[k], want, nan), (where, p, k)
        if r.obj is not None:
            assert _same(s["obj_acc"], r.obj, nan), (where, p, "obj_acc")


def _outputs(env):
    f = lambda *s: torch.full(s, SENT, device=env.device)
    return f(env.P, env.N, env.O), f(env.P, env.N, env.M), f(env.P, env.N)


def _reset(env, refs, raw_obs):
    obs_out, _, _ = _outputs(env)
    env.reset(raw_obs, obs_out)
    got = obs_out.cpu().numpy()
    for p, r in enumerate(refs):
        assert _same(got[p], r.reset(raw_obs[p])), ("reset", p)
    _check_state(env, refs, where="reset")
    return got


def _step(env, refs, raw_obs, raw_rew, raw_obj, done, nan=False, where=""):
    """One step of every task on the device and on its reference; returns the device outputs (host arrays)."""
    obs_out, obj_out, mask = _outputs(env)
    env.step(raw_obs, raw_rew, raw_obj, done, obs_out, obj_out, mask)
    got = obs_out.cpu().numpy(), obj_out.cpu().numpy(), mask.cpu().numpy()
    with np.errstate(invalid="ignore", over="ignore"):
        for p, r in enumerate(refs):
            o, _, j = r.step(raw_obs[p], raw_rew[p], raw_obj[p], done[p])
            assert _same(got[0][p], o, nan), (where, p, "obs")
            assert _same(got[1][p], j, nan), (where, p, "obj")
            assert _same(got[2][p], 1.0 - done[p]), (where, p, "mask")
    _check_state(env, refs, nan, where)
    return got


def _set_training(env, refs, on):
    for x in [env] + refs:
        x.train() if on else x.eval()


def _make(P, N, O, M, **kw):
    from pgmorl_b200.vec_normalize import DeviceVecNormalize
    return DeviceVecNormalize(P, N, O, M, **kw), [vecnorm_ref.VecNormalize(N, O, **kw) for _ in range(P)]


def _draw(rng, P, N, O, M, obs_scale, obj_scale, p_done=0.2):
    """One step of raw simulator output, a different stream per task."""
    obs = (rng.standard_normal((P, N, O)) + 0.3) * obs_scale
    rew = rng.standard_normal((P, N)) * 3.0
    obj = rng.uniform(-1.0, 5.0, (P, N, M)) * obj_scale
    return obs, rew, obj, rng.uniform(size=(P, N)) < p_done


def _script(env, refs, rng, steps=6, obs_scale=None, obj_scale=None):
    """reset, `steps` steps with dones, VecNormalize.reset after step 2, step 4 under eval()."""
    P, N, O, M = env.P, env.N, env.O, env.M
    obs_scale = rng.uniform(0.1, 30.0, (P, 1, O)) if obs_scale is None else obs_scale
    obj_scale = rng.uniform(0.01, 40.0, (P, 1, M)) if obj_scale is None else obj_scale
    _reset(env, refs, _draw(rng, P, N, O, M, obs_scale, obj_scale)[0])
    for t in range(steps):
        if t == 3:
            _reset(env, refs, _draw(rng, P, N, O, M, obs_scale, obj_scale)[0])
        _set_training(env, refs, t != 4)
        _step(env, refs, *_draw(rng, P, N, O, M, obs_scale, obj_scale), where=t)


SWEEP_N = [1, 2, 7, 8, 9, 15, 16, 17, 31, 32, 33, 64, 100, 127, 128]
SWEEP_OM = [(1, 1), (1, 2), (2, 1), (17, 2), (11, 3), (27, 4), (129, 1), (376, 2)]


@pytest.mark.parametrize("O,M", SWEEP_OM)
@pytest.mark.parametrize("N", SWEEP_N)
def test_shape_sweep(N, O, M):
    """Width 1 (O = 1 or M = 1) from N = 8 on is where numpy's column sum is pairwise; N = 16, 17, 31 ... run the
    8-lane blocks of that sum once, twice and with a remainder; O = 129 spans more features than the CTA has threads."""
    env, refs = _make(3, N, O, M, ob=True, ret=True, obj_rms=True)
    _script(env, refs, np.random.RandomState(1000 * N + 10 * O + M))


CONFIGS = [(ob, ret, obj) for ob in (True, False) for ret, obj in ((False, False), (True, False), (True, True))]


@pytest.mark.parametrize("N,O,M", [(33, 3, 2), (16, 1, 1)])
@pytest.mark.parametrize("ob,ret,obj_rms", CONFIGS)
def test_configurations(ob, ret, obj_rms, N, O, M):
    """Every combination of observation / return / objective normalisation (objective moments need the return's), with
    gamma 0.9, clipob 5, cliprew 2 and epsilon 1e-4; what is switched off passes through or is not tracked."""
    kw = dict(ob=ob, ret=ret, obj_rms=obj_rms, gamma=0.9, clipob=5.0, cliprew=2.0, epsilon=1e-4)
    env, refs = _make(3, N, O, M, **kw)
    _script(env, refs, np.random.RandomState(7 + 2 * N + O))


def _rms(mean, var, count):
    r = vecnorm_ref.RunningMeanStd()
    r.mean, r.var, r.count = mean, var, count
    return r


@pytest.mark.parametrize("M", [1, 3])
def test_loaded_moments_and_snapshot_round_trip(M):
    """load_task of moments that carry 10^9 samples (task 0) and of a scalar-shaped obj_rms (task 1: shape () until its
    first update, as the reference creates it), stepping from there; then snapshot -> load_task into task 2 mid-stream."""
    P, N, O = 3, 20, 4
    env, refs = _make(P, N, O, M, ob=True, ret=True, obj_rms=True)
    rng = np.random.RandomState(40 + M)
    loads = {0: dict(ob_rms=_rms(rng.standard_normal(O), rng.uniform(0.5, 4.0, O), 1e9),
                     ret_rms=_rms(np.float64(0.3), np.float64(2.5), 1e9),
                     obj_rms=_rms(rng.standard_normal(M), rng.uniform(0.5, 4.0, M), 1e9)),
             1: dict(ob_rms=_rms(rng.standard_normal(O), rng.uniform(0.5, 4.0, O), 37.0),
                     ret_rms=_rms(np.float64(-1.25), np.float64(0.75), 37.0),
                     obj_rms=_rms(np.array(0.7), np.array(3.5), 37.0))}
    for p, params in loads.items():
        env.load_task(p, copy.deepcopy(params))
        for k, v in params.items():
            setattr(refs[p], k, copy.deepcopy(v))
    snap = env.snapshot(1)
    assert np.ndim(snap["obj_rms"].mean) == 0 and snap["obj_rms"].mean == 0.7 and snap["obj_rms"].var == 3.5
    _check_state(env, refs, where="loaded")
    obs_scale, obj_scale = rng.uniform(0.5, 5.0, (P, 1, O)), rng.uniform(0.5, 5.0, (P, 1, M))
    for t in range(8):
        if t == 4:
            snap = env.snapshot(0)
            for k in ("ob_rms", "ret_rms", "obj_rms"):
                r = getattr(refs[0], k)
                assert _same(snap[k].mean, r.mean) and _same(snap[k].var, r.var) and snap[k].count == r.count, k
                setattr(refs[2], k, copy.deepcopy(r))
            env.load_task(2, snap)
            _check_state(env, refs, where="round trip")
        _step(env, refs, *_draw(rng, P, N, O, M, obs_scale, obj_scale), where=t)


def test_clipping_engages():
    """Moments loaded with 10^6 samples of N(0, 1) barely move under inputs 15x wider: most observations and objective
    vectors land on +-clip, on both sides (at least 5 % of each output at exactly +-10)."""
    P, N, O, M = 3, 64, 6, 2
    env, refs = _make(P, N, O, M, ob=True, ret=True, obj_rms=True)
    for p in range(P):
        params = dict(ob_rms=_rms(np.zeros(O), np.ones(O), 1e6), ret_rms=_rms(np.float64(0.0), np.float64(1.0), 1e6),
                      obj_rms=_rms(np.zeros(M), np.ones(M), 1e6))
        env.load_task(p, copy.deepcopy(params))
        for k, v in params.items():
            setattr(refs[p], k, v)
    rng = np.random.RandomState(2)
    for t in range(4):
        obs, rew, obj, done = _draw(rng, P, N, O, M, 15.0, 1.0)
        obj = rng.uniform(-40.0, 40.0, (P, N, M))
        got_obs, got_obj, _ = _step(env, refs, obs, rew, obj, done, where=t)
        for got in (got_obs, got_obj):
            assert np.mean(got == 10.0) >= 0.05 and np.mean(got == -10.0) >= 0.05, t


def test_constant_feature_then_jump():
    """A feature (and an objective) constant across every environment for four steps -- its batch variance is exactly 0
    and its running variance decays towards epsilon's floor -- then a jump by 10^3."""
    P, N, O, M = 3, 24, 3, 2
    env, refs = _make(P, N, O, M, ob=True, ret=True, obj_rms=True)
    rng = np.random.RandomState(3)
    for t in range(8):
        obs, rew, obj, done = _draw(rng, P, N, O, M, 2.0, 1.0, p_done=0.0 if t < 4 else 0.2)
        obs[:, :, 0] = 3.25 if t < 4 else 3250.0
        obj[:, :, 1] = 2.0 if t < 4 else 2000.0
        _step(env, refs, obs, rew, obj, done, where=t)


@pytest.mark.parametrize("N", [5, 40])
def test_extreme_magnitudes(N):
    """Features scaled 1e-150 ... 1e150 (squares down to 1e-300 and up to 1e300, still normal FP64) and objectives at
    1e-150, 1 and 1e150."""
    P, O, M = 3, 31, 3
    env, refs = _make(P, N, O, M, ob=True, ret=True, obj_rms=True)
    obs_scale = np.broadcast_to(10.0 ** np.linspace(-150, 150, O), (P, 1, O))
    obj_scale = np.broadcast_to(np.array([1e-150, 1.0, 1e150]), (P, 1, M))
    _script(env, refs, np.random.RandomState(N), steps=5, obs_scale=obs_scale, obj_scale=obj_scale)


def test_nan_and_inf_from_one_environment():
    """NaN, +inf and -inf in one environment of task 1 at one step (observation features, objectives and the reward):
    task 1 follows the reference -- the affected features and objectives turn NaN from then on and stay NaN in the
    outputs (np.clip keeps NaN, it is not clipped to -clip) -- and tasks 0 and 2 are bit-identical to a run without it."""
    P, N, O, M, bad_t = 3, 16, 5, 2, 2
    env, refs = _make(P, N, O, M, ob=True, ret=True, obj_rms=True)
    clean, clean_refs = _make(P, N, O, M, ob=True, ret=True, obj_rms=True)
    rng = np.random.RandomState(4)
    for t in range(6):
        obs, rew, obj, done = _draw(rng, P, N, O, M, 3.0, 2.0)
        clean_out = _step(clean, clean_refs, obs, rew, obj, done, where=("clean", t))
        if t == bad_t:
            obs, rew, obj = obs.copy(), rew.copy(), obj.copy()
            obs[1, 3, 0], obs[1, 3, 1], obs[1, 3, 2] = np.nan, np.inf, -np.inf
            obj[1, 3, 0], obj[1, 3, 1], rew[1, 3] = np.nan, -np.inf, np.inf
        out = _step(env, refs, obs, rew, obj, done, nan=True, where=t)
        if t >= bad_t:
            assert np.isnan(out[0][1][:, :3]).all() and not np.isnan(out[0][1][:, 3:]).any()
            assert np.isnan(out[1][1]).all()
        for a, b in zip(out, clean_out):
            assert np.array_equal(a[[0, 2]], b[[0, 2]]), t
        for p in (0, 2):
            s, c = _state(env, p), _state(clean, p)
            assert all(np.array_equal(s[k], c[k]) for k in s), (t, p)


@pytest.mark.parametrize("N,O,M", [(17, 1, 1), (9, 11, 3)])
def test_rollout_slot_entry_point(N, O, M):
    """pgm_vecnorm_rollout_step_f64 driven through its control word {t, flags} into rollout buffers with padded task
    strides full of a sentinel: t = 0 with flag bit 1 clear writes nothing (buffers and moments untouched); t = 1 ... T
    write the observation into slot t, the reward vector into slot t-1, 1 - done and the bad-transition mask into slot t
    and nothing else, equal to the reference and bit-identical to step mode fed the same stream (the last step frozen)."""
    from pgmorl_b200._lib import check, lib, ptr
    P, T, pad = 3, 5, 37
    vn, refs = _make(P, N, O, M, ob=True, ret=True, obj_rms=True)
    stepper, _ = _make(P, N, O, M, ob=True, ret=True, obj_rms=True)
    cuda = torch.device("cuda")
    size = {"obs": (T + 1) * N * O, "rew": T * N * M, "mask": (T + 1) * N, "bad": (T + 1) * N}
    buf = {k: torch.full((P, n + pad), SENT, device=cuda) for k, n in size.items()}
    want = {k: np.full((P, n + pad), SENT, dtype=np.float32) for k, n in size.items()}
    ctl = torch.zeros(4, dtype=torch.int32, device=cuda)
    rng = np.random.RandomState(N + O)
    obs_scale, obj_scale = rng.uniform(0.1, 30.0, (P, 1, O)), rng.uniform(0.01, 40.0, (P, 1, M))

    def launch(t, flags, obs, rew, obj, done, bad):
        d64 = lambda x: torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64).to(cuda)
        d_obs, d_rew, d_obj = d64(obs), d64(rew), d64(obj)
        d_done = torch.as_tensor(done.astype(np.uint8)).to(cuda)
        d_bad = torch.as_tensor(bad, dtype=torch.float32).to(cuda)
        ctl.copy_(torch.tensor([t, flags, 0, 0], dtype=torch.int32))
        check(lib().pgm_vecnorm_rollout_step_f64(
            ptr(ctl), ptr(d_obs), ptr(d_rew), ptr(d_obj), ptr(d_done), ptr(d_bad),
            ptr(vn.ob_mean), ptr(vn.ob_var), ptr(vn.ob_count), ptr(vn.ret_acc), ptr(vn.ret_stat), ptr(vn.obj_acc),
            ptr(vn.obj_started), ptr(vn.obj_mean), ptr(vn.obj_var), ptr(vn.obj_count),
            ptr(buf["obs"]), buf["obs"].stride(0), ptr(buf["rew"]), buf["rew"].stride(0),
            ptr(buf["mask"]), buf["mask"].stride(0), ptr(buf["bad"]), buf["bad"].stride(0),
            vn.gamma, vn.clipob, vn.cliprew, vn.epsilon, int(vn.training), P, N, O, M,
            C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        torch.cuda.synchronize()

    def check_buffers(where):
        for k in buf:
            assert _same(buf[k].cpu().numpy(), want[k]), (where, k)

    before = {k: v.clone() for k, v in vars(vn).items() if torch.is_tensor(v)}
    obs, rew, obj, done = _draw(rng, P, N, O, M, obs_scale, obj_scale)
    launch(0, 1, obs, rew, obj, done, (rng.uniform(size=(P, N)) < 0.5).astype(np.float32))
    check_buffers("t = 0")
    assert all(torch.equal(v, getattr(vn, k)) for k, v in before.items())
    for t in range(1, T + 1):
        _set_training(vn, refs + [stepper], t < T)
        obs, rew, obj, done = _draw(rng, P, N, O, M, obs_scale, obj_scale)
        bad = (rng.uniform(size=(P, N)) < 0.5).astype(np.float32)
        launch(t, 2 | (t & 1), obs, rew, obj, done, bad)
        s_obs, s_obj, s_mask = _outputs(stepper)
        stepper.step(obs, rew, obj, done, s_obs, s_obj, s_mask)
        for p, r in enumerate(refs):
            o, _, j = r.step(obs[p], rew[p], obj[p], done[p])
            want["obs"][p, t * N * O:(t + 1) * N * O] = o.astype(np.float32).ravel()
            want["rew"][p, (t - 1) * N * M:t * N * M] = j.astype(np.float32).ravel()
            want["mask"][p, t * N:(t + 1) * N] = 1.0 - done[p]
            want["bad"][p, t * N:(t + 1) * N] = bad[p]
        check_buffers(t)
        _check_state(vn, refs, where=t)
        assert torch.equal(buf["obs"][:, t * N * O:(t + 1) * N * O], s_obs.reshape(P, -1))
        assert torch.equal(buf["rew"][:, (t - 1) * N * M:t * N * M], s_obj.reshape(P, -1))
        assert torch.equal(buf["mask"][:, t * N:(t + 1) * N], s_mask)
        for k, v in vars(vn).items():
            if torch.is_tensor(v) and not k.startswith("_"):
                assert torch.equal(v, getattr(stepper, k)), (t, k)


# ---------------------------------------------------------------------------------------------------- one feature, end to end
D1 = NetDims(1, 3, 2)


@pytest.mark.parametrize("T", [50, 300])
def test_k1_forward_at_one_observation_feature(T):
    """K1 at O = 1 (T = 300: >= 1024 rows, several chunks per CTA) against the float64 oracle, gate 2e-5 norm-wise."""
    from pgmorl_b200 import kernels as K
    P, N = 2, 4
    params, traj, eps, _, _, _, ref = make_case(D1, P, T, N, seed=3)
    obs = dev(traj["obs"]).reshape(P, (T + 1) * N, D1.obs)
    value, action, logp = K.policy_forward(dev(params), obs, D1, eps=dev(eps).reshape(1, T * N, D1.act), rows_a=T * N)
    torch.cuda.synchronize()
    for p in range(P):
        assert rel_err(value[p].cpu().numpy().reshape(T + 1, N, -1), ref[p]["value"]) < 2e-5
        assert rel_err(action[p].cpu().numpy().reshape(T, N, -1), ref[p]["action"]) < 2e-5
        assert rel_err(logp[p].cpu().numpy().reshape(T, N), ref[p]["logp"]) < 2e-5


@pytest.mark.parametrize("cluster", [0, 1, 2, 16])
def test_k3_gradient_at_one_observation_feature(cluster):
    """K3's PPO gradient at O = 1 against the float64 oracle: 5e-5 norm-wise (whole vector), losses 2e-5."""
    from pgmorl_b200 import kernels as K
    P, T, N, mb = 2, 64, 4, 256
    cur, pk, _ = _ppo_inputs(D1, P, T, N, seed=11)
    idx = np.random.RandomState(0).permutation(T * N)[:mb]
    g, losses = K.ppo_grad(dev(cur), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]),
                           dev(pk["returns"]), dev(pk["adv"]), dev(idx, torch.int32), D1,
                           hyper=K.PpoHyper(entropy_coef=0.01), cluster=cluster)
    torch.cuda.synchronize()
    for p in range(P):
        net = orc.Net(cur[p].copy(), D1.obs, D1.act, D1.obj)
        gref, lref = orc.ppo_grad(net, pk["obs"][p][:T * N][idx].astype(np.float64), pk["action"][p][idx],
                                  pk["logp"][p][idx], pk["value"][p][:T * N][idx], pk["returns"][p][idx],
                                  pk["adv"][p][idx], ecoef=0.01)
        assert rel_err(g[p].cpu().numpy(), gref) < 5e-5
        assert rel_err(losses[p].cpu().numpy(), np.array(lref)) < 2e-5


def test_fused_rollout_loop_equals_numpy_normalised_loop_at_one_feature(tmp_path):
    """mopg_population_update at one observation feature and 16 environments: normalising on the device (K6) gives the
    same offspring -- parameters, Adam state, objectives and running moments bit for bit -- as normalising on the host
    with the numpy reference (where the observation moments are a pairwise column sum)."""
    import synth_envs
    from pgmorl_b200 import mopg, warm_up
    from pgmorl_b200.sample import Task
    from tests.test_gpu_vecnorm import _HostNormalised, _RawEnv

    class HostNumpy(_HostNormalised):
        def __init__(self, raw, dims, gamma):
            super().__init__(raw, dims, gamma)
            self.vn = vecnorm_ref.VecNormalize(raw.N, raw.O, ob=True, ret=True, obj_rms=True, gamma=gamma)

    d = D1
    args = synth_envs.run_args_2d(str(tmp_path), T=32, N=16)
    mopg.set_env_hooks(make_vec_envs=lambda **kw: HostNumpy(_RawEnv(args.num_processes, d.obs, d.obj), d, args.gamma),
                       gym_make=lambda name: synth_envs.ToyEvalEnv(d), make_raw_vec_envs=False)
    torch.manual_seed(0)
    elites, scals = warm_up.initialize_warm_up_batch(args, "cuda")
    tasks = [Task(e, s) for e, s in zip(elites[:3], scals[:3])]
    host = mopg.mopg_population_update(args, tasks, torch.device("cuda"), 0, 3)
    mopg.set_env_hooks(make_raw_vec_envs=lambda **kw: _RawEnv(args.num_processes, d.obs, d.obj))
    try:
        tasks = [Task(e, s) for e, s in zip(elites[:3], scals[:3])]
        fused = mopg.mopg_population_update(args, tasks, torch.device("cuda"), 0, 3)
    finally:
        mopg.set_env_hooks(make_raw_vec_envs=False)
    for hs, fs in zip(host, fused):
        assert len(hs) == len(fs) == 3
        for a, b in zip(hs, fs):
            assert torch.equal(a.actor_critic.flat, b.actor_critic.flat)
            assert torch.equal(a.agent.optimizer.exp_avg_sq, b.agent.optimizer.exp_avg_sq)
            assert np.array_equal(a.objs, b.objs)
            for key in ("ob_rms", "ret_rms", "obj_rms"):
                assert np.array_equal(a.env_params[key].mean, b.env_params[key].mean), key
                assert np.array_equal(a.env_params[key].var, b.env_params[key].var), key
                assert a.env_params[key].count == b.env_params[key].count
