"""K1 / K3 at every network shape, kernel family and PPO setting the C ABI accepts, against the float64 oracle.

The named reference shapes (Walker2d / HalfCheetah, Hopper-v2 / -v3, Ant, Swimmer, Humanoid) and test-only shapes at the
edges of the K3 planner: (16,16,2) runs four head passes in the small-population kernel, (48,16,16) is the upper edge of
that kernel, (45,16,3) switches between it and the generic double-buffered kernel with the minibatch split, (60,6,2) and
(64,4,4) only fit the generic double-buffered kernel, (33,17,2) takes the generic "big" kernel at every cluster size.
Tolerances as in test_gpu_kernels.py (norm-wise, max|a-b| <= tol * max|b|), written beside each assert.
"""
import re

import numpy as np
import pytest
import torch

import ppo_options_ref as ref
from oracle import mopg_oracle as orc
from pgmorl_b200 import synthetic
from pgmorl_b200.layout import param_layout
from tests.helpers import rel_err
from tests.test_gpu_kernels import DIMS, TAIL0, _ppo_inputs, dev

pytestmark = pytest.mark.gpu

# The planner's choice per case: (name, P, mb, cluster) -> instantiation, VU (unclipped value loss) filled in per run.
# k3_ppo_fast_kernel<C, TM, TAIL, VU>, k3_ppo_kernel<C, TM, KG1, NA, DB, VU>, k3_tc_kernel<O, A, M, RS, VU>,
# k3_tcw_kernel<O, A, M, RS, VU>. Clusters of two CTAs run the fast kernel with tail 0 (tails 1-6 need two CTAs per half);
# larger clusters run the default tail 5, and tail 0 when the TAIL0 flag asks for it.
ROUTES = [
    # small-population FFMA kernel
    ("walker", 2, 256, 2, "k3_ppo_fast_kernel<2,4,0,{vu}>"),
    ("ant", 2, 256, 2, "k3_ppo_fast_kernel<2,2,0,{vu}>"),           # TM = 4 needs 237 664 B: falls back to TM = 2
    ("s16_16_2", 2, 256, 2, "k3_ppo_fast_kernel<2,2,0,{vu}>"),      # 252 448 B at TM = 4
    ("hopper2", 2, 64, 4, "k3_ppo_fast_kernel<4,2,5,{vu}>"),
    ("ant", 2, 256, 4, "k3_ppo_fast_kernel<4,4,5,{vu}>"),
    ("swimmer", 2, 64, 8, "k3_ppo_fast_kernel<8,2,5,{vu}>"),
    ("ant", 2, 256, 8, "k3_ppo_fast_kernel<8,4,5,{vu}>"),
    ("walker", 2, 256, 16, "k3_ppo_fast_kernel<16,2,5,{vu}>"),
    ("s16_16_2", 2, 256, 16, "k3_ppo_fast_kernel<16,2,5,{vu}>"),
    ("s48_16_16", 2, 256, 16, "k3_ppo_fast_kernel<16,2,5,{vu}>"),
    ("s45_16_3", 2, 256, 16, "k3_ppo_fast_kernel<16,2,5,{vu}>"),
    ("hopper2", 2, 512, 16, "k3_ppo_fast_kernel<16,4,5,{vu}>"),
    ("hopper2", 2, 64, 4 | TAIL0, "k3_ppo_fast_kernel<4,2,0,{vu}>"),
    ("ant", 2, 256, 4 | TAIL0, "k3_ppo_fast_kernel<4,4,0,{vu}>"),
    ("swimmer", 2, 64, 8 | TAIL0, "k3_ppo_fast_kernel<8,2,0,{vu}>"),
    ("ant", 2, 256, 8 | TAIL0, "k3_ppo_fast_kernel<8,4,0,{vu}>"),
    ("walker", 2, 256, 16 | TAIL0, "k3_ppo_fast_kernel<16,2,0,{vu}>"),
    ("hopper2", 2, 512, 16 | TAIL0, "k3_ppo_fast_kernel<16,4,0,{vu}>"),
    # generic double-buffered kernel
    ("s60_6_2", 2, 32, 2, "k3_ppo_kernel<2,2,1,1,true,{vu}>"),
    ("s48_16_16", 2, 32, 2, "k3_ppo_kernel<2,2,1,1,true,{vu}>"),    # the fast kernel at TM = 2 needs more than 227 KB
    ("s60_6_2", 2, 256, 2, "k3_ppo_kernel<2,4,1,1,true,{vu}>"),
    ("s64_4_4", 2, 64, 4, "k3_ppo_kernel<4,2,1,1,true,{vu}>"),
    ("s60_6_2", 2, 256, 4, "k3_ppo_kernel<4,4,1,1,true,{vu}>"),
    ("s60_6_2", 2, 128, 8, "k3_ppo_kernel<8,2,1,1,true,{vu}>"),
    ("s45_16_3", 2, 256, 8, "k3_ppo_kernel<8,4,1,1,true,{vu}>"),
    ("s64_4_4", 2, 256, 16, "k3_ppo_kernel<16,2,1,1,true,{vu}>"),
    ("s60_6_2", 2, 512, 16, "k3_ppo_kernel<16,4,1,1,true,{vu}>"),
    # generic kernel, both halves in one CTA
    ("swimmer", 2, 32, 1, "k3_ppo_kernel<1,2,1,1,false,{vu}>"),
    ("ant", 2, 256, 1, "k3_ppo_kernel<1,4,1,1,false,{vu}>"),
    # generic "big" kernel (O > 64, A > 16 or M > 16)
    ("s33_17_2", 2, 256, 1, "k3_ppo_kernel<1,2,6,2,false,{vu}>"),
    ("s33_17_2", 2, 256, 2, "k3_ppo_kernel<2,2,6,2,false,{vu}>"),
    ("s33_17_2", 2, 256, 4, "k3_ppo_kernel<4,2,6,2,false,{vu}>"),
    ("humanoid", 2, 256, 8, "k3_ppo_kernel<8,2,6,2,false,{vu}>"),
    ("s33_17_2", 2, 256, 16, "k3_ppo_kernel<16,2,6,2,false,{vu}>"),
    # tensor-core kernels
    ("walker", 2, 256, 32, "k3_tc_kernel<17,6,2,1,{vu}>"),
    ("walker", 2, 256, 64, "k3_tc_kernel<17,6,2,2,{vu}>"),
    ("hopper3", 2, 256, 32, "k3_tc_kernel<11,3,3,1,{vu}>"),
    ("hopper3", 2, 256, 64, "k3_tc_kernel<11,3,3,2,{vu}>"),
    ("humanoid", 2, 256, 32, "k3_tcw_kernel<376,17,2,1,{vu}>"),
    ("humanoid", 2, 256, 64, "k3_tcw_kernel<376,17,2,2,{vu}>"),
    ("humanoid", 2, 256, 128, "k3_tcw_kernel<376,17,2,4,{vu}>"),
]

# Every instantiation k3_launch / k3_launch_c can reach with the default step tail or tail 0, written out independently
# of ROUTES: a case that is the only one to reach an instantiation cannot be dropped without this list noticing. Tails
# 1-4 and 6 are bit-identical to tail 0 (test_gpu_kernels.py::test_k3_step_tails_bit_identical).
ALL_K3 = sorted(
    [f"k3_ppo_fast_kernel<{c},{tm},0,{{vu}}>" for c in (2, 4, 8, 16) for tm in (2, 4)] +
    [f"k3_ppo_fast_kernel<{c},{tm},5,{{vu}}>" for c in (4, 8, 16) for tm in (2, 4)] +
    [f"k3_ppo_kernel<{c},{tm},1,1,true,{{vu}}>" for c in (2, 4, 8, 16) for tm in (2, 4)] +
    [f"k3_ppo_kernel<1,{tm},1,1,false,{{vu}}>" for tm in (2, 4)] +
    [f"k3_ppo_kernel<{c},2,6,2,false,{{vu}}>" for c in (1, 2, 4, 8, 16)] +
    [f"k3_tc_kernel<{s},{rs},{{vu}}>" for s in ("17,6,2", "11,3,3") for rs in (1, 2)] +
    [f"k3_tcw_kernel<376,17,2,{rs},{{vu}}>" for rs in (1, 2, 4)])

VU = {False: "false", True: "true"}


def _grad_case(name, P, mb, seed=41):
    """Inputs of one PPO gradient: S = 4 * mb rows (T = mb, N = 4), idx = mb distinct rows. Observations ~ N(0, 1) and the
    initial parameters keep every tensor-core operand inside its range (pgmorl_b200.h: |obs| < 65 504, |parameter| <
    255.9, |backward signal| < 16)."""
    d = DIMS[name]
    Pd = min(P, 3)                                        # distinct tasks, tiled with per-task parameter offsets
    cur, pk, _ = _ppo_inputs(d, Pd, mb, 4, seed)
    if P > Pd:
        reps = (P + Pd - 1) // Pd
        cur = np.tile(cur, (reps, 1))[:P] + np.random.RandomState(seed).randn(P, d.n_par) * 1e-3
        pk = {k: np.tile(v, (reps,) + (1,) * (v.ndim - 1))[:P] for k, v in pk.items()}
    idx = np.random.RandomState(seed + 2).permutation(4 * mb)[:mb]
    return d, cur, pk, idx


def _run_grad(d, cur, pk, idx, cluster, vu, hyper):
    from pgmorl_b200 import kernels as K
    g, losses = K.ppo_grad(dev(cur), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]), dev(pk["value"]),
                           dev(pk["returns"]), dev(pk["adv"]), dev(idx, torch.int32), d, hyper=hyper, cluster=cluster,
                           clipped_value_loss=not vu)
    torch.cuda.synchronize()
    return g.cpu().numpy(), losses.cpu().numpy()


def _ref_grad(d, cur, pk, idx, p, vu, ecoef):
    S = pk["action"].shape[1]
    rows = lambda a: a[p][:S][idx].astype(np.float64)
    net = orc.Net(cur[p].astype(np.float64).copy(), d.obs, d.act, d.obj)
    return ref.ppo_grad_np(net, rows(pk["obs"]), rows(pk["action"]), rows(pk["logp"]), rows(pk["value"]),
                           rows(pk["returns"]), rows(pk["adv"]), ecoef=ecoef, clipped_value_loss=not vu)


def _kernel_names(prof):
    names = set()
    for e in prof.events():
        m = re.search(r"(k[13]_\w+_kernel<[^()]*>)", e.name.replace(" ", ""))
        if m:
            names.add(m.group(1))
    return names


def test_route_coverage():
    """Every case of ROUTES runs the instantiation the table names (both value losses), the cases together reach every
    K3 instantiation of ALL_K3, and K1's FFMA kernel for whole trajectories runs at >= 1024 rows of a shape without a
    tensor-core forward."""
    from torch.profiler import ProfilerActivity, profile

    from pgmorl_b200 import kernels as K
    hyper = K.PpoHyper(entropy_coef=0.01)
    seen, wrong = set(), []
    for name, P, mb, cluster, kern in ROUTES:
        d, cur, pk, idx = _grad_case(name, P, mb)
        for vu in (False, True):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                _run_grad(d, cur, pk, idx, cluster, vu, hyper)
            names = {n for n in _kernel_names(prof) if n.startswith("k3_") and "pack" not in n}
            assert names, f"the profiler reported no K3 kernel for {name} cluster {cluster}"
            want = kern.format(vu=VU[vu])
            if names != {want}:
                wrong.append((name, P, mb, cluster, vu, want, sorted(names)))
            seen |= names
    assert not wrong, wrong
    expect = {k.format(vu=v) for k in ALL_K3 for v in VU.values()}
    assert seen == expect, (sorted(expect - seen), sorted(seen - expect))
    # K1: 8 tasks x 2049 x 4 rows of Ant dims, several 264-row chunks per CTA
    d = DIMS["ant"]
    obs = torch.randn(8, 2049 * 4, d.obs, device="cuda")
    params = dev(np.stack([synthetic.init_policy_flat(d, seed=p).numpy() for p in range(8)]))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        K.policy_forward(params, obs, d, eps=torch.randn(1, 2048 * 4, d.act, device="cuda"), rows_a=2048 * 4)
        torch.cuda.synchronize()
    assert "k1_forward_kernel<4,false>" in _kernel_names(prof)


# Per-tensor gate on the raw gradient, for every case of ROUTES and both value losses. The whole-vector gate (5e-5 of the
# largest element, the critic head bias) would let an actor-tensor error of ~8e-4 of that tensor's own scale through.
# Worst per-tensor error measured on one B200 (1000 W), over every case and both value losses: 3.4e-6 on the FP32 FFMA
# kernels (fast: actor.2.bias of (45,16,3) at C = 16; generic DB 2.6e-6, one CTA 1.6e-6, big 3.3e-6), 1.9e-6 on the
# tensor-core kernel and 7.0e-6 on the wide tensor-core kernel (Humanoid, logstd). Gates about 5x above that:
PER_TENSOR_TOL = 2e-5
PER_TENSOR_TOL_TCW = 4e-5
KERNEL = {r[:4]: r[4] for r in ROUTES}


@pytest.mark.parametrize("vu", [False, True])
@pytest.mark.parametrize("name,P,mb,cluster", [r[:4] for r in ROUTES])
def test_k3_gradient_per_tensor(name, P, mb, cluster, vu):
    from pgmorl_b200 import kernels as K
    d, cur, pk, idx = _grad_case(name, P, mb)
    g, losses = _run_grad(d, cur, pk, idx, cluster, vu, K.PpoHyper(entropy_coef=0.01))
    layout, _ = param_layout(d)
    for p in range(P):
        gref, lref = _ref_grad(d, cur, pk, idx, p, vu, 0.01)
        assert rel_err(g[p], gref) < 5e-5                         # whole vector: 5e-5
        assert rel_err(losses[p], np.array(lref)) < 1e-4
        for tname, (off, shape) in layout.items():
            n = int(np.prod(shape))
            err = rel_err(g[p][off:off + n], gref[off:off + n])
            assert err < (PER_TENSOR_TOL_TCW if KERNEL[name, P, mb, cluster].startswith("k3_tcw") else PER_TENSOR_TOL), \
                (tname, err)


# Acceptance sweep: every shape of the table at every cluster size, small and large populations, three minibatch sizes
# (mb = 32 at two CTAs per task sends (48,16,16) and (45,16,3) from the fast kernel, which no longer fits at TM = 2, to
# the generic double-buffered one). Nothing inside the documented range is refused for shared memory, and every plan
# computes the oracle's gradient.
SWEEP_SHAPES = ["hopper2", "ant", "swimmer", "s16_16_2", "s48_16_16", "s45_16_3", "s60_6_2", "s64_4_4", "s33_17_2"]


@pytest.mark.parametrize("name", SWEEP_SHAPES)
def test_k3_plan_acceptance_sweep(name):
    from pgmorl_b200 import kernels as K
    hyper = K.PpoHyper(entropy_coef=0.01)
    for P in (2, 40):
        for mb in (32, 64, 256):
            d, cur, pk, idx = _grad_case(name, P, mb)
            refs = {p: _ref_grad(d, cur, pk, idx, p, False, 0.01) for p in sorted({0, 1, P // 2, P - 1})}
            for cluster in (0, 1, 2, 4, 8, 16):
                g, losses = _run_grad(d, cur, pk, idx, cluster, False, hyper)
                for p, (gref, lref) in refs.items():
                    assert rel_err(g[p], gref) < 5e-5, (P, mb, cluster, p)        # whole vector: 5e-5
                    assert rel_err(losses[p], np.array(lref)) < 1e-4, (P, mb, cluster, p)


def test_k3_cluster_1_refusal_names_shared_memory():
    """cluster = 1 keeps both halves in one CTA: at Humanoid dims that needs 317 920 B, more than the 227 KB a block may
    have, and no other family runs one CTA per task. The refusal says so (cluster >= 2 runs the shape, ROUTES)."""
    from pgmorl_b200 import _lib
    from pgmorl_b200 import kernels as K
    d, cur, pk, idx = _grad_case("humanoid", 1, 64)
    with pytest.raises(_lib.PgmError, match="317920 B of shared memory"):
        _run_grad(d, cur, pk, idx, 1, False, K.PpoHyper())


# One case per kernel family, non-default hyperparameters: (name, P, T, N, B, cluster) with E = 2 epochs.
HYPER_CASES = [("walker", 2, 64, 4, 2, 16),          # fast, C = 16
               ("ant", 2, 64, 4, 2, 8),              # fast, C = 8
               ("s45_16_3", 2, 128, 4, 2, 8),        # generic double-buffered (mb = 256, TM = 4)
               ("walker", 2, 64, 4, 2, 1),           # generic, one CTA
               ("humanoid", 2, 64, 8, 2, 8),         # generic big
               ("walker", 2, 64, 4, 2, 32), ("walker", 2, 64, 4, 2, 64),
               ("humanoid", 2, 64, 8, 2, 32), ("humanoid", 2, 64, 8, 2, 64), ("humanoid", 2, 64, 8, 2, 128)]


@pytest.mark.parametrize("clip_mode", ["never", "some"])
@pytest.mark.parametrize("name,P,T,N,B,cluster", HYPER_CASES)
def test_k3_update_hyperparameters(name, P, T, N, B, cluster, clip_mode):
    """clip 0.1, value coefficient 1.0, entropy 0.01, betas (0.8, 0.99), eps 1e-6, and max_grad_norm either 1e3 (the
    clip never engages: coef = 1) or between the smallest and largest gradient norm of the oracle's own chain (both
    branches of coef = min(1, max_norm / (norm + 1e-6)) run in one launch). Inputs as in test_gpu_kernels (observations
    ~ N(0, 1), initial parameters): inside the tensor-core operand ranges."""
    from pgmorl_b200 import kernels as K
    d = DIMS[name]
    cur, pk, perm = _ppo_inputs(d, P, T, N, seed=43)
    kw = dict(clip=0.1, vcoef=1.0, ecoef=0.01, adam_eps=1e-6, beta1=0.8, beta2=0.99)
    rng = np.random.RandomState(4)
    m0, v0 = rng.randn(P, d.n_par) * 1e-3, rng.rand(P, d.n_par) * 1e-5
    step0, lr = np.array([0, 7][:P], dtype=np.int32), np.array([3e-4, 2.5e-4][:P])
    f64 = lambda t: dev(t).cpu().numpy().astype(np.float64)      # the kernel sees float32-rounded state

    def oracle(p, mgn, norms=None):
        flat, m, v = f64(cur[p]), f64(m0[p]), f64(v0[p])
        step, lref = orc.ppo_update(flat, m, v, int(step0[p]), lr[p], (d.obs, d.act, d.obj),
                                    pk["obs"][p].reshape(T + 1, N, d.obs).astype(np.float64),
                                    pk["action"][p].reshape(T, N, -1), pk["logp"][p].reshape(T, N),
                                    pk["value"][p].reshape(T + 1, N, -1), pk["returns"][p].reshape(T, N, -1),
                                    pk["adv"][p].reshape(T, N), perm, B, max_grad_norm=mgn, norms=norms, **kw)
        return flat, m, v, step, lref

    if clip_mode == "never":
        mgn = 1e3
    else:
        norms = []
        for p in range(P):
            oracle(p, 1e3, norms)
        mgn = float(np.median(norms))
    norms = []
    refs = [oracle(p, mgn, norms) for p in range(P)]
    clipped = [n + 1e-6 > mgn for n in norms]
    if clip_mode == "never":
        assert not any(clipped)
    else:                                               # not vacuous: some steps clip, others do not
        assert any(clipped) and not all(clipped)
    hyper = K.PpoHyper(clip_param=0.1, value_loss_coef=1.0, entropy_coef=0.01, max_grad_norm=mgn, beta1=0.8, beta2=0.99,
                       adam_eps=1e-6)
    gp, gm, gv, gstep = dev(cur), dev(m0), dev(v0), dev(step0, torch.int32)
    losses = K.ppo_update(gp, gm, gv, gstep, dev(lr, torch.float64), dev(pk["obs"]), dev(pk["action"]), dev(pk["logp"]),
                          dev(pk["value"]), dev(pk["returns"]), dev(pk["adv"]), dev(perm[None], torch.int32), B, d,
                          hyper=hyper, cluster=cluster)
    torch.cuda.synchronize()
    for p, (flat, m, v, step, lref) in enumerate(refs):
        assert int(gstep[p]) == step
        assert rel_err(gp[p].cpu().numpy(), flat) < 1e-5          # parameters (gate 1e-4)
        assert rel_err(gm[p].cpu().numpy(), m) < 1e-4            # Adam first moment
        assert rel_err(gv[p].cpu().numpy(), v) < 1e-4            # Adam second moment
        assert rel_err(losses[p].cpu().numpy(), np.array(lref)) < 1e-4


@pytest.mark.parametrize("name,cluster,gamma", [("hopper2", 0, 0.995), ("hopper2", 16, 0.995), ("ant", 0, 0.995),
                                                ("ant", 16, 0.995), ("swimmer", 0, 0.995), ("swimmer", 16, 0.995),
                                                ("ant", 0, 0.99)])     # 0.99: the Humanoid script's discount
def test_population_iteration_other_reference_shapes(name, cluster, gamma):
    """Whole MOPG iterations (K1 -> K2 -> K3) through PopulationMOPG at the reference's Hopper-v2, Ant and Swimmer shapes,
    against orc.mopg_iteration per task. 257 x 4 rows per task: K1's FFMA forward over several chunks. Tolerances of
    test_population_iterations_match_reference_goldens: 1e-4 norm-wise, Adam moments and losses 1e-3."""
    from pgmorl_b200.population_state import PopulationMOPG
    d = DIMS[name]
    P, T, N, E, B = 3, 256, 4, 2, 4
    rng = np.random.RandomState(9)
    init = np.stack([synthetic.init_policy_flat(d, seed=200 + p).numpy().astype(np.float64) for p in range(P)])
    init[:, -d.act:] = rng.uniform(-0.5, 0.3, (P, d.act))
    weights, obj_var = rng.dirichlet(np.ones(d.obj), P), rng.uniform(0.5, 2.0, (P, d.obj))
    lr = 3e-4
    pop = PopulationMOPG(d, P, T, N, ppo_epoch=E, num_mini_batch=B, gamma=gamma, gae_lambda=0.95, cluster=cluster)
    for p in range(P):
        pop.load_task(p, init[p], weights=weights[p], obj_var=obj_var[p])
    pop.set_lr(lr)
    traj = synthetic.make_trajectories(P, T, N, d, seed=21, p_done=0.02)
    eps, perm = synthetic.host_rng_streams(3, T, N, d.act, E)
    eps = eps.to(torch.float32)
    losses = pop.step_from_host(traj["obs"], traj["rewards"], traj["masks"], traj["bad_masks"], eps,
                                perm.to(torch.int32))
    for p in range(P):
        flat = dev(init[p]).cpu().numpy().astype(np.float64)
        m, v = np.zeros_like(flat), np.zeros_like(flat)
        out = orc.mopg_iteration(flat, m, v, 0, lr, (d.obs, d.act, d.obj), {k: t[p].numpy() for k, t in traj.items()},
                                 eps.double().numpy(), perm.numpy(), weights[p], obj_var[p], gamma=gamma, lam=0.95,
                                 num_mini_batch=B)
        pf, pm, pv, step = pop.task_state(p)
        assert step == out["step"] == E * B
        assert rel_err(pop.value[p].cpu().numpy().reshape(T + 1, N, -1), out["value"]) < 1e-4
        assert rel_err(pop.action[p].cpu().numpy().reshape(T, N, -1), out["action"]) < 1e-4
        assert rel_err(pop.returns[p].cpu().numpy(), out["returns"]) < 1e-4
        assert rel_err(pop.adv[p].cpu().numpy(), out["adv"]) < 1e-4
        assert rel_err(pf, flat) < 1e-4
        assert rel_err(pm, m) < 1e-3 and rel_err(pv, v) < 1e-3
        assert rel_err(losses[p], out["losses"]) < 1e-3
