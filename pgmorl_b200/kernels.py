"""Torch-tensor level launchers over the C ABI. PyTorch only owns memory and streams here;
all arithmetic runs in the hand-written sm_100a kernels of libpgmorl_b200.so."""
import ctypes as C

import torch

from ._lib import PpoHyper, check, lib, ptr
from ._nvtx import rng as _nvtx
from .layout import NetDims

ACT_SAMPLE, ACT_DETERMINISTIC, ACT_EVALUATE = 0, 1, 2
RET_GAE, RET_PROPER_TIME_LIMITS = 1, 2        # mode bits of pgm_returns_adv_f32
PPO_VALUE_UNCLIPPED = 0x10000                 # flag OR-ed into K3's `cluster`: value loss without the clip


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t, name):
    if t is None:
        return None
    if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
        raise ValueError(f"{name}: expected a contiguous float32 CUDA tensor, got {t.dtype} {t.device} "
                         f"contiguous={t.is_contiguous()}")
    return t


def policy_forward(params, obs, dims: NetDims, eps=None, action=None, mode=ACT_SAMPLE, rows_a=None,
                   out=None, entropy=None):
    """K1. params [P,n_par]; obs [P,rows_v,O]; eps [P or 1,rows_a,A] (SAMPLE);
    action [P,rows_a,A] given for EVALUATE. Returns (value [P,rows_v,M], action, logp [P,rows_a]).
    Categorical head (dims.categorical, A = n): eps holds Exponential(1) draws, actions are [P,rows_a,1] category indices
    as float32, and `entropy` (float32 [P,rows_a], optional) receives each row's entropy."""
    _f32c(params, "params"); _f32c(obs, "obs"); _f32c(eps, "eps"); _f32c(entropy, "entropy")
    P, rows_v, O = obs.shape
    assert O == dims.obs and params.shape == (P, dims.n_par)
    if rows_a is None:
        rows_a = rows_v
    dev = obs.device
    if out is not None:
        value, act_out, logp = out
    else:
        value = torch.empty(P, rows_v, dims.obj, device=dev, dtype=torch.float32)
        act_out = torch.empty(P, rows_a, dims.act_cols, device=dev, dtype=torch.float32) if mode != ACT_EVALUATE else None
        logp = torch.empty(P, rows_a, device=dev, dtype=torch.float32)
    if mode == ACT_EVALUATE:
        act_out = _f32c(action, "action")
        assert act_out.shape == (P, rows_a, dims.act_cols)
    if entropy is not None:
        assert entropy.shape == (P, rows_a)
    eps_shared = 0
    if mode == ACT_SAMPLE and rows_a > 0:
        assert eps is not None and eps.shape[1:] == (rows_a, dims.act) and eps.shape[0] in (1, P)
        eps_shared = int(eps.shape[0] == 1 and P > 1)
    check(lib().pgm_policy_forward_x_f32(ptr(params), ptr(obs), ptr(eps), eps_shared, ptr(act_out), ptr(value),
                                         ptr(logp), ptr(entropy), mode, P, rows_v, rows_a, dims.obs, dims.act, dims.obj,
                                         dims.hidden, dims.dist, _stream()))
    return value, act_out, logp


def policy_step(params, ctl, obs_stage, eps, obs_buf, value_buf, action_buf, logp_buf, act_out, N, dims: NetDims):
    """K1 per-step mode (pgm_policy_step_f32): value / action / log-prob of every task's N current observations written
    into time slot ctl[0] of the rollout buffers; ctl = int32 [2] on the device {t, sample flag}. eps [P or 1,N,A] (A = n
    Exponential(1) draws for a Categorical head, whose action_buf / act_out have one column)."""
    P = params.shape[0]
    assert ctl.is_cuda and ctl.dtype == torch.int32 and ctl.numel() >= 2
    for n, t in (("params", params), ("obs_stage", obs_stage), ("eps", eps), ("obs_buf", obs_buf), ("value_buf", value_buf),
                 ("action_buf", action_buf), ("logp_buf", logp_buf), ("act_out", act_out)):
        _f32c(t, n)
    assert eps.shape[-2:] == (N, dims.act) and eps.shape[0] in (1, P)
    check(lib().pgm_policy_step_x_f32(ptr(params), ptr(ctl), ptr(obs_stage), ptr(eps), int(eps.shape[0] == 1 and P > 1),
                                      ptr(obs_buf), obs_buf.stride(0), ptr(value_buf), value_buf.stride(0),
                                      ptr(action_buf), action_buf.stride(0), ptr(logp_buf), logp_buf.stride(0), ptr(act_out),
                                      P, N, dims.obs, dims.act, dims.obj, dims.hidden, dims.dist, _stream()))


def gae_adv(rewards, value, masks, bad_masks, gamma, lam, weights=None, obj_var=None, out=None):
    """K2. rewards [P,T,N,M]; value [P,T+1,N,M]; masks/bad_masks [P,T+1,N]; weights/obj_var [P,M].
    Returns (returns [P,T,N,M], adv [P,T,N] or None)."""
    for n, t in (("rewards", rewards), ("value", value), ("masks", masks), ("bad_masks", bad_masks),
                 ("weights", weights), ("obj_var", obj_var)):
        _f32c(t, n)
    P, T, N, M = rewards.shape
    assert value.shape == (P, T + 1, N, M) and masks.shape == (P, T + 1, N) and bad_masks.shape == (P, T + 1, N)
    if out is not None:
        returns, adv = out
    else:
        returns = torch.empty_like(rewards)
        adv = torch.empty(P, T, N, device=rewards.device, dtype=torch.float32) if weights is not None else None
    check(lib().pgm_gae_adv_f32(ptr(rewards), ptr(value), ptr(masks), ptr(bad_masks), ptr(weights), ptr(obj_var),
                                float(gamma), float(lam), ptr(returns), ptr(adv), P, T, N, M, _stream()))
    return returns, adv


def returns_adv(rewards, value, masks, bad_masks, gamma, lam, use_gae=True, use_proper_time_limits=True, weights=None,
                obj_var=None, boot=None, out=None):
    """K2 with the branch of RolloutStorage.compute_returns chosen by use_gae / use_proper_time_limits (storage.py:77-116).
    Shapes as gae_adv; boot [P,N,M] = bootstrap value of the n-step branches (None: value row T; the GAE branches always
    bootstrap from value row T). Returns (returns [P,T,N,M], adv [P,T,N] or None); adv = normalised scalarisation of
    returns - value[:T]."""
    for n, t in (("rewards", rewards), ("value", value), ("masks", masks), ("bad_masks", bad_masks),
                 ("weights", weights), ("obj_var", obj_var), ("boot", boot)):
        _f32c(t, n)
    P, T, N, M = rewards.shape
    assert value.shape == (P, T + 1, N, M) and masks.shape == (P, T + 1, N) and bad_masks.shape == (P, T + 1, N)
    assert boot is None or boot.shape == (P, N, M)
    if out is not None:
        returns, adv = out
    else:
        returns = torch.empty_like(rewards)
        adv = torch.empty(P, T, N, device=rewards.device, dtype=torch.float32) if weights is not None else None
    mode = (RET_GAE if use_gae else 0) | (RET_PROPER_TIME_LIMITS if use_proper_time_limits else 0)
    check(lib().pgm_returns_adv_f32(ptr(rewards), ptr(value), ptr(boot), ptr(masks), ptr(bad_masks), ptr(weights),
                                    ptr(obj_var), float(gamma), float(lam), mode, ptr(returns), ptr(adv), P, T, N, M,
                                    _stream()))
    return returns, adv


def ppo_workspace(P, S, dims: NetDims, device, cluster=0):
    n = lib().pgm_ppo_workspace_bytes_x(P, S, dims.obs, dims.act, dims.obj, cluster, dims.hidden, dims.dist)
    return torch.empty(n + 256, dtype=torch.uint8, device=device)


def _aligned(ws):
    off = (-ws.data_ptr()) % 256
    return C.c_void_p(ws.data_ptr() + off), ws.numel() - off


def ppo_update(params, adam_m, adam_v, adam_step, lr, obs, action, logp_old, value_old, returns, adv, perm,
               num_mini_batch, dims: NetDims, hyper: PpoHyper = None, workspace=None, cluster=0, losses=None,
               clipped_value_loss=True):
    """K3. In place on params/adam_m/adam_v [P,n_par] and adam_step [P] int32.
    obs [P,>=S,O] / value_old [P,>=S,M] may carry the extra T+1 slot (only the first S rows are read);
    action [P,S,A] ([P,S,1] category indices as float32 for a Categorical head); logp_old, adv [P,S]; returns [P,S,M];
    perm int32 [P or 1,E,S]; lr float64 [P].
    clipped_value_loss=False: value loss 0.5 * mean((V - R)^2) (PPO(use_clipped_value_loss=False), ppo.py:86-94).
    Returns losses [P,3] = (value_loss, action_loss, entropy) averaged over the E*B updates."""
    P, S, A = action.shape
    assert A == dims.act_cols
    for n, t in (("params", params), ("adam_m", adam_m), ("adam_v", adam_v), ("obs", obs), ("action", action),
                 ("logp_old", logp_old), ("value_old", value_old), ("returns", returns), ("adv", adv)):
        _f32c(t, n)
    assert adam_step.dtype == torch.int32 and lr.dtype == torch.float64 and perm.dtype == torch.int32
    assert perm.is_cuda and perm.is_contiguous() and perm.shape[-1] == S and perm.shape[0] in (1, P)
    assert obs.shape[0] == P and obs.shape[1] >= S and obs.shape[2] == dims.obs
    assert value_old.shape[0] == P and value_old.shape[1] >= S and value_old.shape[2] == dims.obj
    hyper = hyper or PpoHyper()
    if workspace is None:
        workspace = ppo_workspace(P, S, dims, params.device, cluster)
    wp, wn = _aligned(workspace)
    if losses is None:
        losses = torch.empty(P, 3, device=params.device, dtype=torch.float32)
    E = perm.shape[1]
    check(lib().pgm_ppo_update_x_f32(
        ptr(params), ptr(adam_m), ptr(adam_v), ptr(adam_step), ptr(lr), ptr(obs), obs.stride(0), ptr(action),
        ptr(logp_old), ptr(value_old), value_old.stride(0), ptr(returns), ptr(adv), ptr(perm),
        int(perm.shape[0] == 1 and P > 1), E, num_mini_batch, C.byref(hyper), ptr(losses), wp, wn,
        cluster if clipped_value_loss else cluster | PPO_VALUE_UNCLIPPED, P, S, dims.obs, dims.act, dims.obj, dims.hidden,
        dims.dist, _stream()))
    return losses


def ppo_grad(params, obs, action, logp_old, value_old, returns, adv, idx, dims: NetDims, hyper=None,
             cluster=0, clipped_value_loss=True):
    """Verification aid: gradient [P,n_par] (before the grad-norm clip) and losses [P,3] of one minibatch `idx`
    (int32 [mb]); clipped_value_loss as in ppo_update."""
    P, S, A = action.shape
    assert A == dims.act_cols
    hyper = hyper or PpoHyper()
    ws = ppo_workspace(P, S, dims, params.device, cluster)
    wp, wn = _aligned(ws)
    grad = torch.zeros(P, dims.n_par, device=params.device, dtype=torch.float32)
    losses = torch.empty(P, 3, device=params.device, dtype=torch.float32)
    check(lib().pgm_ppo_grad_x_f32(ptr(params), ptr(obs), obs.stride(0), ptr(action), ptr(logp_old), ptr(value_old),
                                   value_old.stride(0), ptr(returns), ptr(adv), ptr(idx), idx.numel(),
                                   C.byref(hyper), ptr(grad), ptr(losses), wp, wn,
                                   cluster if clipped_value_loss else cluster | PPO_VALUE_UNCLIPPED, P, S, dims.obs, dims.act,
                                   dims.obj, dims.hidden, dims.dist, _stream()))
    return grad, losses


# ---------------------------------------------------------------------------------------------
# K5: Pareto filter, hypervolume / sparsity, greedy pick (float64, bit-exact with the reference)
# ---------------------------------------------------------------------------------------------
def _dev_f64(x, device=None):
    import numpy as np
    if isinstance(x, torch.Tensor):
        t = x.to(dtype=torch.float64)
        return t.cuda() if not t.is_cuda else t.contiguous()
    a = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
    return torch.from_numpy(a).to(device or "cuda")


def _ws(nbytes, device):
    t = torch.empty(nbytes + 256, dtype=torch.uint8, device=device)
    return t, _aligned(t)


def ep_filter(objs):
    """utils.get_ep_indices on the GPU. objs [n,M] (host or device) -> numpy int64 indices of the
    non-dominated, non-negative points in ascending objective-0 order."""
    import numpy as np
    if len(objs) == 0:
        return np.zeros(0, dtype=np.int64)
    d = _dev_f64(objs)
    n, M = d.shape
    idx = torch.empty(2 * n, dtype=torch.int32, device=d.device)
    cnt = torch.zeros(1, dtype=torch.int32, device=d.device)
    check(lib().pgm_ep_filter_f64(ptr(d), n, M, ptr(idx), ptr(cnt), _stream()))
    k = int(cnt.item())
    return idx[:k].cpu().numpy().astype(np.int64)


SEL_GLOBAL = 0x1      # PGM_SEL_GLOBAL: the 3-objective global-memory path of K5 at any front size


def front_metrics(pts, force_global=False):
    """(hypervolume, sparsity) of a point set: Population2d semantics for M=2 (get_ep_indices first, hypervolume not
    rounded); for M=3 and M=4 utils.compute_hypervolume (InnerHyperVolume, round(hv, 4)) and utils.compute_sparsity of
    the points as given. M=4 leaves points with a negative coordinate out of the hypervolume, as InnerHyperVolume does;
    M=3 expects none. M=3 takes any size (past 3 936 points K5's global-memory path, with the same bits); at most
    2 202 points at M=4 (the 4-D scorer's shared memory); more raise. force_global=True takes the global-memory path
    at any size (M=3 only), so that tests can compare the two paths."""
    if len(pts) == 0:
        return 0.0, 0.0
    d = _dev_f64(pts)
    n, M = d.shape
    flags = SEL_GLOBAL if force_global else 0
    out = torch.empty(2, dtype=torch.float64, device=d.device)
    nb = lib().pgm_select_workspace_bytes_x(n, 1, M, 1, flags)
    ws, (wp, wn) = _ws(nb, d.device)
    check(lib().pgm_front_metrics_x_f64(ptr(d), n, M, flags, ptr(out), wp, wn, _stream()))
    h, s = out.cpu().tolist()
    return h, s


def select_greedy(ep, cand, alpha, num_tasks, force_global=False):
    """Greedy prediction-guided pick. ep [E,M] archive front, cand [C,M] predicted objectives.
    Returns (best_ids [num_tasks] (-1 = no candidate left), hv [num_tasks,C], sparsity [num_tasks,C],
    final virtual front [n,M]) as numpy arrays. M=3 takes any archive size (past E + num_tasks + 1 = 2 111 points
    K5's global-memory path, with the same bits); force_global=True takes that path at any size (M=3 only)."""
    import numpy as np
    cand_d = _dev_f64(cand)
    C, M = cand_d.shape
    ep = np.asarray(ep, dtype=np.float64).reshape(-1, M)
    E = ep.shape[0]
    ep_d = _dev_f64(ep) if E else torch.zeros(1, M, dtype=torch.float64, device=cand_d.device)
    dev = cand_d.device
    best = torch.empty(num_tasks, dtype=torch.int32, device=dev)
    hv = torch.empty(num_tasks, max(C, 1), dtype=torch.float64, device=dev)
    sp = torch.empty(num_tasks, max(C, 1), dtype=torch.float64, device=dev)
    front = torch.empty(E + num_tasks + 1, M, dtype=torch.float64, device=dev)
    nfront = torch.zeros(1, dtype=torch.int32, device=dev)
    flags = SEL_GLOBAL if force_global else 0
    nb = lib().pgm_select_workspace_bytes_x(E, C, M, num_tasks, flags)
    ws, (wp, wn) = _ws(nb, dev)
    with _nvtx("selection.k5_greedy"):
        check(lib().pgm_select_greedy_x_f64(ptr(ep_d), E, ptr(cand_d), C, M, float(alpha), num_tasks, flags, ptr(best),
                                            ptr(hv), ptr(sp), ptr(front), ptr(nfront), wp, wn, _stream()))
        nf = int(nfront.item())
    return (best.cpu().numpy().astype(np.int64), hv[:, :C].cpu().numpy(), sp[:, :C].cpu().numpy(),
            front[:nf].cpu().numpy())


# ---------------------------------------------------------------------------------------------
# K4: batched hyperbolic-model fits (float64)
# ---------------------------------------------------------------------------------------------
def _fit_result_buffers(F, dev):
    """One float64 buffer for all K4 outputs (a single device -> host copy collects them):
    theta [F,4] | cost [F] | status [F], nfev [F] as int32."""
    res = torch.empty(6 * F, dtype=torch.float64, device=dev)
    ints = res[5 * F:].view(torch.int32)
    return res, res[:4 * F].view(F, 4), res[4 * F:5 * F], ints[:F], ints[F:2 * F]


def fit_hyperbolic_launch(xs, ys, ws, ubs):
    """Upload F ragged fit problems and launch K4 on the current stream WITHOUT waiting for it; the returned
    handle goes to `fit_hyperbolic_collect`. Host work that does not need the fits can run in between."""
    import numpy as np
    F = len(xs)
    if F == 0:
        return None
    klen = np.array([len(v) for v in xs], dtype=np.int32)
    Kmax = max(int(klen.max()), 1)
    pack = np.zeros((3, F, Kmax), dtype=np.float64)
    for f in range(F):
        k = klen[f]
        pack[0, f, :k] = xs[f]; pack[1, f, :k] = ys[f]; pack[2, f, :k] = ws[f]
    dev = torch.device("cuda")
    d = torch.from_numpy(pack).to(dev)
    kl = torch.from_numpy(klen).to(dev)
    ub = _dev_f64(np.asarray(ubs, dtype=np.float64).reshape(F, 4))
    res, theta, cost, status, nfev = _fit_result_buffers(F, dev)
    check(lib().pgm_fit_hyperbolic_f64(ptr(d[0]), ptr(d[1]), ptr(d[2]), ptr(kl), ptr(ub), ptr(theta), ptr(status),
                                       ptr(nfev), ptr(cost), F, Kmax, _stream()))
    return dict(inputs=(d, kl, ub), res=res, F=F)     # inputs kept alive until collect


def fit_inputs_launch(objs, parent, edge_w, edge_dy, node_ids, cap_threshold, force_global_scratch=False):
    """K4 front-end (csrc/k4_inputs.cu): neighbourhood search + widening for every member, then the gather of the
    K4 inputs. objs [n_nodes,M], edges ordered by source node then successor: parent [E], edge_w / edge_dy [E,M];
    node_ids [n]. Returns a dict: device `pack` [3,F,Kmax] (x, y filled; w left for the caller), `ub` [F,4], `klen_f` [F];
    host `klen`, `steps` [n] and `source` [n,Kmax] (source node of every listed edge, zero padded)."""
    import numpy as np
    objs = np.ascontiguousarray(objs, dtype=np.float64)
    n_nodes, M = objs.shape
    E, n = len(parent), len(node_ids)
    dev = torch.device("cuda")
    if n == 0:
        return dict(n=0, M=M, Kmax=1, klen=np.zeros(0, dtype=np.int32), steps=np.zeros(0, dtype=np.int32),
                    source=np.zeros((0, 1), dtype=np.int32))
    # two uploads: the float64 tables and the int32 tables
    fbuf = np.concatenate([objs.reshape(-1), np.asarray(edge_w, dtype=np.float64).reshape(-1),
                           np.asarray(edge_dy, dtype=np.float64).reshape(-1)])
    ibuf = np.concatenate([np.asarray(parent, dtype=np.int32), np.asarray(node_ids, dtype=np.int32)])
    d_f, d_i = torch.from_numpy(fbuf).to(dev), torch.from_numpy(ibuf).to(dev)
    d_objs, d_ew, d_dy = d_f[:n_nodes * M], d_f[n_nodes * M:n_nodes * M + E * M], d_f[n_nodes * M + E * M:]
    d_parent, d_nodes = d_i[:E], d_i[E:]
    ks = torch.empty(2, n, dtype=torch.int32, device=dev)
    edge_idx = torch.empty(n * max(E, 1), dtype=torch.int32, device=dev)
    nb = lib().pgm_fit_neighbours_workspace_bytes(n_nodes, M, E, n)       # 0 unless the graph outgrows shared memory
    if force_global_scratch:
        nb = max(nb, n * ((E * (8 * M + 4) + 2 * n_nodes + 15) // 16 * 16))
    ws, (wp, wn) = _ws(nb, dev) if nb else (None, (None, 0))
    check(lib().pgm_fit_neighbours_f64(ptr(d_objs), n_nodes, M, ptr(d_parent) if E else None, E, ptr(d_ew) if E else None,
                                       ptr(d_nodes), n, int(bool(cap_threshold)), ptr(ks[0]), ptr(ks[1]), ptr(edge_idx),
                                       wp, wn, _stream()))
    ks_h = ks.cpu().numpy()
    Kmax = max(int(ks_h[0].max()), 1)
    F = n * M
    pack = torch.empty(3, F, Kmax, dtype=torch.float64, device=dev)
    ub = torch.empty(F, 4, dtype=torch.float64, device=dev)
    klen_f = torch.empty(F, dtype=torch.int32, device=dev)
    source = torch.zeros(n, Kmax, dtype=torch.int32, device=dev)
    check(lib().pgm_fit_gather_f64(ptr(edge_idx), ptr(ks[0]), n, E, M, ptr(d_parent) if E else None,
                                   ptr(d_ew) if E else None, ptr(d_dy) if E else None, Kmax, ptr(pack[0]), ptr(pack[1]),
                                   ptr(ub), ptr(klen_f), ptr(source), _stream()))
    return dict(n=n, M=M, Kmax=Kmax, pack=pack, ub=ub, klen_f=klen_f, klen=ks_h[0], steps=ks_h[1],
                source=source.cpu().numpy(), keep=(d_f, d_i, edge_idx, ks, ws))


def fit_hyperbolic_launch_packed(front, coef):
    """Launch K4 on the inputs `fit_inputs_launch` left on the device; coef [n,Kmax] (host, float64) = the Gaussian
    point weights of every member, shared by its M fits. Returns the handle `fit_hyperbolic_collect` takes."""
    n, M, Kmax = front["n"], front["M"], front["Kmax"]
    if n == 0:
        return None
    pack, dev = front["pack"], front["pack"].device
    import numpy as np
    c = torch.from_numpy(np.ascontiguousarray(coef, dtype=np.float64)).to(dev)
    pack[2].view(n, M, Kmax).copy_(c.view(n, 1, Kmax).expand(n, M, Kmax))
    F = n * M
    res, theta, cost, status, nfev = _fit_result_buffers(F, dev)
    check(lib().pgm_fit_hyperbolic_f64(ptr(pack[0]), ptr(pack[1]), ptr(pack[2]), ptr(front["klen_f"]), ptr(front["ub"]),
                                       ptr(theta), ptr(status), ptr(nfev), ptr(cost), F, Kmax, _stream()))
    return dict(inputs=front, res=res, F=F)


def fit_hyperbolic_collect(handle):
    """Wait for a `fit_hyperbolic_launch` and return (theta [F,4], status [F], nfev [F], cost [F]) as numpy arrays."""
    import numpy as np
    if handle is None:
        return np.zeros((0, 4)), np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64), np.zeros(0)
    F = handle["F"]
    res = handle["res"].cpu().numpy()                                  # one copy: theta | cost | status, nfev
    ints = res[5 * F:].view(np.int32)
    return (res[:4 * F].reshape(F, 4).copy(), ints[:F].astype(np.int64), ints[F:2 * F].astype(np.int64),
            res[4 * F:5 * F].copy())


def fit_hyperbolic(xs, ys, ws, ubs):
    """Fit F models at once. xs/ys/ws: lists of 1-D arrays (ragged, K_f points each); ubs [F,4].
    Returns (theta [F,4], status [F], nfev [F], cost [F]) as numpy arrays."""
    return fit_hyperbolic_collect(fit_hyperbolic_launch(xs, ys, ws, ubs))
