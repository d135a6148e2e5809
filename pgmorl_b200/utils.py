"""Selection helpers with the reference's names and semantics (mirror of morl/utils.py:21-106).
The arithmetic-heavy ones run in the float64 CUDA kernels of K5 (bit-exact with the reference);
there is no CPU implementation behind them."""
from copy import deepcopy

import math

import numpy as np

from . import kernels as K


def print_info(*message):
    print('\033[96m', *message, '\033[0m')


def print_warning(*message):
    print('\033[93m', *message, '\033[0m')


def check_dominated(obj_batch, obj):
    """True if some row of obj_batch weakly dominates obj with one strict inequality (utils.py:24-28).
    Single-point query used only by callers outside the hot path; plain numpy comparison."""
    obj_batch = np.asarray(obj_batch)
    return bool(np.logical_and((obj_batch >= obj).all(axis=1), (obj_batch > obj).any(axis=1)).any())


def get_ep_indices(obj_batch_input):
    """Sorted (ascending objective 0) indices of the non-dominated, non-negative points (utils.py:31-39)."""
    if len(obj_batch_input) == 0:
        return np.array([])
    return K.ep_filter(np.array(obj_batch_input, dtype=np.float64)).tolist()


def update_ep(ep_objs_batch, new_objs):
    """Fold one point into a front with the reference's 1e-5 tolerances (utils.py:42-65); the front stays
    ordered by objective 0. Runs the same device routine the 3- and 4-objective greedy selection uses."""
    from .hypervolume import MAX_OBJECTIVES
    new_objs = np.asarray(new_objs, dtype=np.float64)
    M = len(new_objs)
    if M > MAX_OBJECTIVES:
        raise NotImplementedError(f"update_ep: the device kernels cover at most {MAX_OBJECTIVES} objectives (got {M})")
    if M < 3:
        raise NotImplementedError("update_ep: the reference calls it for 3 or more objectives only; so does the kernel")
    ep = np.asarray(ep_objs_batch, dtype=np.float64).reshape(-1, M)
    front = K.select_greedy(ep, new_objs[None, :], 0.0, 1)[3]      # one candidate, one round: it is folded in
    return [row.copy() for row in front]


def generate_weights_batch_dfs(i, obj_num, min_weight, max_weight, delta_weight, weight, weights_batch):
    """Simplex-grid enumeration with the reference's float accumulation `w += delta` (utils.py:67-78)."""
    if i == obj_num - 1:
        weight.append(1.0 - np.sum(weight[0:i]))
        weights_batch.append(deepcopy(weight))
        weight = weight[0:i]
        return
    w = min_weight
    while w < max_weight + 0.5 * delta_weight and np.sum(weight[0:i]) + w < 1.0 + 0.5 * delta_weight:
        weight.append(w)
        generate_weights_batch_dfs(i + 1, obj_num, min_weight, max_weight, delta_weight, weight, weights_batch)
        weight = weight[0:i]
        w += delta_weight


def compute_hypervolume(ep_objs_batch):
    """Exact hypervolume of a front w.r.t. the origin (utils.py:81-84 -> InnerHyperVolume)."""
    from .hypervolume import InnerHyperVolume
    n = len(ep_objs_batch[0])
    return InnerHyperVolume(np.zeros(n)).compute(ep_objs_batch)


def compute_sparsity(ep_objs_batch):
    """Per-dimension sorted squared gaps / (n - 1) (utils.py:87-100)."""
    from .hypervolume import MAX_OBJECTIVES
    if len(ep_objs_batch) < 2:
        return 0.0
    pts = np.asarray(ep_objs_batch, dtype=np.float64)
    if pts.shape[1] > MAX_OBJECTIVES:
        raise NotImplementedError(f"compute_sparsity: the device kernels cover at most {MAX_OBJECTIVES} objectives "
                                  f"(got {pts.shape[1]})")
    if pts.shape[1] not in (3, 4):
        raise NotImplementedError("compute_sparsity: the device kernel covers 3 and 4 objectives (2 objectives use "
                                  "Population.compute_sparsity)")
    return K.front_metrics(pts)[1]


def update_ep_and_compute_hypervolume_sparsity(task_id, ep_objs_batch, new_objs, queue):
    """Process entry point of the reference's 3-objective scorer (utils.py:102-106); kept for API parity."""
    new_ep = update_ep(ep_objs_batch, new_objs)
    queue.put([task_id, compute_hypervolume(new_ep), compute_sparsity(new_ep)])


def norm2(v):
    """np.linalg.norm of a real 1-D vector without its Python overhead: the same two operations numpy performs
    (sqnorm = v.dot(v); sqrt(sqnorm)), hence the same bits -- the selection compares these against thresholds."""
    v = np.asarray(v)
    return math.sqrt(v.dot(v))


# ---------------------------------------------------------------------------------------------
# Row-wise versions of the scalar numpy expressions the reference evaluates per point. The selection
# front-end batches them over the whole population, and the batched form has to give the SAME BITS as
# the scalar calls it replaces: BLAS ddot (np.dot / np.linalg.norm of a short vector) accumulates with
# fused multiply-adds, C pow (`float ** 2`) is not always the correctly rounded square. np.vecdot and
# np.float_power go through the same code as the scalar calls; that is checked once on this machine's
# numpy / BLAS build, and the scalar loop is used instead should it ever not hold.
# ---------------------------------------------------------------------------------------------
def _rowdot_loop(a, b):
    out = np.empty(a.shape[:-1])
    flat_a, flat_b, flat_o = a.reshape(-1, a.shape[-1]), b.reshape(-1, b.shape[-1]), out.reshape(-1)
    for i in range(len(flat_o)):
        flat_o[i] = flat_a[i].dot(flat_b[i])
    return out


def _pow2_loop(x):
    out = np.empty(x.shape)
    flat_x, flat_o = x.reshape(-1), out.reshape(-1)
    for i in range(len(flat_o)):
        flat_o[i] = math.pow(flat_x[i], 2.0)
    return out


def _batched_forms_match():
    rng = np.random.RandomState(12345)
    if not hasattr(np, "vecdot"):
        return False, False
    dot_ok = True
    for m in (2, 3, 4):
        a = rng.rand(512, m) * rng.choice([1e-3, 1.0, 50.0], size=(512, 1))
        b = rng.rand(512, m) - 0.5
        dot_ok = dot_ok and np.array_equal(np.vecdot(a, b), _rowdot_loop(a, b))
    x = np.abs(rng.randn(4096)) * 3.0
    pow_ok = np.array_equal(np.float_power(x, 2.0), _pow2_loop(x))
    return dot_ok, pow_ok


_ROWDOT_FAST, _POW2_FAST = _batched_forms_match()


def rowdot(a, b):
    """dot product of corresponding rows (last axis), bit-identical to `a[i].dot(b[i])`."""
    a, b = np.broadcast_arrays(a, b)
    a, b = np.ascontiguousarray(a, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    return np.vecdot(a, b) if _ROWDOT_FAST else _rowdot_loop(a, b)


def rownorm(a):
    """np.linalg.norm of every row (last axis), bit-identical to the per-row call (sqrt of the BLAS dot)."""
    return np.sqrt(rowdot(a, a))


def pow2(x):
    """x ** 2 as Python floats / numpy scalars compute it (C pow), element-wise."""
    x = np.asarray(x, dtype=np.float64)
    return np.float_power(x, 2.0) if _POW2_FAST else _pow2_loop(x)
