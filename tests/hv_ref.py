"""Test infrastructure: a literal restatement, for any number of objectives, of the reference's exact hypervolume
(morl/hypervolume.py:41-153, the Fonseca-Paquete-Lopez-Ibanez dimension sweep over `MultiList`), and the greedy pick
of population_3d.py:294-333 built on it.

`oracle/selection_oracle.py` restates the 2-D and 3-D sweeps in closed form; the reference goldens pin those. At 4
objectives the closed form (3-D volumes of the objective-3 prefixes times the gaps) is NOT the reference's arithmetic:
`hvRecursive` reuses a node's stored slice area instead of recomputing it once a fresh area did not grow
(`ignore = dimIndex`), and those flags persist across calls, which moves some results by an ulp. This module keeps the
linked lists, bounds, stored volumes/areas and ignore flags exactly as the reference does, so its float64 operations
are the reference's, one for one. tests/test_oracle_hv_md.py pins it against the 3-D goldens of the unmodified
reference; no golden of the reference exists at 4 objectives.
"""
import numpy as np

from oracle import selection_oracle as so

# how often hvRecursive took a stored area instead of recomputing it (the `q.ignore >= dimIndex` branch), summed over
# every call since the last reset_reuse_count(); tests use it to show their inputs reach that branch
reuse_count = 0


def reset_reuse_count():
    global reuse_count
    reuse_count = 0


class _Node:
    __slots__ = ("cargo", "next", "prev", "ignore", "area", "volume")

    def __init__(self, m, cargo=None):
        self.cargo = cargo
        self.next = [None] * m
        self.prev = [None] * m
        self.ignore = 0
        self.area = [0.0] * m
        self.volume = [0.0] * m


class _MultiList:
    def __init__(self, m):
        self.m = m
        self.sentinel = _Node(m)
        self.sentinel.next = [self.sentinel] * m
        self.sentinel.prev = [self.sentinel] * m

    def extend(self, nodes, index):
        sentinel = self.sentinel
        for node in nodes:
            last = sentinel.prev[index]
            node.next[index] = sentinel
            node.prev[index] = last
            sentinel.prev[index] = node
            last.next[index] = node

    def remove(self, node, index, bounds):
        for i in range(index):
            pred, succ = node.prev[i], node.next[i]
            pred.next[i] = succ
            succ.prev[i] = pred
            if bounds[i] > node.cargo[i]:
                bounds[i] = node.cargo[i]
        return node

    def reinsert(self, node, index, bounds):
        for i in range(index):
            node.prev[i].next[i] = node
            node.next[i].prev[i] = node
            if bounds[i] > node.cargo[i]:
                bounds[i] = node.cargo[i]


def _hv_recursive(lst, dim, length, bounds):
    global reuse_count
    hvol = 0.0
    sentinel = lst.sentinel
    if length == 0:
        return hvol
    if dim == 0:
        return -sentinel.next[0].cargo[0]
    if dim == 1:
        q = sentinel.next[1]
        h = q.cargo[0]
        p = q.next[1]
        while p is not sentinel:
            pc = p.cargo
            hvol += h * (q.cargo[1] - pc[1])
            if pc[0] < h:
                h = pc[0]
            q = p
            p = q.next[1]
        hvol += h * q.cargo[1]
        return hvol
    p = sentinel
    q = p.prev[dim]
    while q.cargo is not None:
        if q.ignore < dim:
            q.ignore = 0
        q = q.prev[dim]
    q = p.prev[dim]
    while length > 1 and (q.cargo[dim] > bounds[dim] or q.prev[dim].cargo[dim] >= bounds[dim]):
        p = q
        lst.remove(p, dim, bounds)
        q = p.prev[dim]
        length -= 1
    q_area, q_cargo, q_prev = q.area, q.cargo, q.prev[dim]
    if length > 1:
        hvol = q_prev.volume[dim] + q_prev.area[dim] * (q_cargo[dim] - q_prev.cargo[dim])
    else:
        q_area[0] = 1
        q_area[1:dim + 1] = [q_area[i] * -q_cargo[i] for i in range(dim)]
    q.volume[dim] = hvol
    if q.ignore >= dim:
        q_area[dim] = q_prev.area[dim]
        reuse_count += 1
    else:
        q_area[dim] = _hv_recursive(lst, dim - 1, length, bounds)
        if q_area[dim] <= q_prev.area[dim]:
            q.ignore = dim
    while p is not sentinel:
        p_cargo_dim = p.cargo[dim]
        hvol += q.area[dim] * (p_cargo_dim - q.cargo[dim])
        bounds[dim] = p_cargo_dim
        lst.reinsert(p, dim, bounds)
        length += 1
        q = p
        p = p.next[dim]
        q.volume[dim] = hvol
        if q.ignore >= dim:
            q.area[dim] = q.prev[dim].area[dim]
            reuse_count += 1
        else:
            q.area[dim] = _hv_recursive(lst, dim - 1, length, bounds)
            if q.area[dim] <= q.prev[dim].area[dim]:
                q.ignore = dim
    hvol -= q.area[dim] * q.cargo[dim]
    return hvol


def hv_raw(front):
    """Un-rounded hypervolume of `front` (maximisation, reference point 0), any number of objectives: negate, keep the
    points that weakly dominate the reference point (hypervolume.py:55-61), preProcess (:156-164: the node list sorted
    stably by each dimension in turn, each order recorded as one linked list), then hvRecursive from the top dimension
    with bounds [-1e308] * M."""
    pts = [[-float(v) for v in p] for p in front]
    pts = [p for p in pts if all(v <= 0.0 for v in p)]
    if not pts:
        return 0.0
    m = len(pts[0])
    lst = _MultiList(m)
    nodes = [_Node(m, p) for p in pts]
    for i in range(m):
        nodes.sort(key=lambda node: node.cargo[i])          # list.sort is stable: ties keep the previous order
        lst.extend(nodes, i)
    return _hv_recursive(lst, m - 1, len(nodes), [-1.0e308] * m)


def hv(front):
    """utils.compute_hypervolume: InnerHyperVolume(zeros).compute(front) -> round(hv, 4) (hypervolume.py:74)."""
    return round(hv_raw(front), 4)


def greedy_select_md(ep_objs, preds, alpha, num_tasks):
    """population_3d.py:294-333 with the serial scorer (:206-214) at any number of objectives. Returns (best ids,
    per-round hv arrays, per-round sparsity arrays, final virtual front)."""
    vep = [np.asarray(p, dtype=np.float64) for p in ep_objs]
    preds = np.asarray(preds, dtype=np.float64)
    mask = np.ones(len(preds), dtype=bool)
    best_ids, hvs, sps = [], [], []
    for _ in range(num_tasks):
        h = np.zeros(len(preds)); s = np.zeros(len(preds))
        for i in range(len(preds)):
            if mask[i]:
                new_ep = so.update_ep(vep, preds[i])
                h[i] = hv(new_ep); s[i] = so.sparsity_md(new_ep)
        hvs.append(h); sps.append(s)
        best, best_v = -1, -np.inf
        for i in range(len(preds)):
            if mask[i] and h[i] - alpha * s[i] > best_v:
                best, best_v = i, h[i] - alpha * s[i]
        if best == -1:
            break
        best_ids.append(best)
        mask[best] = False
        vep = so.update_ep(vep, preds[best])
    return best_ids, hvs, sps, vep
