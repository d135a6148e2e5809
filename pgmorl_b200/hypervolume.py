"""Exact hypervolume indicator with the reference's interface (morl/hypervolume.py:23-74).

The reference implements variant 3 of the Fonseca-Paquete-Lopez-Ibanez dimension sweep with linked
lists; for 2 and 3 objectives it reduces to a sorted sweep / z-slices of 2-D areas, and at 4 objectives
the kernel replays the sweep's stored volumes, areas and area-reuse flags. `compute` runs it on the GPU
(csrc/k5_select.cu) in float64 with the reference's operations and order and returns `round(hv, 4)`
like hypervolume.py:74. The device kernels stop at 4 objectives (MAX_OBJECTIVES)."""
import numpy as np

from . import kernels as K

MAX_OBJECTIVES = 4


class InnerHyperVolume:
    def __init__(self, referencePoint):
        self.referencePoint = np.asarray(referencePoint, dtype=np.float64)

    def compute(self, front):
        """Hypervolume dominated by `front` (maximisation) w.r.t. the reference point."""
        pts = np.asarray(front, dtype=np.float64)
        if pts.size == 0:
            return 0.0
        pts = pts - self.referencePoint
        pts = pts[(pts >= 0).all(axis=1)]          # only points dominating the reference point count (:57-61)
        if len(pts) == 0:
            return 0.0
        M = pts.shape[1]
        if M in (3, 4):
            return K.front_metrics(pts)[0]
        if M == 2:
            return round(K.front_metrics(pts)[0], 4)
        raise NotImplementedError(f"InnerHyperVolume: device kernels cover 2 to {MAX_OBJECTIVES} objectives (got {M})")
