"""Flat parameter layout of one (policy, value) network of the population.

The order is the reference's ``Policy.named_parameters()`` order
(a2c_ppo_acktr/model.py:201-256 MLPBase/MOMLPBase with layernorm off,
distributions.py:71-79 DiagGaussian, utils.py:32-35 AddBias), so that a flat
vector converts to / from a reference ``state_dict`` by plain slicing:

    base.actor.0.{weight[H,O],bias[H]}, base.actor.2.{weight[H,H],bias[H]},
    base.critic.0.{...}, base.critic.2.{...},
    base.critic_linear.{weight[M,H],bias[M]},
    dist.fc_mean.{weight[A,H],bias[A]}, dist.logstd._bias[A,1]

A Categorical head (Discrete(n) actions, distributions.py Categorical) ends in
``dist.linear.{weight[n,H],bias[n]}`` instead: 12 tensors, no logstd.

The same offsets are compiled into the CUDA side (csrc/common.cuh,
``struct NetLayout``, exported as ``pgm_param_offsets``); tests/test_cabi.py checks
that both agree for every named environment shape.
"""
from collections import OrderedDict
from dataclasses import dataclass


DIST_GAUSSIAN, DIST_CATEGORICAL = 0, 1   # action heads (PGM_DIST_* of include/pgmorl_b200.h)
CATEGORICAL_MAX = 32                     # categories the kernels accept (K3's head tile)


@dataclass(frozen=True)
class NetDims:
    obs: int      # O
    act: int      # A: action dimension (Gaussian) or number of categories n (Categorical)
    obj: int      # M
    hidden: int = 64
    dist: int = DIST_GAUSSIAN

    @property
    def n_par(self):
        return param_layout(self)[1]

    @property
    def categorical(self):
        return self.dist == DIST_CATEGORICAL

    @property
    def act_cols(self):
        """Columns of an action in the rollout buffers: A, or 1 (the category index) for a Categorical head."""
        return 1 if self.categorical else self.act


def param_layout(d):
    """-> (OrderedDict name -> (offset, shape), n_par)."""
    O, A, M, H = d.obs, d.act, d.obj, d.hidden
    head = ([("dist.linear.weight", (A, H)), ("dist.linear.bias", (A,))] if d.dist == DIST_CATEGORICAL else
            [("dist.fc_mean.weight", (A, H)), ("dist.fc_mean.bias", (A,)), ("dist.logstd._bias", (A, 1))])
    spec = [
        ("base.actor.0.weight", (H, O)), ("base.actor.0.bias", (H,)),
        ("base.actor.2.weight", (H, H)), ("base.actor.2.bias", (H,)),
        ("base.critic.0.weight", (H, O)), ("base.critic.0.bias", (H,)),
        ("base.critic.2.weight", (H, H)), ("base.critic.2.bias", (H,)),
        ("base.critic_linear.weight", (M, H)), ("base.critic_linear.bias", (M,)),
    ] + head
    out, off = OrderedDict(), 0
    for name, shape in spec:
        n = 1
        for s in shape:
            n *= s
        out[name] = (off, shape)
        off += n
    return out, off


# Named environment shapes from the reference's launch scripts (SURVEY.md section 8). Ant's 27 observations are qpos[2:]
# and qvel of the reference's environments/ant.py, without contact forces.
ENV_SHAPES = {
    "walker2d": NetDims(17, 6, 2),
    "halfcheetah": NetDims(17, 6, 2),
    "hopper2": NetDims(11, 3, 2),
    "hopper3": NetDims(11, 3, 3),
    "ant": NetDims(27, 8, 2),
    "swimmer": NetDims(8, 2, 2),
    "humanoid": NetDims(376, 17, 2),
}
