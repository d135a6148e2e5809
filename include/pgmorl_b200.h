/*
 * pgmorl_b200.h -- C ABI of the B200-native PG-MORL hot path.
 *
 * The reference (albo437/PGMORL) is pure Python and has no FFI layer; the
 * "binding" a maintainer adds is a ctypes stub (see INTEGRATION.md). Each entry
 * point below names the reference code whose arithmetic it replaces
 * (paths relative to the reference root; a2c = externals/pytorch-a2c-ppo-acktr-gail/a2c_ppo_acktr).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *     the caller owns all buffers, kernels never allocate;
 *   - arrays are dense, row-major, in the shapes written beside them;
 *   - P = tasks in the population shard, T = num_steps, N = envs per task,
 *     O/A/M = obs / action / objective dims, S = T*N samples per task,
 *     n_par = pgm_n_par(O,A,M) parameters per task in the reference's
 *     named_parameters() order (pgmorl_b200/layout.py);
 *   - `stream` is a cudaStream_t (NULL = legacy default stream); calls are
 *     asynchronous w.r.t. the host unless stated;
 *   - return value 0 = success, otherwise an error code; pgm_last_error()
 *     gives the message of the last failure on the calling thread.
 *   - hidden width: 64 (a2c/model.py:202 default, warm_up.py:34-38) in every entry point without a `hidden`
 *     argument; the *_h entry points take it explicitly and accept 32, 64 and 128 (MLPBase(hidden_size=...)).
 *     Any other width is an error. Width 64 runs the same kernels as the entry points without `hidden`; 32 and 128 run
 *     the FP32 FFMA kernels only (K1's FFMA forward, K3's generic cluster kernel at 2..16 CTAs per task).
 *     Shared memory bounds the observation width: at 128 one network half of Walker2d's shape is about 80 KB and
 *     Humanoid (O = 376, 194 KB for W1 alone) fits neither K1 nor K3; at 32 every named shape fits, Humanoid included.
 */
#ifndef PGMORL_B200_H
#define PGMORL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGM_ABI_VERSION 1
#define PGM_HIDDEN 64

enum {
    PGM_OK = 0,
    PGM_ERR_ARG = 1,      /* bad shape / null pointer / unsupported size */
    PGM_ERR_CUDA = 2,     /* a CUDA runtime call failed */
    PGM_ERR_WORKSPACE = 3 /* workspace too small */
};

/* action mode of pgm_policy_forward_f32 */
enum {
    PGM_ACT_SAMPLE = 0,        /* action = mean + exp(logstd)*eps   (a2c/model.py:64-65)  */
    PGM_ACT_DETERMINISTIC = 1, /* action = mean                      (a2c/model.py:61-62)  */
    PGM_ACT_EVALUATE = 2       /* action given, only log-prob        (a2c/model.py:75-82)  */
};

/* action distribution head (`dist` argument of the _x entry points) */
enum {
    PGM_DIST_GAUSSIAN = 0,   /* Box actions: DiagGaussian, mean head + state-independent logstd (a2c/distributions.py:71-90) */
    PGM_DIST_CATEGORICAL = 1 /* Discrete(n) actions: Categorical, logits head, no logstd (a2c/distributions.py Categorical) */
};
/* categories of a Categorical head the kernels accept: 1 <= n <= PGM_CATEGORICAL_MAX (the head rows of K3's generic kernel) */
#define PGM_CATEGORICAL_MAX 32

int pgm_abi_version(void);
const char *pgm_last_error(void);

/* number of parameters of one policy (actor H-H + critic H-H + heads + logstd; H = 64, or `hidden` for the _h form,
 * which returns -1 and sets pgm_last_error() for a width other than 32, 64, 128) */
int pgm_n_par(int obs_dim, int act_dim, int obj_num);
int pgm_n_par_h(int obs_dim, int act_dim, int obj_num, int hidden);
/* offsets (in elements) of the 13 parameter tensors of one policy inside its flat vector, in the reference's
 * named_parameters() order: base.actor.0.{weight,bias}, base.actor.2.{weight,bias}, base.critic.0.{...}, base.critic.2.{...},
 * base.critic_linear.{weight,bias}, dist.fc_mean.{weight,bias}, dist.logstd._bias (a2c/model.py:201-256) */
int pgm_param_offsets(int obs_dim, int act_dim, int obj_num, int *out13);
int pgm_param_offsets_h(int obs_dim, int act_dim, int obj_num, int hidden, int *out13);
/* _x forms: hidden width `hidden` and action head `dist`. For PGM_DIST_CATEGORICAL, act_dim is the number of categories n
 * and the layout has 12 tensors: the 10 base tensors, then dist.linear.{weight [n,H], bias [n]} (the Categorical
 * module of a2c/distributions.py; Policy.__init__ in a2c/model.py builds base, then dist), no logstd. pgm_param_offsets_x writes one offset per
 * tensor (13 or 12). Both return -1 / PGM_ERR_ARG and set pgm_last_error() for an unsupported width, head or n. */
int pgm_n_par_x(int obs_dim, int act_dim, int obj_num, int hidden, int dist);
int pgm_param_offsets_x(int obs_dim, int act_dim, int obj_num, int hidden, int dist, int *out);

/* ---------------------------------------------------------------------------
 * K1  population-batched actor-critic forward.
 * Replaces Policy.act / get_value / evaluate_actions (a2c/model.py:57-82),
 * MLPBase/MOMLPBase.forward (a2c/model.py:237-256), DiagGaussian + FixedNormal
 * (a2c/distributions.py:30-40,71-90) as called 2048x per iteration from
 * morl/mopg.py:103-135.
 *
 *   params  [P, n_par]
 *   obs     [P, rows_v, O]          value is produced for all rows_v rows
 *   eps     [P or 1, rows_a, A]     N(0,1) draws (SAMPLE mode); eps_shared!=0 => one copy for all tasks
 *   action  [P, rows_a, A]          out (SAMPLE/DETERMINISTIC) or in (EVALUATE); first rows_a rows of obs
 *   value   [P, rows_v, M]  out ;   logp [P, rows_a] out
 * Trajectory mode: rows_v=(T+1)*N, rows_a=T*N.  Per-step mode: rows_v=rows_a=N.
 * get_value: rows_a=0.
 * pgm_policy_forward_h_f32: the same at hidden width `hidden` (32, 64, 128). The tensor-core forwards serve width 64;
 * 32 and 128 run on the FP32 FFMA kernel, which refuses an observation width whose parameter image exceeds 227 KB of
 * shared memory (Humanoid at 128).
 */
int pgm_policy_forward_f32(const float *params, const float *obs, const float *eps, int eps_shared,
                           float *action, float *value, float *logp, int mode, int P, int rows_v,
                           int rows_a, int O, int A, int M, void *stream);
int pgm_policy_forward_h_f32(const float *params, const float *obs, const float *eps, int eps_shared,
                             float *action, float *value, float *logp, int mode, int P, int rows_v,
                             int rows_a, int O, int A, int M, int hidden, void *stream);
/* pgm_policy_forward_x_f32: the _h form with the action head `dist`; _h is its PGM_DIST_GAUSSIAN case (entropy NULL).
 * PGM_DIST_CATEGORICAL (Categorical / FixedCategorical of a2c/distributions.py), A = n categories
 * (1 <= n <= PGM_CATEGORICAL_MAX), logits z = W h2 + b:
 *   eps     [P or 1, rows_a, n]  Exponential(1) draws q (SAMPLE mode): action = first argmax_j softmax(z)_j / q_j, the
 *                                single-sample path of torch.multinomial(probs, 1, True) in torch 2.11 (dist.sample())
 *   action  [P, rows_a, 1]       the category index as a float (exact up to 2^24); DETERMINISTIC = first argmax_j z_j
 *                                (dist.mode()), EVALUATE reads it
 *   logp    [P, rows_a]          z_a - logsumexp(z)
 *   entropy [P, rows_a] or NULL  per-row -sum_j p_j log p_j (Categorical only; must be NULL for a Gaussian head)
 * Categorical heads always run on the FP32 FFMA kernel (no tensor-core forward). */
int pgm_policy_forward_x_f32(const float *params, const float *obs, const float *eps, int eps_shared,
                             float *action, float *value, float *logp, float *entropy, int mode, int P, int rows_v,
                             int rows_a, int O, int A, int M, int hidden, int dist, void *stream);

/* K1 in per-step mode for real environment loops (morl/mopg.py:103-135: one Policy.act per environment step): every
 * task's N current observations -> value / sampled action / log-prob written STRAIGHT INTO time slot t of the rollout
 * buffers (what RolloutStorage.insert does, a2c/storage.py:50-62), plus a dense copy of the actions for the host.
 *   ctl      [2] int32 in DEVICE memory: {t, sample}. sample = 0: value only (the bootstrap get_value of mopg.py:132-135).
 *            Read by the kernel, so ONE captured CUDA graph (H2D of the staged step -> this launch -> D2H of the
 *            actions) serves every step of every iteration.
 *   obs_stage [P,N,O] dense block of this step's observations, copied by the kernel into slot t of obs_buf; or NULL:
 *            the observations are already in slot t of obs_buf (written there by K6, pgm_vecnorm_step_f64).
 *   eps      [P or 1, N, A] N(0,1) draws of this step
 *   obs_buf [P,(T+1)N,O], value_buf [P,(T+1)N,M], action_buf [P,TN,A], logp_buf [P,TN]: rollout buffers, row = t*N + n,
 *            task strides in elements;  act_out [P,N,A] dense (may be NULL). */
int pgm_policy_step_f32(const float *params, const int32_t *ctl, const float *obs_stage, const float *eps,
                        int eps_shared, float *obs_buf, size_t obs_task_stride, float *value_buf,
                        size_t value_task_stride, float *action_buf, size_t action_task_stride, float *logp_buf,
                        size_t logp_task_stride, float *act_out, int P, int N, int O, int A, int M, void *stream);
int pgm_policy_step_h_f32(const float *params, const int32_t *ctl, const float *obs_stage, const float *eps,
                          int eps_shared, float *obs_buf, size_t obs_task_stride, float *value_buf,
                          size_t value_task_stride, float *action_buf, size_t action_task_stride, float *logp_buf,
                          size_t logp_task_stride, float *act_out, int P, int N, int O, int A, int M, int hidden,
                          void *stream);
/* the _h form with the action head `dist`; for PGM_DIST_CATEGORICAL eps is [P or 1, N, n] Exponential(1) draws and
 * action_buf [P,TN,1] / act_out [P,N,1] receive the sampled category index (pgm_policy_forward_x_f32) */
int pgm_policy_step_x_f32(const float *params, const int32_t *ctl, const float *obs_stage, const float *eps,
                          int eps_shared, float *obs_buf, size_t obs_task_stride, float *value_buf,
                          size_t value_task_stride, float *action_buf, size_t action_task_stride, float *logp_buf,
                          size_t logp_task_stride, float *act_out, int P, int N, int O, int A, int M, int hidden,
                          int dist, void *stream);

/* ---------------------------------------------------------------------------
 * K2  vector-reward returns + scalarised, normalised advantage.
 * Replaces RolloutStorage.compute_returns (a2c/storage.py:77-116) and the PPO.update preamble
 * (a2c/algo/ppo.py:43-56) with WeightedSumScalarization.evaluate (morl/scalarization_methods.py:28-29).
 *
 *   rewards [P,T,N,M]  value [P,T+1,N,M]  masks,bad_masks [P,T+1,N]
 *   weights [P,M]  obj_var [P,M] or NULL (NULL => no un-normalisation)
 *   returns [P,T,N,M] out     adv [P,T,N] out (skipped when weights==NULL or adv==NULL)
 *
 * pgm_returns_adv_f32: the branch of compute_returns is `mode`, an OR of
 *   PGM_RET_GAE                 use_gae: generalised advantage estimation with lambda = lam
 *                               (otherwise n-step discounted returns; lam is ignored)
 *   PGM_RET_PROPER_TIME_LIMITS  use_proper_time_limits: bad_masks cut the recursion at time-limit ends
 *                               (otherwise bad_masks is read by no branch)
 *   boot [P,N,M] or NULL: the bootstrap value of the n-step branches (returns[-1] = next_value); NULL = value row T.
 *   The GAE branches bootstrap from value row T and ignore boot. The advantage is returns - value[:T] in every branch.
 * pgm_gae_adv_f32 = pgm_returns_adv_f32 with mode PGM_RET_GAE | PGM_RET_PROPER_TIME_LIMITS and boot NULL
 *   (storage.py:83-94, the branch PG-MORL runs).
 */
enum {
    PGM_RET_GAE = 1,
    PGM_RET_PROPER_TIME_LIMITS = 2
};

int pgm_returns_adv_f32(const float *rewards, const float *value, const float *boot, const float *masks,
                        const float *bad_masks, const float *weights, const float *obj_var, float gamma, float lam,
                        int mode, float *returns, float *adv, int P, int T, int N, int M, void *stream);

int pgm_gae_adv_f32(const float *rewards, const float *value, const float *masks,
                    const float *bad_masks, const float *weights, const float *obj_var,
                    float gamma, float lam, float *returns, float *adv, int P, int T, int N, int M,
                    void *stream);

/* ---------------------------------------------------------------------------
 * K3  PPO update: E epochs x B minibatches of clipped surrogate + (clipped) vector
 * value loss (- ecoef*entropy), backward, global grad-norm clip, Adam -- all tasks
 * in one launch, each task's chain of E*B dependent steps run by one thread-block
 * cluster. Replaces PPO.update (a2c/algo/ppo.py:62-115), feed_forward_generator
 * (a2c/storage.py:118-154), nn.utils.clip_grad_norm_ and torch.optim.Adam.step.
 *
 *   params, adam_m, adam_v [P, n_par]  in/out     adam_step [P] int32 in/out
 *   lr  [P] double (per-task learning rate of this iteration, a2c/utils.py:46-50)
 *   obs [P,S(+N),O] (first S rows used)   action [P,S,A]   logp_old [P,S]
 *   value_old [P,S(+N),M] (first S rows; task stride given)   returns [P,S,M]   adv [P,S]
 *   perm [P or 1, E, S] int32 : minibatch b of epoch e = perm[e, b*mb:(b+1)*mb], mb = S / B
 *   losses [P,3] out: mean over E*B updates of (value_loss, action_loss, entropy)
 *   workspace: >= pgm_ppo_workspace_bytes(...) bytes, 256-byte aligned
 *   cluster: 1,2,4,8,16 = CTAs per task of the FP32 FFMA kernels (O <= 384, A <= 32, M <= 16 at 2..16; cluster 1 keeps
 *            both halves in one CTA and refuses shapes whose halves need more than 227 KB together, e.g. Humanoid's);
 *            32 / 64 = the tensor-core kernel (tcgen05 UMMA on FP16 operand pairs, FP32 accumulate, FP32-level
 *            accuracy) with 2 / 4 CTAs per task, built for the (O,A,M) shapes (17,6,2) and (11,3,3); 0 = choose
 *            from P, the shape and the SM count (tensor cores from 8 tasks on).
 *            Tensor-core operand ranges: |obs| < 65 504 (unscaled fp16 pairs), |parameter| < 255.9, |backward signal| < 16;
 *            beyond them the task's outputs become inf / NaN (non-saturating conversions), never a silently clamped result.
 *            OR-able flags 0x100 / 0x200 / 0x400 / 0x800 / 0x1000 / 0x2000 / 0x4000 select the step tail of the FFMA cluster
 *            kernel (A/B and tests; bit-identical results; default = 0x2000, csrc/k3_ppo.cu).
 *            OR-able flag PGM_PPO_VALUE_UNCLIPPED (every kernel family): the value loss is 0.5 * mean((V - R)^2)
 *            (use_clipped_value_loss=False, a2c/algo/ppo.py:86-94 else branch) instead of the clipped
 *            0.5 * mean(max((V - R)^2, (V_clip - R)^2)); losses[:,0] reports the loss that was minimised.
 *   S and B must satisfy S % B < S / B (the reference's BatchSampler(drop_last=True) then yields exactly B minibatches).
 * The _h forms take the hidden width (32, 64, 128). At 32 and 128 only the generic FFMA cluster kernel exists: cluster
 *   0 (auto, 2..16 CTAs per task), 2, 4, 8 or 16; cluster 1 and the tensor-core values 32 / 64 / 128 are refused with an
 *   error naming the width. A shape whose network half exceeds 227 KB of shared memory is refused (Humanoid at 128);
 *   at 128 the observation width is also limited to O <= 128 (the register tile of dW1), at 32 to O <= 384.
 *   At 64 they are the functions without `hidden`.
 * The _x forms take the hidden width and the action head `dist`; the _h forms are their PGM_DIST_GAUSSIAN case.
 *   PGM_DIST_CATEGORICAL: A = n categories (1 <= n <= PGM_CATEGORICAL_MAX), action [P,S,1] holds the category index as a
 *   float; log-prob z_a - logsumexp(z) and entropy -sum_j p_j log p_j per row (FixedCategorical of a2c/distributions.py),
 *   whose gradient d(-entropy_coef * mean_i H_i)/dz_ij = entropy_coef / mb * p_ij (log p_ij + H_i) joins the surrogate's;
 *   losses[:,2] is the entropy averaged over rows and updates. Only the generic FFMA cluster kernel serves this head, at
 *   every hidden width: cluster 0 (auto), 2, 4, 8 or 16. cluster 1 and the tensor-core values 32 / 64 / 128 are refused
 *   with an error naming the categorical head.
 */
#define PGM_PPO_VALUE_UNCLIPPED 0x10000

typedef struct {
    double clip_param;      /* 0.2  a2c/algo/ppo.py:83-84  */
    double value_loss_coef; /* 0.5  */
    double entropy_coef;    /* 0.0  */
    double max_grad_norm;   /* 0.5  */
    double beta1, beta2;    /* 0.9, 0.999 (torch.optim.Adam defaults) */
    double adam_eps;        /* 1e-5 morl/sample.py:31, warm_up.py:50 */
} pgm_ppo_hyper;

size_t pgm_ppo_workspace_bytes(int P, int S, int O, int A, int M, int cluster);
/* 0 for an unsupported hidden width */
size_t pgm_ppo_workspace_bytes_h(int P, int S, int O, int A, int M, int cluster, int hidden);
/* 0 for an unsupported hidden width or head */
size_t pgm_ppo_workspace_bytes_x(int P, int S, int O, int A, int M, int cluster, int hidden, int dist);

int pgm_ppo_update_f32(float *params, float *adam_m, float *adam_v, int32_t *adam_step,
                       const double *lr, const float *obs, size_t obs_task_stride,
                       const float *action, const float *logp_old, const float *value_old,
                       size_t value_task_stride, const float *returns, const float *adv,
                       const int32_t *perm, int perm_shared, int E, int B,
                       const pgm_ppo_hyper *hyper_host, float *losses, void *workspace,
                       size_t workspace_bytes, int cluster, int P, int S, int O, int A, int M,
                       void *stream);
int pgm_ppo_update_h_f32(float *params, float *adam_m, float *adam_v, int32_t *adam_step,
                         const double *lr, const float *obs, size_t obs_task_stride,
                         const float *action, const float *logp_old, const float *value_old,
                         size_t value_task_stride, const float *returns, const float *adv,
                         const int32_t *perm, int perm_shared, int E, int B,
                         const pgm_ppo_hyper *hyper_host, float *losses, void *workspace,
                         size_t workspace_bytes, int cluster, int P, int S, int O, int A, int M, int hidden,
                         void *stream);
int pgm_ppo_update_x_f32(float *params, float *adam_m, float *adam_v, int32_t *adam_step,
                         const double *lr, const float *obs, size_t obs_task_stride,
                         const float *action, const float *logp_old, const float *value_old,
                         size_t value_task_stride, const float *returns, const float *adv,
                         const int32_t *perm, int perm_shared, int E, int B,
                         const pgm_ppo_hyper *hyper_host, float *losses, void *workspace,
                         size_t workspace_bytes, int cluster, int P, int S, int O, int A, int M, int hidden,
                         int dist, void *stream);

/* Debug/verification aid: gradient of one minibatch (rows idx[0..mb)) of every task,
 * before clipping; grad [P, n_par], losses [P,3]. Same device code as pgm_ppo_update_f32. */
int pgm_ppo_grad_f32(const float *params, const float *obs, size_t obs_task_stride,
                     const float *action, const float *logp_old, const float *value_old,
                     size_t value_task_stride, const float *returns, const float *adv,
                     const int32_t *idx, int mb, const pgm_ppo_hyper *hyper_host, float *grad,
                     float *losses, void *workspace, size_t workspace_bytes, int cluster, int P,
                     int S, int O, int A, int M, void *stream);
int pgm_ppo_grad_h_f32(const float *params, const float *obs, size_t obs_task_stride,
                       const float *action, const float *logp_old, const float *value_old,
                       size_t value_task_stride, const float *returns, const float *adv,
                       const int32_t *idx, int mb, const pgm_ppo_hyper *hyper_host, float *grad,
                       float *losses, void *workspace, size_t workspace_bytes, int cluster, int P,
                       int S, int O, int A, int M, int hidden, void *stream);
int pgm_ppo_grad_x_f32(const float *params, const float *obs, size_t obs_task_stride,
                       const float *action, const float *logp_old, const float *value_old,
                       size_t value_task_stride, const float *returns, const float *adv,
                       const int32_t *idx, int mb, const pgm_ppo_hyper *hyper_host, float *grad,
                       float *losses, void *workspace, size_t workspace_bytes, int cluster, int P,
                       int S, int O, int A, int M, int hidden, int dist, void *stream);

/* ---------------------------------------------------------------------------
 * K4  batched fit of the hyperbolic prediction model (FLOAT64, one warp per fit).
 * Replaces the scipy.optimize.least_squares call of predict_hyperbolic
 * (morl/population_2d.py:56-108, morl/population_3d.py:51-103): bounded Trust Region Reflective,
 * loss='soft_l1', f_scale=20, start ones(4), bounds ([0,.1,-5,-500], ub), max_nfev 400.
 *   x, y, w [F,Kmax]: per fit the training weights / objective gains / Gaussian point weights,
 *   k_len [F] valid points per fit, ub [F,4] upper bounds (A_ub, 20, 5, 500)
 *   theta [F,4], status [F] (scipy codes 0..4), nfev [F], cost [F] out.
 * Kmax <= 2558 (one fit's data and Jacobians stay in one CTA's shared memory); F == 0 is a no-op.
 * The launch is asynchronous on `stream`; inputs must stay alive until it completes.
 */
int pgm_fit_hyperbolic_f64(const double *x, const double *y, const double *w, const int32_t *k_len,
                           const double *ub, double *theta, int32_t *status, int32_t *nfev, double *cost,
                           int F, int Kmax, void *stream);

/* ---------------------------------------------------------------------------
 * K4 front-end  training data of the prediction models (FLOAT64 compares, bit-identical to numpy).
 * Replaces the neighbourhood search and the widening loop of collect_nearest_data / predict_hyperbolic
 * (morl/population_2d.py:12-21,37-54, morl/population_3d.py:13-21,33-49) for a whole population in one launch.
 * Opt-graph as flat arrays: objs [n_nodes,M]; the E edges (source -> successor) ordered by source node, then by
 * successor (the order the reference walks opt_graph.succ): parent [E] = source node, edge_w [E,M] = successor weight
 * divided by its sum, edge_dy [E,M] = delta_objs of the successor.
 *
 * pgm_fit_neighbours_f64: per member b (opt-graph node node_ids[b]) the edges whose source node i satisfies
 *   |objs_k - objs_i| < |objs_k| * threshold in every objective, threshold doubled from 0.1 until those edges carry
 *   more than 3 successor weights that are pairwise >= 1e-5 apart (first-occurrence scan), or -- cap_threshold != 0, the
 *   3-objective variant -- until threshold >= 1, or until the threshold has overflowed to +inf (where the reference
 *   would loop forever). klen [n] = number of edges, steps [n] = doublings done (threshold = 0.1 * 2^steps, sigma =
 *   0.03 * 2^steps), edge_idx [n,E] = the edges in order (first klen[b] entries of row b).
 * pgm_fit_gather_f64: the K4 inputs of the n*M fits (fit f = b*M + objective): x, y [n*M,Kmax] = edge_w / edge_dy
 *   columns, ub [n*M,4] = (clip(max y - min y, 1, 500), 20, 5, 500) (population_2d.py:100-104), klen_f [n*M], and
 *   source [n,Kmax] = source node of every listed edge. Kmax >= max(klen). The Gaussian point weights
 *   exp(-(dist / sigma)^2 / 2) (population_2d.py:90-96) need numpy's exp bit for bit and are formed by the host from
 *   `source`.
 * M in 2..4. Per-member scratch of E*(8M+4) + 2*n_nodes bytes lives in shared memory up to 200 KB; larger opt-graphs need
 * a device workspace of pgm_fit_neighbours_workspace_bytes(...) bytes, 16-byte aligned (0 when shared memory suffices:
 * pass NULL then; a non-NULL workspace of n * scratch bytes is always used, which is how the tests reach that variant).
 */
size_t pgm_fit_neighbours_workspace_bytes(int n_nodes, int M, int E, int n);
int pgm_fit_neighbours_f64(const double *objs, int n_nodes, int M, const int32_t *parent, int E, const double *edge_w,
                           const int32_t *node_ids, int n, int cap_threshold, int32_t *klen, int32_t *steps,
                           int32_t *edge_idx, void *workspace, size_t workspace_bytes, void *stream);
int pgm_fit_gather_f64(const int32_t *edge_idx, const int32_t *klen, int n, int E, int M, const int32_t *parent,
                       const double *edge_w, const double *edge_dy, int Kmax, double *x, double *y, double *ub,
                       int32_t *klen_f, int32_t *source, void *stream);

/* ---------------------------------------------------------------------------
 * K5  Pareto filtering, exact hypervolume / sparsity, greedy candidate pick (all FLOAT64, and
 * bit-exact with the reference: same summation order, separate multiply / add, no FMA contraction).
 */

/* Replaces utils.get_ep_indices / check_dominated (morl/utils.py:24-39), the core of EP.update
 * (morl/ep.py:23-31). objs [n,M]; keep_idx [2n] int32: the first n_keep entries return the indices
 * of the non-dominated points with all objectives >= 0, ordered by ascending objective 0 (ties by
 * index); the upper n entries are scratch. n_keep [1] out (device). */
int pgm_ep_filter_f64(const double *objs, int n, int M, int32_t *keep_idx, int32_t *n_keep, void *stream);

/* Metrics of one point set, out[0] = hypervolume, out[1] = sparsity (device).
 *   M == 2: Population.compute_hypervolume / compute_sparsity (morl/population_2d.py:185-202):
 *           Pareto-filter, then closed forms on the front sorted by objective 0.
 *   M == 3: utils.compute_hypervolume (InnerHyperVolume, morl/hypervolume.py:41-153, round(hv,4))
 *           and utils.compute_sparsity (morl/utils.py:87-100) of the given front (all coords >= 0). Any size:
 *           fronts of up to 3 936 points are scored in one CTA's shared memory (52 bytes per point), larger ones
 *           on the global-memory path (see pgm_select_greedy_x_f64), with bit-identical results.
 *   M == 4: the same two functions (hypervolume.py:41-153 with its stored volumes / areas and area-reuse
 *           flags, utils.py:87-100); points with a negative coordinate are left out of the hypervolume as
 *           hypervolume.py:55-61 does. At most 2 202 points (the scorer's 93 bytes of shared memory per
 *           point within 200 KB), else an error.
 *   M >= 5 or M < 2: error.
 * workspace >= pgm_select_workspace_bytes(n, 1, M, 1). */
int pgm_front_metrics_f64(const double *pts, int n, int M, double *out, void *workspace,
                          size_t workspace_bytes, void *stream);
/* pgm_front_metrics_x_f64: the same with `flags` (PGM_SEL_GLOBAL forces the global-memory path at M = 3);
 * pgm_front_metrics_f64 is its flags = 0 case. workspace >= pgm_select_workspace_bytes_x(n, 1, M, 1, flags). */
int pgm_front_metrics_x_f64(const double *pts, int n, int M, int flags, double *out, void *workspace,
                            size_t workspace_bytes, void *stream);

/* Replaces evaluate_hv / evaluate_sparsity and the greedy loop of prediction_guided_selection
 * (morl/population_2d.py:207-224,264-302; morl/population_3d.py:206-214,294-331, update_ep
 * morl/utils.py:42-65). ep [E,M] = current archive front (ordered by objective 0); cand [C,M] =
 * predicted objectives of every candidate (sample, weight) pair.
 * Per round r < num_tasks: hv[r,c], sparsity[r,c] of EP_r + {cand c} for unmasked c (0 for masked),
 * best_ids[r] = first argmax of hv - alpha*sparsity (or -1 when no candidate is left, then stops);
 * EP_{r+1} = EP_r with the winner's prediction folded in. n_front [1] out: size of the final
 * virtual front, written to front_out [E+num_tasks, M] (both optional / may be NULL).
 * 3 objectives: every candidate of a round is scored on top of the round's shared base front (sorted lists, slice areas
 * and the head of the hypervolume sum are built once per round in the workspace). No size limit besides the workspace:
 * while the per-candidate scratch of 97 * (E + num_tasks + 1) bytes fits 200 KB of shared memory
 * (E + num_tasks + 1 <= 2 111) one CTA per candidate scores in shared memory; past that (or with PGM_SEL_GLOBAL) a grid
 * of at most 296 CTAs loops over the candidates with one scratch each in the workspace, about
 * 97 * min(C, 296) * (E + num_tasks + 1) bytes, and the base front is built by multi-CTA kernels. Both paths perform
 * the same float64 operations in the same order: their results are bit-identical.
 * 4 objectives (update_ep utils.py:42-65, hypervolume.py:41-153, compute_sparsity utils.py:87-100): one CTA per
 * candidate replays the reference's 4-D dimension sweep, stored level-2 volumes / areas and area-reuse flags included;
 * the per-candidate scratch of 93 * (E + num_tasks + 1) bytes must fit 200 KB of shared memory
 * (E + num_tasks + 1 <= 2 202), else an error. M >= 5: error.
 * pgm_select_workspace_bytes covers M = 2, 3 and 4. */
size_t pgm_select_workspace_bytes(int E, int C, int M, int num_tasks);
int pgm_select_greedy_f64(const double *ep, int E, const double *cand, int C, int M, double alpha,
                          int num_tasks, int32_t *best_ids, double *hv, double *sparsity,
                          double *front_out, int32_t *n_front, void *workspace, size_t workspace_bytes,
                          void *stream);

/* Selection flags of the _x entry points. PGM_SEL_GLOBAL: take the 3-objective global-memory path even where the
 * front fits shared memory (M = 3 only; other M: error), so both paths can be compared on one input. The entry points
 * without _x are the flags = 0 case: the path follows the front's size. */
#define PGM_SEL_GLOBAL 0x1
size_t pgm_select_workspace_bytes_x(int E, int C, int M, int num_tasks, int flags);
int pgm_select_greedy_x_f64(const double *ep, int E, const double *cand, int C, int M, double alpha,
                            int num_tasks, int flags, int32_t *best_ids, double *hv, double *sparsity,
                            double *front_out, int32_t *n_front, void *workspace, size_t workspace_bytes,
                            void *stream);

/* ---------------------------------------------------------------------------
 * K6  running normalisation of raw simulator output, all P x N environments of the shard in one launch per
 * environment step. Replaces, per task, VecNormalize.step_wait / reset
 * (externals/baselines/baselines/common/vec_env/vec_normalize.py:29-66), the a2c override of _obfilt
 * (a2c/envs.py:197-211) and RunningMeanStd.update (baselines/common/running_mean_std.py:10-31), so that the host
 * environment workers exchange only raw observations / actions with the GPU (SURVEY 8(f2)).
 *   raw_obs [P,N,O], raw_rew [P,N] (scalar reward; may be NULL), raw_obj [P,N,M] (may be NULL), done [P,N] (1 = episode ended)
 *   running moments, FP64, updated in place, bit-identical to numpy's:
 *     ob_mean/ob_var [P,O], ob_count [P]       (all NULL: observations pass through unnormalised)
 *     ret_acc [P,N] discounted return, ret_stat [P,3] = mean, var, count    (NULL: not tracked)
 *     obj_acc [P,N,M] discounted objective sums, obj_started [P] (0 until the first step),
 *     obj_mean/obj_var [P,M], obj_count [P]    (moments NULL: objectives pass through unnormalised)
 *   outputs, FP32: obs_out = clip((obs - mean) / sqrt(var + epsilon), +-clipob) for task p at obs_out + p * obs_task_stride
 *     ([N,O] rows, i.e. the slot of the rollout buffer K1 reads next); obj_out = clip(obj / sqrt(obj_var + epsilon), +-cliprew)
 *     at obj_out + p * obj_task_stride ([N,M]); mask_out [N] at mask_out + p * mask_task_stride = 1 - done.
 *   update = 0 freezes the observation moments (VecNormalize.eval()); reset = 1 is VecNormalize.reset(): only the
 *   observations are processed and ret_acc restarts at 0. N <= 128. */
int pgm_vecnorm_step_f64(const double *raw_obs, const double *raw_rew, const double *raw_obj, const uint8_t *done,
                         double *ob_mean, double *ob_var, double *ob_count, double *ret_acc, double *ret_stat,
                         double *obj_acc, int32_t *obj_started, double *obj_mean, double *obj_var, double *obj_count,
                         float *obs_out, size_t obs_task_stride, float *obj_out, size_t obj_task_stride,
                         float *mask_out, size_t mask_task_stride, double gamma, double clipob, double cliprew,
                         double epsilon, int update, int reset, int P, int N, int O, int M, void *stream);

/* K6 in rollout-slot mode (one captured CUDA graph per environment step, together with pgm_policy_step_f32): the staged
 * block holds the simulators' answer to the actions of time slot t-1; with ctl = {t, flags} in DEVICE memory (flags bit 1
 * set) the kernel writes the normalised next observation into slot t of obs_buf [P,(T+1)N,O], the normalised reward
 * vector into slot t-1 of rewards_buf [P,T,N,M], 1 - done into slot t of masks_buf [P,(T+1),N] and bad_in [P,N] into slot t
 * of bad_masks_buf (what RolloutStorage.insert stores, a2c/storage.py:50-62); flags bit 1 clear: no-op (t = 0).
 * Moments and arithmetic exactly as pgm_vecnorm_step_f64. */
int pgm_vecnorm_rollout_step_f64(const int32_t *ctl, const double *raw_obs, const double *raw_rew, const double *raw_obj,
                                 const uint8_t *done, const float *bad_in, double *ob_mean, double *ob_var,
                                 double *ob_count, double *ret_acc, double *ret_stat, double *obj_acc,
                                 int32_t *obj_started, double *obj_mean, double *obj_var, double *obj_count,
                                 float *obs_buf, size_t obs_task_stride, float *rewards_buf, size_t rewards_task_stride,
                                 float *masks_buf, size_t masks_task_stride, float *bad_masks_buf,
                                 size_t bad_masks_task_stride, double gamma, double clipob, double cliprew,
                                 double epsilon, int update, int P, int N, int O, int M, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PGMORL_B200_H */
