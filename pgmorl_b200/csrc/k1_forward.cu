// K1 -- population-batched actor-critic forward (rollout inference).
//
// Replaces the reference's per-step Policy.act / get_value / evaluate_actions
// (a2c/model.py:57-82 -> MLPBase.forward :237-246, DiagGaussian distributions.py:81-90,
// FixedNormal.log_probs :33-36), called 2048x per iteration from morl/mopg.py:103-135.
//
// One CTA = one task's parameter image resident in shared memory (both halves, ~49 KB at
// Walker2d dims) + a stream of 64-row observation chunks of that task. Algorithmic traffic per
// row: read O (+A eps) floats, write M + A + 1 floats; 21.8 kFLOP per row at Walker2d dims, so
// the kernel is FP32-FFMA bound, not HBM bound (SURVEY.md section 8(d)).
#include "net.cuh"

namespace pgm {

struct K1Args {
    const float *params, *obs, *eps;
    float *action, *value, *logp;
    int eps_shared, mode, P, rows_v, rows_a, chunks_per_cta;
    NetLayout L;
    // per-step mode (pgm_policy_step_f32): element strides between tasks (0 = dense), the device control word
    // {time slot t, sample flag}, the rollout slot the observation rows are copied to, and a dense copy of the actions
    size_t obs_ts, val_ts, act_ts, logp_ts;
    const int32_t *ctl;
    float *obs_copy; size_t obs_copy_ts;
    float *act_out;
    float *entropy;   // Categorical head, bulk mode: per-row entropy [P][rows_a] (may be null)
};

__host__ __device__ inline int k1_ldo(const NetLayout &L) { return (L.A > L.M ? L.A : L.M) | 1; }

// SPLIT = false: both halves resident (small networks). SPLIT = true: one half resident at a time, the CTA walks
// its chunks once per half (wide observations, e.g. Humanoid O = 376: one half's W1 alone is 97 KB).
__host__ inline size_t k1_smem_bytes(const NetLayout &L, int TM, bool split, int hw = H) {
    const int RC = 16 * TM;
    const size_t h0 = halfnet_smem_floats(L, 0, hw), h1 = halfnet_smem_floats(L, 1, hw);
    size_t f = split ? (h0 > h1 ? h0 : h1) : h0 + h1;
    f += (size_t)RC * L.ldw1;            // x
    f += 2 * (size_t)RC * (hw + 4);      // h1, h2
    f += 2 * (size_t)RC * k1_ldo(L);     // mean, value
    return f * sizeof(float);
}

// HW: hidden width (32, 64, 128; net.cuh RowTile). The body is shared by k1_forward_kernel (HW = 64) and
// k1_forward_h_kernel (HW = 32, 128).
// CAT: Categorical head (k1_forward_cat_kernel, every width): the head emits A = n logits, an action is one column holding
// the category index, eps holds n Exponential(1) draws per row.
template <int TM, bool SPLIT, int HW, bool CAT = false>
__device__ __forceinline__ void k1_forward_body(const K1Args a) {
    constexpr int RC = 16 * TM, LD = RowTile<HW>::LD;
    extern __shared__ __align__(16) float smem[];
    const NetLayout &L = a.L;
    const int tid = threadIdx.x, tr = tid & (RowTile<HW>::RT - 1), tc = tid >> RowTile<HW>::RT_LOG2;
    const int task = blockIdx.y;
    const int ldo = k1_ldo(L), ldx = L.ldw1;

    HalfNet actor, critic;
    float *p = halfnet_carve<HW>(actor, smem, L, 0);
    if (SPLIT) {
        float *pc = halfnet_carve<HW>(critic, smem, L, 1);  // same storage, used in a different pass
        p = p > pc ? p : pc;
    } else {
        p = halfnet_carve<HW>(critic, p, L, 1);
    }
    float *x = p;  p += RC * ldx;
    float *h1 = p; p += RC * LD;
    float *h2 = p; p += RC * LD;
    float *mu = p; p += RC * ldo;
    float *vo = p;

    const float *gp = a.params + (size_t)task * L.n_par;
    const int O = L.O, A = L.A, M = L.M;
    const int AC = CAT ? 1 : A;   // action columns
    // per-step mode: outputs land in time slot t of the rollout buffers (t and the sample flag come from device memory, so
    // that one captured CUDA graph serves every step); bulk mode: dense [P][rows][.] tensors
    const int slot_row = a.ctl ? __ldg(a.ctl) * a.rows_v : 0;
    const int rows_a = a.ctl ? ((__ldg(a.ctl + 1) & 1) ? a.rows_v : 0) : a.rows_a;
    const float *obs = a.obs + (size_t)task * (a.obs_ts ? a.obs_ts : (size_t)a.rows_v * O) + (a.obs_copy ? 0 : (size_t)slot_row * O);
    const float *eps = a.eps ? a.eps + (a.eps_shared ? 0 : (size_t)task * rows_a * A) : nullptr;
    float *action = a.action ? a.action + (size_t)task * (a.act_ts ? a.act_ts : (size_t)rows_a * AC) + (size_t)slot_row * AC : nullptr;
    float *value = a.value + (size_t)task * (a.val_ts ? a.val_ts : (size_t)a.rows_v * M) + (size_t)slot_row * M;
    float *logp = a.logp ? a.logp + (size_t)task * (a.logp_ts ? a.logp_ts : (size_t)rows_a) + slot_row : nullptr;
    float *obs_copy = a.obs_copy ? a.obs_copy + (size_t)task * a.obs_copy_ts + (size_t)slot_row * O : nullptr;
    float *act_out = a.act_out ? a.act_out + (size_t)task * a.rows_v * AC : nullptr;
    float *entropy = (CAT && a.entropy) ? a.entropy + (size_t)task * rows_a : nullptr;

    const int nchunks = (a.rows_v + RC - 1) / RC;
    const int c0 = blockIdx.x * a.chunks_per_cta;
    const int c1 = min(nchunks, c0 + a.chunks_per_cta);

    // pass 0 = critic (value for every row), pass 1 = actor (rows that carry an action); one pass if !SPLIT
    for (int pass = 0; pass < (SPLIT ? 2 : 1); ++pass) {
        if (SPLIT && pass == 1 && (long long)c0 * RC >= rows_a) break;      // no action rows in this CTA's range
        __syncthreads();
        if (!SPLIT) { halfnet_load<false, HW, !CAT>(actor, gp, L, 0); halfnet_load<false, HW, !CAT>(critic, gp, L, 1); }
        else if (pass == 0) halfnet_load<false, HW, !CAT>(critic, gp, L, 1);
        else halfnet_load<false, HW, !CAT>(actor, gp, L, 0);
        for (int i = tid; i < RC * ldx; i += NTHREADS) x[i] = 0.f;   // padded columns stay zero; loads touch k < O
        __syncthreads();
        for (int c = c0; c < c1; ++c) {
            const int row0 = c * RC;
            const int nrow = min(RC, a.rows_v - row0);
            const float *src = obs + (size_t)row0 * O;
            for (int i = tid; i < RC * O; i += NTHREADS) {         // coalesced copy of the dense [nrow][O] block
                int r = i / O, k = i - r * O;
                const float v = r < nrow ? __ldg(src + i) : 0.f;
                x[r * ldx + k] = v;
                if (obs_copy && r < nrow && pass == 0) obs_copy[(size_t)row0 * O + i] = v;   // observation -> its rollout slot
            }
            __syncthreads();
            if (!SPLIT || pass == 0) {
                half_forward<TM, HW>(x, ldx, critic, L, h1, h2, vo, ldo, tr, tc);
                for (int i = tid; i < nrow * M; i += NTHREADS) {
                    int r = i / M, m = i - r * M;
                    value[(size_t)row0 * M + i] = vo[r * ldo + m];
                }
            }
            const int nact = min(nrow, rows_a - row0);   // rows of this chunk that carry an action
            if ((!SPLIT || pass == 1) && nact > 0) {        // uniform across the CTA
                half_forward<TM, HW>(x, ldx, actor, L, h1, h2, mu, ldo, tr, tc);
                if (CAT) {
                    // thread per row over the n logits: max-subtracted log-sum-exp, the action, its log-prob, the entropy
                    for (int r = tid; r < nact; r += NTHREADS) {
                        const float *z = mu + r * ldo;
                        const size_t row = (size_t)row0 + r;
                        float mx = z[0];
                        for (int j = 1; j < A; ++j) mx = fmaxf(mx, z[j]);
                        float se = 0.f;
                        for (int j = 0; j < A; ++j) se += expf(z[j] - mx);
                        const float lse = mx + logf(se);
                        int act = 0;
                        if (a.mode == PGM_ACT_SAMPLE) {         // first argmax of p_j / q_j (torch.multinomial, one sample)
                            const float *q = eps + row * A;
                            float best = expf(z[0] - lse) / __ldg(q);
                            for (int j = 1; j < A; ++j) {
                                const float v = expf(z[j] - lse) / __ldg(q + j);
                                if (v > best) { best = v; act = j; }
                            }
                        } else if (a.mode == PGM_ACT_DETERMINISTIC) {   // first argmax of the logits (probs.argmax)
                            for (int j = 1; j < A; ++j) if (z[j] > z[act]) act = j;
                        } else {
                            act = min(max((int)__ldg(action + row), 0), A - 1);
                        }
                        if (a.mode != PGM_ACT_EVALUATE) action[row] = (float)act;
                        if (act_out) act_out[row] = (float)act;
                        logp[row] = z[act] - lse;
                        if (entropy) {
                            float h = 0.f;
                            for (int j = 0; j < A; ++j) { const float lpj = z[j] - lse; h -= expf(lpj) * lpj; }
                            entropy[row] = h;
                        }
                    }
                    __syncthreads();
                    continue;
                }
                // thread per (row, action dim): action + per-element log-density into mu[][] in place
                for (int i = tid; i < nact * A; i += NTHREADS) {
                    int r = i / A, d = i - r * A;
                    const float mean = mu[r * ldo + d];
                    const float ls = actor.ls[d];
                    const float sd = expf(ls);
                    float act;
                    if (a.mode == PGM_ACT_SAMPLE) act = fmaf(sd, __ldg(eps + (size_t)row0 * A + i), mean);
                    else if (a.mode == PGM_ACT_DETERMINISTIC) act = mean;
                    else act = __ldg(action + (size_t)row0 * A + i);
                    if (a.mode != PGM_ACT_EVALUATE) action[(size_t)row0 * A + i] = act;
                    if (act_out) act_out[(size_t)row0 * A + i] = act;
                    const float diff = act - mean;
                    // Normal.log_prob: -(x-mu)^2/(2 var) - log(std) - log(sqrt(2 pi))
                    mu[r * ldo + d] = -(diff * diff) / (2.f * sd * sd) - ls - 0.91893853320467274178f;
                }
                __syncthreads();
                for (int r = tid; r < nact; r += NTHREADS) {
                    float s = 0.f;
                    for (int d = 0; d < A; ++d) s += mu[r * ldo + d];
                    logp[row0 + r] = s;
                }
            }
            __syncthreads();
        }
    }
}

template <int TM, bool SPLIT>
__global__ void __launch_bounds__(NTHREADS, SPLIT ? 1 : 2) k1_forward_kernel(const K1Args a) { k1_forward_body<TM, SPLIT, H>(a); }

template <int TM, bool SPLIT, int HW>
__global__ void __launch_bounds__(NTHREADS, SPLIT ? 1 : 2) k1_forward_h_kernel(const K1Args a) { k1_forward_body<TM, SPLIT, HW>(a); }

template <int TM, bool SPLIT, int HW>
__global__ void __launch_bounds__(NTHREADS, SPLIT ? 1 : 2) k1_forward_cat_kernel(const K1Args a) {
    k1_forward_body<TM, SPLIT, HW, true>(a);
}

}  // namespace pgm
#include "k1_tc.cuh"
#include "k1_tcw.cuh"

using namespace pgm;

// bulk forward over trajectories on the tensor-core kernel (shapes it is instantiated for, enough rows to amortise the
// per-CTA weight-image setup); per-step inference (a few rows) stays on the FFMA kernel
static bool k1_tc_wanted(int O, int A, int M, int rows_v) {
    return ((O == 17 && A == 6 && M == 2) || (O == 11 && A == 3 && M == 3)) && rows_v >= 1024;
}

template <typename Kern>
static int k1_tc_launch(Kern kern, K1Args &a, int P, int O, cudaStream_t st) {
    int dev = 0, sms = 148;
    PGM_CUDA(cudaGetDevice(&dev));
    PGM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int ntiles = (a.rows_v + 127) / 128;
    int nblk = (sms + 2 * P - 1) / (2 * P);                 // CTAs per (task, half): fill the SMs once
    if (nblk > (ntiles + 1) / 2) nblk = (ntiles + 1) / 2;
    if (nblk < 1) nblk = 1;
    a.chunks_per_cta = ((ntiles + nblk - 1) / nblk + 1) / 2 * 2;   // whole pairs of tiles
    nblk = (ntiles + a.chunks_per_cta - 1) / a.chunks_per_cta;
    const size_t smem = k1t_smem_layout(O).total;
    PGM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<dim3(nblk, 2, P), K1T_THREADS, smem, st>>>(a);
    PGM_CUDA(cudaGetLastError());
    return PGM_OK;
}

// wide observations (Humanoid): one tile at a time, CTAs per (task, half) sized to fill the SMs once
static int k1_tcw_launch(K1Args &a, int P, cudaStream_t st) {
    int dev = 0, sms = 148;
    PGM_CUDA(cudaGetDevice(&dev));
    PGM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int ntiles = (a.rows_v + 127) / 128;
    int nblk = sms / (2 * P);
    if (nblk > ntiles) nblk = ntiles;
    if (nblk < 1) nblk = 1;
    a.chunks_per_cta = (ntiles + nblk - 1) / nblk;
    nblk = (ntiles + a.chunks_per_cta - 1) / a.chunks_per_cta;
    const size_t smem = k1w_smem_layout().total;
    PGM_CUDA(cudaFuncSetAttribute(k1_tcw_kernel<376, 17, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k1_tcw_kernel<376, 17, 2><<<dim3(nblk, 2, P), K1T_THREADS, smem, st>>>(a);
    PGM_CUDA(cudaGetLastError());
    return PGM_OK;
}

static int k1_ffma_launch(K1Args &a, int P, int rows_v, int O, int hidden, cudaStream_t stream);

extern "C" int pgm_policy_forward_x_f32(const float *params, const float *obs, const float *eps, int eps_shared,
                                        float *action, float *value, float *logp, float *entropy, int mode, int P,
                                        int rows_v, int rows_a, int O, int A, int M, int hidden, int dist, void *stream) {
    PGM_REQUIRE(params && obs && value, "pgm_policy_forward_f32: null params/obs/value");
    PGM_REQUIRE(P > 0 && rows_v > 0 && rows_a >= 0 && rows_a <= rows_v, "pgm_policy_forward_f32: bad row counts");
    PGM_REQUIRE(O > 0 && A > 0 && M > 0 && A <= 64 && M <= 16, "pgm_policy_forward_f32: unsupported dims O=%d A=%d M=%d", O, A, M);
    PGM_REQUIRE(hidden_supported(hidden), "pgm_policy_forward_f32: hidden width %d is not one of {32, 64, 128}", hidden);
    PGM_REQUIRE(dist_supported(dist), "pgm_policy_forward_f32: unknown action head %d", dist);
    const bool cat = dist == PGM_DIST_CATEGORICAL;
    PGM_REQUIRE(!cat || A <= CAT_MAX, "pgm_policy_forward_f32: a categorical head has 1..%d categories, got %d", CAT_MAX, A);
    PGM_REQUIRE(cat || !entropy, "pgm_policy_forward_f32: the per-row entropy output is for categorical heads only");
    PGM_REQUIRE(mode >= 0 && mode <= 2, "pgm_policy_forward_f32: bad mode %d", mode);
    if (rows_a > 0) {
        PGM_REQUIRE(action && logp, "pgm_policy_forward_f32: rows_a>0 needs action and logp");
        PGM_REQUIRE(mode != PGM_ACT_SAMPLE || eps, "pgm_policy_forward_f32: SAMPLE mode needs eps");
    }
    K1Args a;
    a.params = params; a.obs = obs; a.eps = eps; a.action = action; a.value = value; a.logp = logp;
    a.eps_shared = eps_shared; a.mode = mode; a.P = P; a.rows_v = rows_v; a.rows_a = rows_a;
    a.L = NetLayout(O, A, M, hidden, dist);
    a.obs_ts = a.val_ts = a.act_ts = a.logp_ts = 0; a.ctl = nullptr; a.obs_copy = nullptr; a.obs_copy_ts = 0; a.act_out = nullptr;
    a.entropy = entropy;
    // Categorical heads run on the FFMA kernel only: decided before the shape checks, which would otherwise send a
    // categorical policy whose (O, n, M) equals an instantiated Gaussian shape to the tensor-core kernels
    if (cat) return k1_ffma_launch(a, P, rows_v, O, hidden, (cudaStream_t)stream);
    // the tensor-core forwards are built for hidden width 64; other widths run on the FFMA kernel
    if (hidden == H && k1_tc_wanted(O, A, M, rows_v)) {
        if (O == 17) return k1_tc_launch(k1_tc_kernel<17, 6, 2>, a, P, O, (cudaStream_t)stream);
        return k1_tc_launch(k1_tc_kernel<11, 3, 3>, a, P, O, (cudaStream_t)stream);
    }
    if (hidden == H && O == 376 && A == 17 && M == 2 && rows_v >= 1024) return k1_tcw_launch(a, P, (cudaStream_t)stream);
    return k1_ffma_launch(a, P, rows_v, O, hidden, (cudaStream_t)stream);
}

extern "C" int pgm_policy_forward_h_f32(const float *params, const float *obs, const float *eps, int eps_shared,
                                        float *action, float *value, float *logp, int mode, int P, int rows_v,
                                        int rows_a, int O, int A, int M, int hidden, void *stream) {
    return pgm_policy_forward_x_f32(params, obs, eps, eps_shared, action, value, logp, nullptr, mode, P, rows_v, rows_a, O, A,
                                    M, hidden, PGM_DIST_GAUSSIAN, stream);
}

extern "C" int pgm_policy_forward_f32(const float *params, const float *obs, const float *eps, int eps_shared,
                                      float *action, float *value, float *logp, int mode, int P, int rows_v,
                                      int rows_a, int O, int A, int M, void *stream) {
    return pgm_policy_forward_h_f32(params, obs, eps, eps_shared, action, value, logp, mode, P, rows_v, rows_a, O, A, M, H,
                                    stream);
}

template <typename Kern>
static int k1_ffma_go(Kern kern, size_t &attr_done, const K1Args &a, dim3 grid, size_t smem, cudaStream_t stream) {
    if (attr_done < smem) {                                              // raise the dynamic shared-memory limit once per size
        PGM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done = smem;
    }
    kern<<<grid, NTHREADS, smem, stream>>>(a);
    return PGM_OK;
}

template <bool SPLIT>
static int k1_cat_go(int hidden, size_t &done, const K1Args &a, dim3 grid, size_t smem, cudaStream_t stream) {
    constexpr int TM = SPLIT ? 2 : 4;
    if (hidden == 32) return k1_ffma_go(k1_forward_cat_kernel<TM, SPLIT, 32>, done, a, grid, smem, stream);
    if (hidden == 128) return k1_ffma_go(k1_forward_cat_kernel<TM, SPLIT, 128>, done, a, grid, smem, stream);
    return k1_ffma_go(k1_forward_cat_kernel<TM, SPLIT, 64>, done, a, grid, smem, stream);
}

// FP32 FFMA kernel (per-step inference with a few rows, shapes without a tensor-core instantiation, hidden widths other
// than 64)
static int k1_ffma_launch(K1Args &a, int P, int rows_v, int O, int hidden, cudaStream_t stream) {
    const bool split = k1_smem_bytes(a.L, 4, false, hidden) > 110 * 1024;   // keep two CTAs per SM for small networks
    const int TM = split ? 2 : 4, RC = 16 * TM;
    const size_t smem = k1_smem_bytes(a.L, TM, split, hidden);
    PGM_REQUIRE(smem <= 227 * 1024, "pgm_policy_forward_f32: obs dim %d needs %zu B shared memory at hidden width %d", O, smem,
                hidden);
    static int sms = 0;                                                  // queried once: this launcher sits in per-step loops
    if (sms == 0) {
        int dev = 0;
        PGM_CUDA(cudaGetDevice(&dev));
        PGM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    }
    const int nchunks = (rows_v + RC - 1) / RC;
    const int slots = (split ? 1 : 2) * sms;            // resident CTAs
    int ctas_per_task = (slots + P - 1) / P;
    if (ctas_per_task > nchunks) ctas_per_task = nchunks;
    a.chunks_per_cta = (nchunks + ctas_per_task - 1) / ctas_per_task;
    ctas_per_task = (nchunks + a.chunks_per_cta - 1) / a.chunks_per_cta;
    dim3 grid(ctas_per_task, P);
    static size_t attr_done[2][3][2] = {};                               // [head][32 | 64 | 128][split]
    const bool cat = a.L.dist == PGM_DIST_CATEGORICAL;
    size_t &done = attr_done[cat][hidden == 32 ? 0 : (hidden == 64 ? 1 : 2)][split];
    int rc;
    if (cat) rc = split ? k1_cat_go<true>(hidden, done, a, grid, smem, stream) : k1_cat_go<false>(hidden, done, a, grid, smem, stream);
    else if (hidden == 32) rc = split ? k1_ffma_go(k1_forward_h_kernel<2, true, 32>, done, a, grid, smem, stream)
                                 : k1_ffma_go(k1_forward_h_kernel<4, false, 32>, done, a, grid, smem, stream);
    else if (hidden == 128) rc = split ? k1_ffma_go(k1_forward_h_kernel<2, true, 128>, done, a, grid, smem, stream)
                                       : k1_ffma_go(k1_forward_h_kernel<4, false, 128>, done, a, grid, smem, stream);
    else rc = split ? k1_ffma_go(k1_forward_kernel<2, true>, done, a, grid, smem, stream)
                    : k1_ffma_go(k1_forward_kernel<4, false>, done, a, grid, smem, stream);
    if (rc) return rc;
    PGM_CUDA(cudaGetLastError());
    return PGM_OK;
}

extern "C" int pgm_policy_step_x_f32(const float *params, const int32_t *ctl, const float *obs_stage, const float *eps,
                                     int eps_shared, float *obs_buf, size_t obs_task_stride, float *value_buf,
                                     size_t value_task_stride, float *action_buf, size_t action_task_stride, float *logp_buf,
                                     size_t logp_task_stride, float *act_out, int P, int N, int O, int A, int M, int hidden,
                                     int dist, void *stream) {
    PGM_REQUIRE(params && ctl && obs_buf && value_buf && action_buf && logp_buf && eps,
                "pgm_policy_step_f32: null pointer argument");
    PGM_REQUIRE(P > 0 && N > 0 && O > 0 && A > 0 && M > 0 && A <= 64 && M <= 16, "pgm_policy_step_f32: unsupported sizes");
    PGM_REQUIRE(hidden_supported(hidden), "pgm_policy_step_f32: hidden width %d is not one of {32, 64, 128}", hidden);
    PGM_REQUIRE(dist_supported(dist), "pgm_policy_step_f32: unknown action head %d", dist);
    PGM_REQUIRE(dist != PGM_DIST_CATEGORICAL || A <= CAT_MAX,
                "pgm_policy_step_f32: a categorical head has 1..%d categories, got %d", CAT_MAX, A);
    K1Args a;
    a.params = params; a.eps = eps; a.eps_shared = eps_shared; a.mode = PGM_ACT_SAMPLE; a.P = P; a.rows_v = N; a.rows_a = N;
    a.L = NetLayout(O, A, M, hidden, dist);
    a.ctl = ctl;
    if (obs_stage) {      // observations arrive in a dense staging block and are copied into their rollout slot by the kernel
        a.obs = obs_stage; a.obs_ts = 0; a.obs_copy = obs_buf; a.obs_copy_ts = obs_task_stride;
    } else {              // observations are already in the rollout slot (written there by K6)
        a.obs = obs_buf; a.obs_ts = obs_task_stride; a.obs_copy = nullptr; a.obs_copy_ts = 0;
    }
    a.value = value_buf; a.val_ts = value_task_stride; a.action = action_buf; a.act_ts = action_task_stride;
    a.logp = logp_buf; a.logp_ts = logp_task_stride; a.act_out = act_out; a.entropy = nullptr;
    return k1_ffma_launch(a, P, N, O, hidden, (cudaStream_t)stream);
}

extern "C" int pgm_policy_step_h_f32(const float *params, const int32_t *ctl, const float *obs_stage, const float *eps,
                                     int eps_shared, float *obs_buf, size_t obs_task_stride, float *value_buf,
                                     size_t value_task_stride, float *action_buf, size_t action_task_stride, float *logp_buf,
                                     size_t logp_task_stride, float *act_out, int P, int N, int O, int A, int M, int hidden,
                                     void *stream) {
    return pgm_policy_step_x_f32(params, ctl, obs_stage, eps, eps_shared, obs_buf, obs_task_stride, value_buf,
                                 value_task_stride, action_buf, action_task_stride, logp_buf, logp_task_stride, act_out, P, N,
                                 O, A, M, hidden, PGM_DIST_GAUSSIAN, stream);
}

extern "C" int pgm_policy_step_f32(const float *params, const int32_t *ctl, const float *obs_stage, const float *eps,
                                   int eps_shared, float *obs_buf, size_t obs_task_stride, float *value_buf,
                                   size_t value_task_stride, float *action_buf, size_t action_task_stride, float *logp_buf,
                                   size_t logp_task_stride, float *act_out, int P, int N, int O, int A, int M, void *stream) {
    return pgm_policy_step_h_f32(params, ctl, obs_stage, eps, eps_shared, obs_buf, obs_task_stride, value_buf,
                                 value_task_stride, action_buf, action_task_stride, logp_buf, logp_task_stride, act_out, P, N,
                                 O, A, M, H, stream);
}
