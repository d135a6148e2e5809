// K6 -- running observation / return / objective normalisation for every task of the shard, one launch per
// environment step (SURVEY 8(f2)). Replaces, per task, VecNormalize.step_wait / reset / _obfilt
// (externals/baselines/baselines/common/vec_env/vec_normalize.py:29-66, a2c/envs.py:197-211) and
// RunningMeanStd.update (baselines/common/running_mean_std.py:10-31): the host sends the RAW simulator output of
// all P x N environments, the kernel updates the FP64 running moments and writes the clipped, normalised
// observation straight into the rollout buffer slot K1 reads next, the normalised reward vector into the
// rewards slot and the termination mask -- the host never touches normalised data.
//
// FP64 in numpy's evaluation order with explicit round-to-nearest mul/add (no FMA contraction), so the running
// moments and the float32 observations are bit-identical to the reference's:
//   batch moments over the N envs (np.mean / np.var, axis 0) of an [N, W] block: rows added one after the other
//   when W >= 2; when W == 1 (O == 1 observations, M == 1 objectives) numpy collapses the C-contiguous [N, 1]
//   block into one contiguous 1-D reduction, which is the pairwise sum, as for the 1-D return vector (a plain loop
//   below 8 elements, 8 interleaved partial sums combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) from 8 to 128).
//   Clipping is np.clip's: a NaN stays NaN (a NaN or inf from a simulator shows up in the outputs, never as -clip).
// One CTA per task; threads stride over observation features, then over objectives; thread 0 owns the scalar
// return statistics and the sample counts.
#include "common.cuh"

namespace pgm {

struct K6Args {
    const double *raw_obs, *raw_rew, *raw_obj;
    const uint8_t *done;
    double *ob_mean, *ob_var, *ob_count;
    double *ret_acc, *ret_stat;
    double *obj_acc, *obj_mean, *obj_var, *obj_count;
    int32_t *obj_started;
    float *obs_out, *obj_out, *mask_out;
    size_t obs_ts, obj_ts, mask_ts;
    double gamma, clipob, cliprew, epsilon;
    int update, reset, P, N, O, M;
    // rollout-slot mode (pgm_vecnorm_rollout_step_f64): outputs are whole rollout buffers and the time slot comes from
    // the device control word {t, flags}; flags bit 1 clear = nothing to normalise this step (t = 0)
    const int32_t *ctl;
    const float *bad_in;
    float *bad_out;
    size_t bad_ts;
};

// update_mean_var_count_from_moments (running_mean_std.py:20-31), same operation order
__device__ __forceinline__ void rms_update(double &mean, double &var, double count, double bmean, double bvar, double bcount) {
    const double delta = __dsub_rn(bmean, mean);
    const double tot = __dadd_rn(count, bcount);
    const double new_mean = __dadd_rn(mean, __ddiv_rn(__dmul_rn(delta, bcount), tot));
    const double m_a = __dmul_rn(var, count), m_b = __dmul_rn(bvar, bcount);
    const double m2 = __dadd_rn(__dadd_rn(m_a, m_b),
                                __ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(delta, delta), count), bcount), tot));
    mean = new_mean;
    var = __ddiv_rn(m2, tot);
}

// np.clip(x, -c, c): comparisons, so a NaN passes through (fmin / fmax would return the bound) and -0.0 stays -0.0
__device__ __forceinline__ double clipd(double x, double c) { return x < -c ? -c : (x > c ? c : x); }

// np.add.reduce of n <= 128 doubles at(0..n-1), starting from its identity 0.0: one after the other when `rows` is set
// (the rows of a C-contiguous [n, w >= 2] block), numpy's pairwise sum of a contiguous 1-D block otherwise
// (numpy/_core/src/umath/loops_utils.h.src)
template <typename F>
__device__ __forceinline__ double np_add_reduce(F at, int n, bool rows) {
    if (rows || n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; ++i) res = __dadd_rn(res, at(i));
        return res;
    }
    double r[8];
    for (int j = 0; j < 8; ++j) r[j] = at(j);
    int i = 8;
    for (; i < n - (n % 8); i += 8)
        for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], at(i + j));
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, at(i));
    return __dadd_rn(0.0, res);
}

// (np.mean(x, axis=0)[j], np.var(x, axis=0)[j]) of a C-contiguous [n, w] block. numpy collapses a width-1 block into
// one contiguous 1-D reduction (pairwise); wider blocks add their rows one after the other.
__device__ __forceinline__ void np_col_moments(const double *x, int n, int w, int j, double &bmean, double &bvar) {
    const double dn = (double)n;
    const auto col = [&](int i) { return x[(size_t)i * w + j]; };
    const double m = __ddiv_rn(np_add_reduce(col, n, w > 1), dn);
    bmean = m;
    bvar = __ddiv_rn(np_add_reduce([&](int i) { const double d = __dsub_rn(col(i), m); return __dmul_rn(d, d); }, n, w > 1), dn);
}

__global__ void __launch_bounds__(128) k6_vecnorm_kernel(K6Args a) {
    const int p = blockIdx.x, tid = threadIdx.x, N = a.N, O = a.O, M = a.M;
    const double dN = (double)N;
    if (a.ctl) {      // the staged block holds the simulators' answer to the actions of slot t-1
        if (!(__ldg(a.ctl + 1) & 2)) return;
        const int t = __ldg(a.ctl);
        a.obs_out += (size_t)t * N * O;               // next observation          -> slot t   (storage.py:51)
        a.obj_out += (size_t)(t - 1) * N * M;         // reward vector of the step -> slot t-1 (storage.py:57)
        a.mask_out += (size_t)t * N;                  // masks / bad_masks         -> slot t   (storage.py:58-59)
        if (a.bad_out)
            for (int n = tid; n < N; n += blockDim.x) a.bad_out[(size_t)p * a.bad_ts + (size_t)t * N + n] = a.bad_in[(size_t)p * N + n];
    }

    // ---- observations: _obfilt (a2c/envs.py:202-211) ----
    {
        const double *x = a.raw_obs + (size_t)p * N * O;
        float *out = a.obs_out + (size_t)p * a.obs_ts;
        const bool stats = a.ob_mean != nullptr;
        const double count = stats ? a.ob_count[p] : 0.0;
        for (int j = tid; j < O; j += blockDim.x) {
            double mean = 0.0, var = 1.0;
            if (stats) {
                mean = a.ob_mean[(size_t)p * O + j]; var = a.ob_var[(size_t)p * O + j];
                if (a.update) {
                    double bmean, bvar;
                    np_col_moments(x, N, O, j, bmean, bvar);
                    rms_update(mean, var, count, bmean, bvar, dN);
                    a.ob_mean[(size_t)p * O + j] = mean; a.ob_var[(size_t)p * O + j] = var;
                }
            }
            const double sd = sqrt(__dadd_rn(var, a.epsilon));
            for (int n = 0; n < N; ++n) {
                const double xv = x[(size_t)n * O + j];
                out[(size_t)n * O + j] = (float)(stats ? clipd(__ddiv_rn(__dsub_rn(xv, mean), sd), a.clipob) : xv);
            }
        }
        __syncthreads();                       // every feature used the old count
        if (tid == 0 && stats && a.update) a.ob_count[p] = __dadd_rn(count, dN);
    }
    if (a.reset) {                             // VecNormalize.reset (vec_normalize.py:62-65): returns restart, obj keeps running
        if (a.ret_acc) for (int n = tid; n < N; n += blockDim.x) a.ret_acc[(size_t)p * N + n] = 0.0;
        return;
    }

    // ---- objectives (vec_normalize.py:33-37, 46-49, 52-53) ----
    if (a.raw_obj) {
        const double *o = a.raw_obj + (size_t)p * N * M;
        double *acc = a.obj_acc + (size_t)p * N * M;
        const bool started = a.obj_started[p] != 0;
        const bool stats = a.obj_mean != nullptr;
        const double count = stats ? a.obj_count[p] : 0.0;
        for (int m = tid; m < M; m += blockDim.x) {
            for (int n = 0; n < N; ++n) {
                const double v = o[(size_t)n * M + m];
                acc[(size_t)n * M + m] = started ? __dadd_rn(__dmul_rn(acc[(size_t)n * M + m], a.gamma), v) : v;
            }
            double sd = 1.0;
            if (stats) {
                double mean = a.obj_mean[(size_t)p * M + m], var = a.obj_var[(size_t)p * M + m];
                double bmean, bvar;
                np_col_moments(acc, N, M, m, bmean, bvar);
                rms_update(mean, var, count, bmean, bvar, dN);
                a.obj_mean[(size_t)p * M + m] = mean; a.obj_var[(size_t)p * M + m] = var;
                sd = sqrt(__dadd_rn(var, a.epsilon));
            }
            float *out = a.obj_out + (size_t)p * a.obj_ts;
            for (int n = 0; n < N; ++n) {
                const double v = o[(size_t)n * M + m];
                out[(size_t)n * M + m] = (float)(stats ? clipd(__ddiv_rn(v, sd), a.cliprew) : v);
                if (a.done[(size_t)p * N + n]) acc[(size_t)n * M + m] = 0.0;
            }
        }
        __syncthreads();
        if (tid == 0) {
            a.obj_started[p] = 1;
            if (stats) a.obj_count[p] = __dadd_rn(count, dN);
        }
    }

    // ---- scalar return statistics (vec_normalize.py:31, 42-44, 51) and termination masks ----
    if (tid == 0 && a.ret_acc && a.raw_rew) {
        double *ret = a.ret_acc + (size_t)p * N;
        const double *rw = a.raw_rew + (size_t)p * N;
        for (int n = 0; n < N; ++n) ret[n] = __dadd_rn(__dmul_rn(ret[n], a.gamma), rw[n]);
        if (a.ret_stat) {
            double *st = a.ret_stat + (size_t)p * 3;
            const double bmean = __ddiv_rn(np_add_reduce([&](int i) { return ret[i]; }, N, false), dN);
            const double bvar = __ddiv_rn(np_add_reduce([&](int i) { const double d = __dsub_rn(ret[i], bmean); return __dmul_rn(d, d); }, N, false), dN);
            double mean = st[0], var = st[1];
            rms_update(mean, var, st[2], bmean, bvar, dN);
            st[0] = mean; st[1] = var; st[2] = __dadd_rn(st[2], dN);
        }
        for (int n = 0; n < N; ++n) if (a.done[(size_t)p * N + n]) ret[n] = 0.0;
    }
    if (a.mask_out)
        for (int n = tid; n < N; n += blockDim.x) a.mask_out[(size_t)p * a.mask_ts + n] = a.done[(size_t)p * N + n] ? 0.f : 1.f;
}

}  // namespace pgm

using namespace pgm;

extern "C" int pgm_vecnorm_step_f64(const double *raw_obs, const double *raw_rew, const double *raw_obj, const uint8_t *done,
                                    double *ob_mean, double *ob_var, double *ob_count, double *ret_acc, double *ret_stat,
                                    double *obj_acc, int32_t *obj_started, double *obj_mean, double *obj_var, double *obj_count,
                                    float *obs_out, size_t obs_task_stride, float *obj_out, size_t obj_task_stride,
                                    float *mask_out, size_t mask_task_stride, double gamma, double clipob, double cliprew,
                                    double epsilon, int update, int reset, int P, int N, int O, int M, void *stream) {
    PGM_REQUIRE(P >= 1 && N >= 1 && N <= 128 && O >= 1 && M >= 0, "vecnorm: bad sizes P=%d N=%d O=%d M=%d (N <= 128)", P, N, O, M);
    PGM_REQUIRE(raw_obs && obs_out, "vecnorm: raw_obs / obs_out must not be NULL");
    PGM_REQUIRE(reset || done, "vecnorm: done flags are required for a step");
    PGM_REQUIRE((ob_mean == nullptr) == (ob_var == nullptr) && (ob_mean == nullptr) == (ob_count == nullptr),
                "vecnorm: ob_mean / ob_var / ob_count go together");
    PGM_REQUIRE((obj_mean == nullptr) == (obj_var == nullptr) && (obj_mean == nullptr) == (obj_count == nullptr),
                "vecnorm: obj_mean / obj_var / obj_count go together");
    PGM_REQUIRE(reset || !raw_obj || (obj_acc && obj_started && obj_out && M >= 1), "vecnorm: objective buffers missing");
    K6Args a;
    a.raw_obs = raw_obs; a.raw_rew = raw_rew; a.raw_obj = reset ? nullptr : raw_obj; a.done = done;
    a.ob_mean = ob_mean; a.ob_var = ob_var; a.ob_count = ob_count; a.ret_acc = ret_acc; a.ret_stat = ret_stat;
    a.obj_acc = obj_acc; a.obj_mean = obj_mean; a.obj_var = obj_var; a.obj_count = obj_count; a.obj_started = obj_started;
    a.obs_out = obs_out; a.obj_out = obj_out; a.mask_out = reset ? nullptr : mask_out;
    a.obs_ts = obs_task_stride; a.obj_ts = obj_task_stride; a.mask_ts = mask_task_stride;
    a.gamma = gamma; a.clipob = clipob; a.cliprew = cliprew; a.epsilon = epsilon;
    a.update = update; a.reset = reset; a.P = P; a.N = N; a.O = O; a.M = M;
    a.ctl = nullptr; a.bad_in = nullptr; a.bad_out = nullptr; a.bad_ts = 0;
    k6_vecnorm_kernel<<<P, 128, 0, (cudaStream_t)stream>>>(a);
    PGM_CUDA(cudaGetLastError());
    return PGM_OK;
}

extern "C" int pgm_vecnorm_rollout_step_f64(const int32_t *ctl, const double *raw_obs, const double *raw_rew, const double *raw_obj,
                                            const uint8_t *done, const float *bad_in, double *ob_mean, double *ob_var,
                                            double *ob_count, double *ret_acc, double *ret_stat, double *obj_acc,
                                            int32_t *obj_started, double *obj_mean, double *obj_var, double *obj_count,
                                            float *obs_buf, size_t obs_task_stride, float *rewards_buf, size_t rewards_task_stride,
                                            float *masks_buf, size_t masks_task_stride, float *bad_masks_buf,
                                            size_t bad_masks_task_stride, double gamma, double clipob, double cliprew,
                                            double epsilon, int update, int P, int N, int O, int M, void *stream) {
    PGM_REQUIRE(P >= 1 && N >= 1 && N <= 128 && O >= 1 && M >= 1, "vecnorm: bad sizes P=%d N=%d O=%d M=%d (N <= 128)", P, N, O, M);
    PGM_REQUIRE(ctl && raw_obs && raw_obj && done && obs_buf && rewards_buf && masks_buf && obj_acc && obj_started,
                "vecnorm (rollout step): null pointer argument");
    PGM_REQUIRE((bad_in == nullptr) == (bad_masks_buf == nullptr), "vecnorm (rollout step): bad_in / bad_masks_buf go together");
    PGM_REQUIRE((ob_mean == nullptr) == (ob_var == nullptr) && (ob_mean == nullptr) == (ob_count == nullptr),
                "vecnorm: ob_mean / ob_var / ob_count go together");
    PGM_REQUIRE((obj_mean == nullptr) == (obj_var == nullptr) && (obj_mean == nullptr) == (obj_count == nullptr),
                "vecnorm: obj_mean / obj_var / obj_count go together");
    K6Args a;
    a.raw_obs = raw_obs; a.raw_rew = raw_rew; a.raw_obj = raw_obj; a.done = done;
    a.ob_mean = ob_mean; a.ob_var = ob_var; a.ob_count = ob_count; a.ret_acc = ret_acc; a.ret_stat = ret_stat;
    a.obj_acc = obj_acc; a.obj_mean = obj_mean; a.obj_var = obj_var; a.obj_count = obj_count; a.obj_started = obj_started;
    a.obs_out = obs_buf; a.obj_out = rewards_buf; a.mask_out = masks_buf;
    a.obs_ts = obs_task_stride; a.obj_ts = rewards_task_stride; a.mask_ts = masks_task_stride;
    a.gamma = gamma; a.clipob = clipob; a.cliprew = cliprew; a.epsilon = epsilon;
    a.update = update; a.reset = 0; a.P = P; a.N = N; a.O = O; a.M = M;
    a.ctl = ctl; a.bad_in = bad_in; a.bad_out = bad_masks_buf; a.bad_ts = bad_masks_task_stride;
    k6_vecnorm_kernel<<<P, 128, 0, (cudaStream_t)stream>>>(a);
    PGM_CUDA(cudaGetLastError());
    return PGM_OK;
}
