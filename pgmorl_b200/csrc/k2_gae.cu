// K2 -- vector-reward returns + weight-scalarised, normalised advantage.
//
// Replaces RolloutStorage.compute_returns (a2c/storage.py:77-116, all four branches of use_gae x
// use_proper_time_limits) and the PPO.update preamble (a2c/algo/ppo.py:43-56) with
// WeightedSumScalarization.evaluate (morl/scalarization_methods.py:28-29).
//
// Every branch of the reference, per env column n and objective m, going backwards in t, is the
// affine map g_t = a_t * g_{t+1} + d_t (m = mask_{t+1}, b = bad_{t+1}, delta_t = r_t + gamma*V_{t+1}*m - V_t):
//     MODE                     a_t           d_t                   g at t = T   ret_t     raw advantage
//     GAE | PROPER_TIME_LIMITS gamma*lam*m*b delta_t * b           0            g + V_t   g
//     PROPER_TIME_LIMITS       gamma*m*b     r_t*b + (1 - b)*V_t   bootstrap    g         g - V_t
//     GAE                      gamma*lam*m   delta_t               0            g + V_t   g
//     (none: n-step returns)   gamma*m       r_t                   bootstrap    g         g - V_t
// The bootstrap is `boot` [P,N,M], or value row T when boot is NULL. MODE is a template parameter, so the
// first row compiles to exactly the instructions it had before the other branches existed.
// One CTA per task, one warp per env column: the warp walks T in blocks of 32 steps (lane = step,
// so global loads of a block are contiguous across the CTA's warps), composes the 32 affine maps
// with a shuffle scan and chains blocks through a carried g. The scalarised raw advantage
// sum_m w_m * sqrt(var_m + 1e-8) * g_{t,m} is written to `adv`, then the CTA normalises it with
// the mean and unbiased std over all T*N samples (two-pass, block reductions by warp shuffles).
//
// Streaming kernel: 36 B per env-step at M = 2 (read r, V, masks; write ret, adv) -> HBM bound.
#include "common.cuh"

namespace pgm {

constexpr int K2_MAXM = 8;

template <int MODE>
__device__ __forceinline__ float k2_boot(const float *__restrict__ boot, const float *__restrict__ value, int task, int T,
                                         int N, int M, int n, int m) {
    if (MODE & PGM_RET_GAE) return 0.f;
    return boot ? __ldg(boot + ((size_t)task * N + n) * M + m) : __ldg(value + ((size_t)T * N + n) * M + m);
}

// d_t of step t for one objective (table above); mk, bd = mask / bad mask of slot t+1, v = V_t, vnp -> V_{t+1}
template <int MODE>
__device__ __forceinline__ float k2_d(float r, float v, const float *__restrict__ vnp, float gamma, float mk, float bd) {
    if (MODE == (PGM_RET_GAE | PGM_RET_PROPER_TIME_LIMITS)) return (r + gamma * __ldg(vnp) * mk - v) * bd;
    if (MODE == PGM_RET_GAE) return r + gamma * __ldg(vnp) * mk - v;
    if (MODE == PGM_RET_PROPER_TIME_LIMITS) return fmaf(r, bd, (1.f - bd) * v);
    return r;
}

template <int M, int MODE>
__global__ void __launch_bounds__(1024) k2_gae_kernel(const float *__restrict__ rewards, const float *__restrict__ value,
                                                      const float *__restrict__ boot,
                                                      const float *__restrict__ masks, const float *__restrict__ bad_masks,
                                                      const float *__restrict__ weights, const float *__restrict__ obj_var,
                                                      float gamma, float lam, float *__restrict__ returns,
                                                      float *__restrict__ adv, int T, int N) {
    constexpr bool GAE = (MODE & PGM_RET_GAE) != 0, PTL = (MODE & PGM_RET_PROPER_TIME_LIMITS) != 0;
    __shared__ float red[34];
    const int task = blockIdx.x;
    const int lane = threadIdx.x & 31, n = threadIdx.x >> 5;   // warp n <-> env column n
    rewards += (size_t)task * T * N * M;
    value += (size_t)task * (T + 1) * N * M;
    masks += (size_t)task * (T + 1) * N;
    bad_masks += (size_t)task * (T + 1) * N;
    returns += (size_t)task * T * N * M;
    const bool do_adv = (weights != nullptr) && (adv != nullptr);
    if (do_adv) adv += (size_t)task * T * N;

    float ws[M];
#pragma unroll
    for (int m = 0; m < M; ++m) {
        float s = obj_var ? sqrtf(__ldg(obj_var + task * M + m) + 1e-8f) : 1.f;
        ws[m] = do_adv ? __ldg(weights + task * M + m) * s : 0.f;
    }
    const float gl = GAE ? gamma * lam : gamma;
    float carry[M];
#pragma unroll
    for (int m = 0; m < M; ++m) carry[m] = k2_boot<MODE>(boot, value, task, T, N, M, n, m);
    float psum = 0.f;

    const int nblk = (T + 31) / 32;
    for (int blk = nblk - 1; blk >= 0; --blk) {
        const int t = blk * 32 + lane;
        const bool ok = t < T;
        float a = 1.f, d[M], v[M];
#pragma unroll
        for (int m = 0; m < M; ++m) { d[m] = 0.f; v[m] = 0.f; }
        if (ok) {
            const float mk = __ldg(masks + (size_t)(t + 1) * N + n);
            const float bd = PTL ? __ldg(bad_masks + (size_t)(t + 1) * N + n) : 1.f;
            a = PTL ? gl * mk * bd : gl * mk;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                const float r = __ldg(rewards + ((size_t)t * N + n) * M + m);
                v[m] = __ldg(value + ((size_t)t * N + n) * M + m);
                d[m] = k2_d<MODE>(r, v[m], value + ((size_t)(t + 1) * N + n) * M + m, gamma, mk, bd);
            }
        }
        // suffix composition over lanes: after the scan, g_t = d + a * carry where (a, d) is the
        // composition of the maps of steps t, t+1, ..., end of block
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const float an = __shfl_down_sync(0xffffffffu, a, off);
            float dn[M];
#pragma unroll
            for (int m = 0; m < M; ++m) dn[m] = __shfl_down_sync(0xffffffffu, d[m], off);
            if (lane + off < 32) {
#pragma unroll
                for (int m = 0; m < M; ++m) d[m] = fmaf(a, dn[m], d[m]);
                a *= an;
            }
        }
        float g[M], s = 0.f;
#pragma unroll
        for (int m = 0; m < M; ++m) {
            g[m] = fmaf(a, carry[m], d[m]);
            s = fmaf(ws[m], GAE ? g[m] : g[m] - v[m], s);
        }
        if (ok) {
#pragma unroll
            for (int m = 0; m < M; ++m) returns[((size_t)t * N + n) * M + m] = GAE ? g[m] + v[m] : g[m];
            if (do_adv) { adv[(size_t)t * N + n] = s; psum += s; }
        }
#pragma unroll
        for (int m = 0; m < M; ++m) carry[m] = __shfl_sync(0xffffffffu, g[m], 0);
    }
    if (!do_adv) return;

    // normalise: (adv - mean) / (unbiased std + 1e-5) over the task's T*N samples
    const int S = T * N;
    const float mean = block_sum(psum, red) / (float)S;   // block_sum syncs -> raw adv visible CTA-wide
    float q = 0.f;
    for (int i = threadIdx.x; i < S; i += blockDim.x) { const float c = adv[i] - mean; q = fmaf(c, c, q); }
    const float var = block_sum(q, red) / (float)(S - 1);
    const float inv = 1.f / (sqrtf(var) + 1e-5f);
    for (int i = threadIdx.x; i < S; i += blockDim.x) adv[i] = (adv[i] - mean) * inv;
}

// Segmented variant for small populations (round 2): with one warp per env column a task of T = 2048 steps is a chain of
// 64 dependent load -> scan -> carry rounds on 4 warps (75 us at 6 tasks: 22 GB/s). Here the CTA has 32 warps; warp w owns
// env column w % N and segment w / N of the time axis (NSEG = 32 / N segments of SEG steps). Phase 1: every warp walks
// ITS segment backwards with a zero carry and keeps, per step, the local solution g_loc and the multiplier A that the
// unknown right-hand carry is scaled by (g_t = g_loc_t + A_t * G_in), both in shared memory. Phase 2: N*M threads chain the
// NSEG segment maps (a handful of steps). Phase 3: every warp finishes its segment. The dependent chain shrinks from T/32
// to T/(32 NSEG) + NSEG rounds.
template <int M, int MODE>
__global__ void __launch_bounds__(1024) k2_gae_seg_kernel(const float *__restrict__ rewards, const float *__restrict__ value,
                                                          const float *__restrict__ boot,
                                                          const float *__restrict__ masks, const float *__restrict__ bad_masks,
                                                          const float *__restrict__ weights, const float *__restrict__ obj_var,
                                                          float gamma, float lam, float *__restrict__ returns,
                                                          float *__restrict__ adv, int T, int N, int NSEG, int SEG) {
    constexpr bool GAE = (MODE & PGM_RET_GAE) != 0, PTL = (MODE & PGM_RET_PROPER_TIME_LIMITS) != 0;
    extern __shared__ float sm[];                 // A[T*N] | Gloc[M][T*N]
    __shared__ float red[34];
    __shared__ float segA[32], segG[32][M], segIn[32][M];     // per warp (= column, segment)
    const int task = blockIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int n = w % N, sg = w / N;
    const bool active = sg < NSEG;
    const int S = T * N;
    float *Ash = sm, *Gsh = sm + S;
    rewards += (size_t)task * T * N * M;
    value += (size_t)task * (T + 1) * N * M;
    masks += (size_t)task * (T + 1) * N;
    bad_masks += (size_t)task * (T + 1) * N;
    returns += (size_t)task * T * N * M;
    const bool do_adv = (weights != nullptr) && (adv != nullptr);
    if (do_adv) adv += (size_t)task * T * N;

    float ws[M];
#pragma unroll
    for (int m = 0; m < M; ++m) {
        float s = obj_var ? sqrtf(__ldg(obj_var + task * M + m) + 1e-8f) : 1.f;
        ws[m] = do_adv ? __ldg(weights + task * M + m) * s : 0.f;
    }
    const float gl = GAE ? gamma * lam : gamma;
    const int t0 = sg * SEG, t1 = min(T, t0 + SEG);          // my segment [t0, t1)

    // ---- phase 1: local solution of my segment (carry 0 from the right) ----
    if (active) {
        float carry[M], cA = 1.f;
#pragma unroll
        for (int m = 0; m < M; ++m) carry[m] = 0.f;
        for (int b0 = t0 + ((max(t1 - t0, 1) - 1) / 32) * 32; b0 >= t0 && t1 > t0; b0 -= 32) {
            const int t = b0 + lane;
            const bool ok = t < t1;
            float a = 1.f, d[M];
#pragma unroll
            for (int m = 0; m < M; ++m) d[m] = 0.f;
            if (ok) {
                const float mk = __ldg(masks + (size_t)(t + 1) * N + n);
                const float bd = PTL ? __ldg(bad_masks + (size_t)(t + 1) * N + n) : 1.f;
                a = PTL ? gl * mk * bd : gl * mk;
#pragma unroll
                for (int m = 0; m < M; ++m) {
                    const float r = __ldg(rewards + ((size_t)t * N + n) * M + m);
                    const float v = __ldg(value + ((size_t)t * N + n) * M + m);
                    d[m] = k2_d<MODE>(r, v, value + ((size_t)(t + 1) * N + n) * M + m, gamma, mk, bd);
                }
            }
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {          // suffix composition over the lanes of the block
                const float an = __shfl_down_sync(0xffffffffu, a, off);
                float dn[M];
#pragma unroll
                for (int m = 0; m < M; ++m) dn[m] = __shfl_down_sync(0xffffffffu, d[m], off);
                if (lane + off < 32) {
#pragma unroll
                    for (int m = 0; m < M; ++m) d[m] = fmaf(a, dn[m], d[m]);
                    a *= an;
                }
            }
            float g[M];
            const float At = a * cA;
#pragma unroll
            for (int m = 0; m < M; ++m) g[m] = fmaf(a, carry[m], d[m]);
            if (ok) {
                Ash[(size_t)t * N + n] = At;
#pragma unroll
                for (int m = 0; m < M; ++m) Gsh[(size_t)m * S + (size_t)t * N + n] = g[m];
            }
#pragma unroll
            for (int m = 0; m < M; ++m) carry[m] = __shfl_sync(0xffffffffu, g[m], 0);
            cA = __shfl_sync(0xffffffffu, At, 0);
        }
        if (lane == 0) {
            segA[w] = cA;
#pragma unroll
            for (int m = 0; m < M; ++m) segG[w][m] = carry[m];
        }
    }
    __syncthreads();
    // ---- phase 2: chain the segment maps from the right: G_in(sg) = g at the first step of segment sg + 1; the last
    //      segment's right-hand carry is 0 (GAE) or the bootstrap (n-step) ----
    if (threadIdx.x < N * M) {
        const int nn = threadIdx.x / M, m = threadIdx.x % M;
        float G = k2_boot<MODE>(boot, value, task, T, N, M, nn, m);
        for (int q = NSEG - 1; q >= 0; --q) {
            const int ww = q * N + nn;
            segIn[ww][m] = G;
            G = fmaf(segA[ww], G, segG[ww][m]);
        }
    }
    __syncthreads();
    // ---- phase 3: finish my segment: g = g_loc + A * G_in; returns, scalarised raw advantage ----
    float psum = 0.f;
    if (active) {
        float gin[M];
#pragma unroll
        for (int m = 0; m < M; ++m) gin[m] = segIn[w][m];
        for (int t = t0 + lane; t < t1; t += 32) {
            const float At = Ash[(size_t)t * N + n];
            float s = 0.f;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                const float g = fmaf(At, gin[m], Gsh[(size_t)m * S + (size_t)t * N + n]);
                const float v = __ldg(value + ((size_t)t * N + n) * M + m);
                returns[((size_t)t * N + n) * M + m] = GAE ? g + v : g;
                s = fmaf(ws[m], GAE ? g : g - v, s);
            }
            if (do_adv) { Ash[(size_t)t * N + n] = s; psum += s; }      // raw advantage stays on chip for the normalisation
        }
    }
    if (!do_adv) return;
    // normalise: (adv - mean) / (unbiased std + 1e-5) over the task's T*N samples (raw values in shared memory)
    const float mean = block_sum(psum, red) / (float)S;
    float q = 0.f;
    for (int i = threadIdx.x; i < S; i += blockDim.x) { const float c = Ash[i] - mean; q = fmaf(c, c, q); }
    const float var = block_sum(q, red) / (float)(S - 1);
    const float inv = 1.f / (sqrtf(var) + 1e-5f);
    for (int i = threadIdx.x; i < S; i += blockDim.x) adv[i] = (Ash[i] - mean) * inv;
}

}  // namespace pgm

using namespace pgm;

template <int MODE>
static int k2_launch(const float *rewards, const float *value, const float *boot, const float *masks, const float *bad_masks,
                     const float *weights, const float *obj_var, float gamma, float lam, float *returns, float *adv, int P,
                     int T, int N, int M, cudaStream_t st) {
    // small populations: 32 warps per task, the time axis cut into 32 / N segments (k2_gae_seg_kernel); needs the task's
    // (1 + M) * T * N floats of scratch in shared memory. Large populations already fill the GPU with one warp per column.
    const size_t seg_smem = (size_t)(1 + M) * T * N * sizeof(float);
    if (P <= 64 && M <= 4 && 32 / N >= 2 && T >= 64 * (32 / N) && seg_smem <= 200 * 1024) {
        const int NSEG = 32 / N;
        const int SEG = ((T + NSEG - 1) / NSEG + 31) / 32 * 32;
#define PGM_K2S(MM) case MM: \
            PGM_CUDA(cudaFuncSetAttribute(k2_gae_seg_kernel<MM, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)seg_smem)); \
            k2_gae_seg_kernel<MM, MODE><<<P, 1024, seg_smem, st>>>(rewards, value, boot, masks, bad_masks, weights, obj_var, gamma, lam, returns, adv, T, N, NSEG, SEG); break;
        switch (M) { PGM_K2S(1) PGM_K2S(2) PGM_K2S(3) PGM_K2S(4) }
#undef PGM_K2S
        PGM_CUDA(cudaGetLastError());
        return PGM_OK;
    }
    dim3 grid(P), block(32 * N);
#define PGM_K2(MM) case MM: k2_gae_kernel<MM, MODE><<<grid, block, 0, st>>>(rewards, value, boot, masks, bad_masks, weights, obj_var, gamma, lam, returns, adv, T, N); break;
    switch (M) { PGM_K2(1) PGM_K2(2) PGM_K2(3) PGM_K2(4) PGM_K2(5) PGM_K2(6) PGM_K2(7) PGM_K2(8) }
#undef PGM_K2
    PGM_CUDA(cudaGetLastError());
    return PGM_OK;
}

// argument checks of both entry points (messages name the function the caller called)
static int k2_check(const char *fn, const float *rewards, const float *value, const float *masks, const float *bad_masks,
                    const float *weights, int mode, const float *returns, const float *adv, int P, int T, int N, int M) {
    PGM_REQUIRE(rewards && value && masks && bad_masks && returns, "%s: null pointer", fn);
    PGM_REQUIRE(P > 0 && T > 0 && N > 0 && N <= 32, "%s: need 1 <= N <= 32 env columns (got %d)", fn, N);
    PGM_REQUIRE(M >= 1 && M <= K2_MAXM, "%s: obj_num %d unsupported", fn, M);
    PGM_REQUIRE(!(weights && adv) || (long long)T * N >= 2, "%s: need >= 2 samples to normalise", fn);
    PGM_REQUIRE((mode & ~(PGM_RET_GAE | PGM_RET_PROPER_TIME_LIMITS)) == 0, "%s: unknown mode bits 0x%x", fn, mode);
    return PGM_OK;
}

static int k2_run(int mode, const float *rewards, const float *value, const float *boot, const float *masks,
                  const float *bad_masks, const float *weights, const float *obj_var, float gamma, float lam, float *returns,
                  float *adv, int P, int T, int N, int M, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    switch (mode) {
        case PGM_RET_GAE | PGM_RET_PROPER_TIME_LIMITS:
            return k2_launch<PGM_RET_GAE | PGM_RET_PROPER_TIME_LIMITS>(rewards, value, boot, masks, bad_masks, weights, obj_var,
                                                                         gamma, lam, returns, adv, P, T, N, M, st);
        case PGM_RET_GAE:
            return k2_launch<PGM_RET_GAE>(rewards, value, boot, masks, bad_masks, weights, obj_var, gamma, lam, returns, adv, P,
                                          T, N, M, st);
        case PGM_RET_PROPER_TIME_LIMITS:
            return k2_launch<PGM_RET_PROPER_TIME_LIMITS>(rewards, value, boot, masks, bad_masks, weights, obj_var, gamma, lam,
                                                         returns, adv, P, T, N, M, st);
        default:
            return k2_launch<0>(rewards, value, boot, masks, bad_masks, weights, obj_var, gamma, lam, returns, adv, P, T, N, M, st);
    }
}

extern "C" int pgm_returns_adv_f32(const float *rewards, const float *value, const float *boot, const float *masks,
                                   const float *bad_masks, const float *weights, const float *obj_var, float gamma, float lam,
                                   int mode, float *returns, float *adv, int P, int T, int N, int M, void *stream) {
    if (int rc = k2_check("pgm_returns_adv_f32", rewards, value, masks, bad_masks, weights, mode, returns, adv, P, T, N, M))
        return rc;
    return k2_run(mode, rewards, value, boot, masks, bad_masks, weights, obj_var, gamma, lam, returns, adv, P, T, N, M, stream);
}

extern "C" int pgm_gae_adv_f32(const float *rewards, const float *value, const float *masks, const float *bad_masks,
                               const float *weights, const float *obj_var, float gamma, float lam, float *returns,
                               float *adv, int P, int T, int N, int M, void *stream) {
    const int mode = PGM_RET_GAE | PGM_RET_PROPER_TIME_LIMITS;
    if (int rc = k2_check("pgm_gae_adv_f32", rewards, value, masks, bad_masks, weights, mode, returns, adv, P, T, N, M))
        return rc;
    return k2_run(mode, rewards, value, nullptr, masks, bad_masks, weights, obj_var, gamma, lam, returns, adv, P, T, N, M,
                  stream);
}
