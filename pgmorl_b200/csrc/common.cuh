// Shared helpers for the sm_100a kernels of the PG-MORL hot path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/pgmorl_b200.h"

namespace pgm {

constexpr int H = PGM_HIDDEN;   // default hidden width (a2c/model.py:202); the FFMA kernels also take 32 and 128
constexpr int LDH = H + 4;      // smem row stride of 64-wide tiles: 68 = 4*17 -> 8 consecutive rows
                                // at the same column land in 8 distinct 16-byte bank groups
__host__ __device__ inline bool hidden_supported(int hw) { return hw == 32 || hw == 64 || hw == 128; }
__host__ __device__ inline bool dist_supported(int d) { return d == PGM_DIST_GAUSSIAN || d == PGM_DIST_CATEGORICAL; }
constexpr int CAT_MAX = 32;     // categories of a Categorical head: K3's generic kernel holds at most 32 head rows
constexpr int NTHREADS = 256;   // every MLP kernel uses 256-thread CTAs (16x16 tiles at hidden width 64, net.cuh)

void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what);

#define PGM_CUDA(call)                                         \
    do {                                                       \
        cudaError_t e_ = (call);                               \
        if (e_ != cudaSuccess) return pgm::cuda_fail(e_, #call); \
    } while (0)

#define PGM_REQUIRE(cond, ...)              \
    do {                                    \
        if (!(cond)) {                      \
            pgm::set_error(__VA_ARGS__);    \
            return PGM_ERR_ARG;             \
        }                                   \
    } while (0)

__host__ __device__ inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
// smallest stride >= x that is 4*odd floats (conflict-free 128-bit row-strided smem access)
__host__ __device__ inline int stride4odd(int x) {
    int s = round_up(x, 4);
    return ((s / 4) & 1) ? s : s + 4;
}

// Offsets of the 13 tensors (12 for a Categorical head: no logstd) inside one flat parameter vector (reference order,
// pgmorl_b200/layout.py) and the two "halves" (actor / critic) the kernels work on. A is the head width: the action
// dimension of a DiagGaussian head, the number of categories of a Categorical head.
struct NetLayout {
    int O, A, M;
    int OP;        // O rounded up to a multiple of 4 (zero padded contraction length of layer 1)
    int ldw1;      // smem row stride of W1 rows / observation rows
    int oW1a, ob1a, oW2a, ob2a, oW1c, ob1c, oW2c, ob2c, oWv, obv, oWmu, obmu, ols, n_par;
    int n_base;    // W1+b1+W2+b2 of one half
    int dist;      // PGM_DIST_GAUSSIAN or PGM_DIST_CATEGORICAL
    int AC;        // action columns of the rollout buffers and K3 records: A (Gaussian) or 1 (the category index)
    int nls;       // logstd entries: A (Gaussian) or 0
    __host__ __device__ NetLayout() {}
    // hw = hidden width (32, 64 or 128)
    __host__ __device__ NetLayout(int O_, int A_, int M_, int hw = H, int dist_ = PGM_DIST_GAUSSIAN)
        : O(O_), A(A_), M(M_), dist(dist_) {
        AC = dist == PGM_DIST_CATEGORICAL ? 1 : A;
        nls = dist == PGM_DIST_CATEGORICAL ? 0 : A;
        OP = round_up(O, 4);
        ldw1 = stride4odd(OP);
        oW1a = 0; ob1a = oW1a + hw * O; oW2a = ob1a + hw; ob2a = oW2a + hw * hw;
        oW1c = ob2a + hw; ob1c = oW1c + hw * O; oW2c = ob1c + hw; ob2c = oW2c + hw * hw;
        oWv = ob2c + hw; obv = oWv + M * hw; oWmu = obv + M; obmu = oWmu + A * hw;
        ols = obmu + A; n_par = ols + nls;
        n_base = hw * O + hw + hw * hw + hw;
    }
    // half 0 = actor (base at 0, head [Wmu bmu logstd] at oWmu), half 1 = critic (contiguous). CAT: a Categorical actor head
    // [W b] has no logstd; the kernels pass the head as a compile-time flag, so the Gaussian code reads no extra field.
    template <bool CAT = false>
    __host__ __device__ int half_size(int half, int hw = H) const { return n_base + (half == 0 ? A * hw + (CAT ? A : 2 * A) : M * hw + M); }
    __host__ __device__ int head_dim(int half) const { return half == 0 ? A : M; }
    __host__ __device__ int half_base(int half) const { return half == 0 ? oW1a : oW1c; }
    __host__ __device__ int half_head(int half) const { return half == 0 ? oWmu : oWv; }
    // half-local flat index -> index in the flat parameter vector
    __host__ __device__ int to_global(int half, int e) const {
        return e < n_base ? half_base(half) + e : half_head(half) + (e - n_base);
    }
};

// ---- device helpers -------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sum over the whole CTA; result valid in every thread. `red` = >= 33 floats of smem.
__device__ __forceinline__ float block_sum(float v, float *red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();                 // protect `red` from a previous use
    if (lane == 0) red[w] = v;
    __syncthreads();
    if (w == 0) {
        float t = lane < nw ? red[lane] : 0.f;
        t = warp_sum(t);
        if (lane == 0) red[32] = t;
    }
    __syncthreads();
    return red[32];
}

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

__device__ __forceinline__ float fast_ex2(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
// tanh(x) = 1 - 2 / (exp(2x) + 1); absolute error ~1e-7 (2 MUFU + 3 FP32 ops instead of ~25 for tanhf)
__device__ __forceinline__ float fast_tanh(float x) {
    const float e = fast_ex2(x * 2.8853900817779268f);
    return 1.f - __fdividef(2.f, e + 1.f);
}
#endif

}  // namespace pgm
