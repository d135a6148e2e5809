// Shared-memory resident HW-HW tanh MLP half (actor or critic) and the register-tiled
// FP32 FFMA building blocks used by K1 (forward) and K3 (forward + backward).
//
// Hidden width HW is a template parameter: 64 (the reference's default) and 32 / 128.
// Thread tiling (RowTile<HW>): a CTA of 256 threads is an RT x CT grid (tr = tid % RT, tc = tid / RT);
// at HW = 64 and 128 that is 16x16, at HW = 32 it is 32x8. For row-tile ops a thread owns rows
// {tr + RT*i, i < RC/RT} and the CG column quads {4*(tc + CT*g) .. +3, g < CG} of a [RC = 16*TM] x HW tile
// (CG = 1 at 32 and 64, 2 at 128). Operands are read from shared memory with 128-bit loads along the
// contraction dimension; row strides are 4*odd floats (HW + 4 = 36, 68, 132) so that the 8 rows touched by
// a quarter warp fall into distinct 16-byte bank groups.
#pragma once
#include "common.cuh"

namespace pgm {

template <int HW>
struct RowTile {
    static_assert(HW == 32 || HW == 64 || HW == 128, "hidden width must be 32, 64 or 128");
    static constexpr int CT = HW < 64 ? HW / 4 : 16;          // column lanes
    static constexpr int RT = NTHREADS / CT;                   // row lanes
    static constexpr int CT_LOG2 = CT == 8 ? 3 : 4;
    static constexpr int RT_LOG2 = RT == 32 ? 5 : 4;
    static constexpr int CG = HW / (4 * CT);                   // column quads per thread
    static constexpr int LD = HW + 4;                          // smem row stride of HW-wide tiles
    static constexpr int LOG2 = HW == 32 ? 5 : (HW == 64 ? 6 : 7);
};

struct HalfNet {           // pointers into shared memory
    float *W1;             // [HW][ldw1]   cols >= O are zero
    float *b1;             // [HW]
    float *W2;             // [HW][HW+4]
    float *b2;             // [HW]
    float *Wh;             // [KH][HW+4]   head: fc_mean (actor) or critic_linear (critic)
    float *bh;             // [KH]
    float *ls;             // [A] logstd (actor only; not loaded for a Categorical head)
    int KH;
};

__host__ __device__ inline int halfnet_smem_floats(const NetLayout &L, int half, int hw = H) {
    int KH = L.head_dim(half);
    return hw * L.ldw1 + hw + hw * (hw + 4) + hw + KH * (hw + 4) + round_up(KH, 4) + (half == 0 ? round_up(L.A, 4) : 0);
}

#ifdef __CUDACC__
template <int HW = H>
__device__ inline float *halfnet_carve(HalfNet &n, float *p, const NetLayout &L, int half) {
    constexpr int LD = RowTile<HW>::LD;
    n.KH = L.head_dim(half);
    n.W1 = p; p += HW * L.ldw1;
    n.b1 = p; p += HW;
    n.W2 = p; p += HW * LD;
    n.b2 = p; p += HW;
    n.Wh = p; p += n.KH * LD;
    n.bh = p; p += round_up(n.KH, 4);
    n.ls = p; if (half == 0) p += round_up(L.A, 4);
    return p;
}

template <bool CG>
__device__ __forceinline__ float ldp(const float *p) { return CG ? __ldcg(p) : __ldg(p); }

// Copy one half's parameters from the flat global vector `g` (reference order) into the padded
// shared-memory image. CG=true reads through L2 only (other CTAs of the cluster just wrote them).
// LS=false: a Categorical head, whose flat vector ends at the head bias (no logstd to load).
template <bool CG, int HW = H, bool LS = true>
__device__ inline void halfnet_load(const HalfNet &n, const float *__restrict__ g, const NetLayout &L, int half) {
    constexpr int LD = RowTile<HW>::LD, LOG2 = RowTile<HW>::LOG2;
    const int tid = threadIdx.x, nt = blockDim.x;
    const float *base = g + L.half_base(half);
    const float *head = g + L.half_head(half);
    const int O = L.O;
    for (int i = tid; i < HW * L.ldw1; i += nt) {
        int j = i / L.ldw1, k = i - j * L.ldw1;
        n.W1[i] = k < O ? ldp<CG>(base + j * O + k) : 0.f;
    }
    const float *b1 = base + HW * O, *W2 = b1 + HW, *b2 = W2 + HW * HW;
    for (int i = tid; i < HW; i += nt) { n.b1[i] = ldp<CG>(b1 + i); n.b2[i] = ldp<CG>(b2 + i); }
    for (int i = tid; i < HW * HW; i += nt) n.W2[(i >> LOG2) * LD + (i & (HW - 1))] = ldp<CG>(W2 + i);
    for (int i = tid; i < n.KH * HW; i += nt) n.Wh[(i >> LOG2) * LD + (i & (HW - 1))] = ldp<CG>(head + i);
    const float *bh = head + n.KH * HW;
    for (int i = tid; i < n.KH; i += nt) n.bh[i] = ldp<CG>(bh + i);
    if (LS && half == 0)
        for (int i = tid; i < L.A; i += nt) n.ls[i] = ldp<CG>(bh + n.KH + i);
}

__device__ __forceinline__ float4 lds4(const float *p) { return *reinterpret_cast<const float4 *>(p); }
__device__ __forceinline__ void sts4(float *p, float4 v) { *reinterpret_cast<float4 *>(p) = v; }

#define PGM_DOT4(acc, a, b) \
    acc = fmaf((a).x, (b).x, acc); acc = fmaf((a).y, (b).y, acc); acc = fmaf((a).z, (b).z, acc); acc = fmaf((a).w, (b).w, acc)

// out[r][j] = tanh(bias[j] + sum_{k<K} in[r][k] * W[j][k]);  r = tr+RT*i, j = 4(tc+CT*g)+c.  K % 4 == 0.
template <int TM, int HW = H>
__device__ __forceinline__ void layer_fwd_tanh(const float *__restrict__ in, int ldi, const float *__restrict__ W,
                                               int ldw, const float *__restrict__ bias, int K,
                                               float *__restrict__ out, int tr, int tc) {
    using T = RowTile<HW>;
    constexpr int RPT = 16 * TM / T::RT, CG = T::CG, CT = T::CT, RT = T::RT;
    float acc[RPT][CG][4];
#pragma unroll
    for (int g = 0; g < CG; ++g) {
        const float4 bv = lds4(bias + 4 * (tc + CT * g));
#pragma unroll
        for (int i = 0; i < RPT; ++i) { acc[i][g][0] = bv.x; acc[i][g][1] = bv.y; acc[i][g][2] = bv.z; acc[i][g][3] = bv.w; }
    }
    const float *ip = in + tr * ldi;
    const float *wp = W + 4 * tc * ldw;
#pragma unroll 2
    for (int k = 0; k < K; k += 4) {
        float4 a[RPT], b[CG][4];
#pragma unroll
        for (int i = 0; i < RPT; ++i) a[i] = lds4(ip + i * RT * ldi + k);
#pragma unroll
        for (int g = 0; g < CG; ++g)
#pragma unroll
            for (int c = 0; c < 4; ++c) b[g][c] = lds4(wp + (4 * CT * g + c) * ldw + k);
#pragma unroll
        for (int i = 0; i < RPT; ++i)
#pragma unroll
            for (int g = 0; g < CG; ++g)
#pragma unroll
                for (int c = 0; c < 4; ++c) { PGM_DOT4(acc[i][g][c], a[i], b[g][c]); }
    }
#pragma unroll
    for (int i = 0; i < RPT; ++i)
#pragma unroll
        for (int g = 0; g < CG; ++g)
            sts4(out + (tr + RT * i) * T::LD + 4 * (tc + CT * g),
                 make_float4(tanhf(acc[i][g][0]), tanhf(acc[i][g][1]), tanhf(acc[i][g][2]), tanhf(acc[i][g][3])));
}

// Head: ho[r][a] = bh[a] + sum_k h[r][k] * Wh[a][k]   (a < KH, ho row stride ldo)
template <int TM, int HW = H>
__device__ __forceinline__ void head_fwd(const float *__restrict__ h, const HalfNet &n, float *__restrict__ ho,
                                         int ldo, int tr, int tc) {
    using T = RowTile<HW>;
    constexpr int RPT = 16 * TM / T::RT, RT = T::RT, LD = T::LD;
    for (int a = tc; a < n.KH; a += T::CT) {
        float acc[RPT];
        const float b = n.bh[a];
#pragma unroll
        for (int i = 0; i < RPT; ++i) acc[i] = b;
        const float *wp = n.Wh + a * LD;
#pragma unroll 4
        for (int k = 0; k < HW; k += 4) {
            const float4 w = lds4(wp + k);
#pragma unroll
            for (int i = 0; i < RPT; ++i) { const float4 x = lds4(h + (tr + RT * i) * LD + k); PGM_DOT4(acc[i], x, w); }
        }
#pragma unroll
        for (int i = 0; i < RPT; ++i) ho[(tr + RT * i) * ldo + a] = acc[i];
    }
}

// Forward of one half for a chunk of RC = 16*TM rows: x [RC][ldx] -> h1, h2 [RC][HW+4], ho [RC][ldo].
// Ends with a __syncthreads() so that ho/h1/h2 are visible to every thread.
template <int TM, int HW = H>
__device__ __forceinline__ void half_forward(const float *x, int ldx, const HalfNet &n, const NetLayout &L,
                                             float *h1, float *h2, float *ho, int ldo, int tr, int tc) {
    constexpr int LD = RowTile<HW>::LD;
    layer_fwd_tanh<TM, HW>(x, ldx, n.W1, L.ldw1, n.b1, L.OP, h1, tr, tc);
    __syncthreads();
    layer_fwd_tanh<TM, HW>(h1, LD, n.W2, LD, n.b2, HW, h2, tr, tc);
    __syncthreads();
    head_fwd<TM, HW>(h2, n, ho, ldo, tr, tc);
    __syncthreads();
}
#endif  // __CUDACC__

}  // namespace pgm
