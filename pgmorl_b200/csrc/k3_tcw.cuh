// K3 tensor-core path for WIDE observations (Humanoid: O = 376, A = 17): the PPO minibatch loop
// (a2c/algo/ppo.py:62-107) on tcgen05 with layer 1 streamed through shared memory in 64-feature blocks.
// Included by k3_ppo.cu after k3_tc.cuh (same FP16-pair arithmetic, same helpers, same K3Args).
//
// What differs from k3_tc.cuh. Layer 1 is 6x the rest of the network (64 x 377 against 64 x 64), so neither the
// x tile (128 rows x 384 features, 192 KB as an FP16 pair) nor W1 (96 KB as a pair, 94 KB as FP32 master) can stay
// resident beside the activations:
//   * x is pre-split ONCE per iteration by k3w_pack_kernel into FP16-pair records [row][6 blocks][a1 64 | a2 64]
//     halfwords (1 536 B per row, the size of the FP32 row); a tile's rows are gathered with 16-byte cp.async
//     straight into SWIZZLE_128B block images -- the forward pass streams the six blocks through two 48 KB
//     stages (x block + W1 block), the backward pass streams them again as MN-major operands;
//   * dW1 is accumulated TRANSPOSED, dW1^T[feature][j] += x^T dz1, with M = 128 features (two blocks) per MMA:
//     three 64-column accumulators instead of six. The ones column of x (feature O) yields db1; db2 comes from a
//     shuffle butterfly in the dz2 epilogue;
//   * FP32 master parameters and Adam moments live in an L2-resident workspace; every CTA of a half owns a 1/RS
//     slice of the half: it reduces that slice of the gradient over the RS row-split CTAs through DSMEM, runs
//     Adam on it and publishes the new weights -- W1 as pre-swizzled FP16-pair block images in global memory
//     (read back by everyone's next forward pass), the small tensors straight into every peer's resident
//     operand images through st.shared::cluster.
// One cluster of 2 RS CTAs per task (ranks [0, RS) actor, [RS, 2 RS) critic), RS = 1, 2 or 4; the 128-row tiles
// of a minibatch go round-robin to the RS CTAs of a half; one tile in flight per CTA, all 8 warps on each epilogue.
#pragma once
#include <cuda_fp16.h>

#include "tc.cuh"
#include "tc_pair.cuh"

namespace pgm {

constexpr int TW_NB = 6;                     // 64-feature blocks of layer 1: O + 1 (ones column) <= 384
constexpr int TW_SCF = 24;                   // floats of per-row scalars: action[A] | logp_old | value_old[M] | return[M] | advantage
constexpr int TW_XROW_HW = TW_NB * 128;      // halfwords of one pre-split x record
constexpr uint32_t TW_STAGE = 49152;         // forward stage: x block a1 | a2 (16 KB each), W1 block a1 | a2 (8 KB each)

__host__ __device__ constexpr int tw_nhp(int O, int A) { return (H * O + H + H * H + H + A * H + 2 * A + 63) / 64 * 64; }

struct TwSmem {
    uint32_t H1, H2, ST, W2a, W2b, Wh1, Wh2, DO, SC, FP, DB2, misc, total;
};
__host__ __device__ inline TwSmem tw_smem_layout() {
    TwSmem s; uint32_t o = 0;
    s.H1 = o; o += 32768; s.H2 = o; o += 32768;         // activation pairs [128 rows][64 halfwords] a1 | a2
    s.ST = o; o += 2 * TW_STAGE;                        // forward: 2 stages; backward: x block slots 1..3 (slot 0 = H2)
    s.W2a = o; o += 8192; s.W2b = o; o += 8192;
    s.Wh1 = o; o += 4096; s.Wh2 = o; o += 4096;         // [32 rows a][64 halfwords k]
    s.DO = o; o += 16384;                               // d loss / d head: a1 in halfwords 0..31, a2 in 32..63
    s.SC = o; o += 128 * TW_SCF * 4;
    s.FP = o; o += 512;                                 // b2[64] | bh[32] | logstd[32] (FP32)
    s.DB2 = o; o += 1024;                               // [8 warps][32] column sums of dz2
    s.misc = o; o += 2560; s.total = o;
    return s;
}
// misc (floats): red[40] | part[8 warps][48] | ssq[2 parities][8 ranks][8 warps]; at byte 2304: double sh_d[4], 8 mbarriers, tmem ptr
constexpr int TWM_RED = 0, TWM_PART = 40, TWM_SSQ = 424, TWM_IV = 552;   // iv[24] = exp(-2 logstd)
// TMEM columns
constexpr uint32_t TW_ACC = 0, TW_D1 = 64, TW_D2 = 128, TW_GW2 = 192, TW_GWH = 256, TW_GW1 = 288;   // GW1: 3 x 64

__device__ __forceinline__ void cp_async16_z(uint32_t sdst, const void *gsrc, bool valid) {    // zero-fills when !valid
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(sdst), "l"(gsrc), "r"(valid ? 16 : 0) : "memory");
}
__device__ __forceinline__ void st_dsmem_u2(uint32_t addr, uint2 v) {
    asm volatile("st.shared::cluster.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ void st_dsmem_h(uint32_t addr, __half v) {
    asm volatile("st.shared::cluster.b16 [%0], %1;" ::"r"(addr), "h"(__half_as_ushort(v)) : "memory");
}

// Pre-split pack (once per iteration): x -> FP16-pair block records with the ones column at feature O; per-row scalars.
template <int O, int A, int M>
__global__ void k3w_pack_kernel(const float *__restrict__ obs, size_t obs_ts, const float *__restrict__ action,
                                const float *__restrict__ logp, const float *__restrict__ vold, size_t v_ts,
                                const float *__restrict__ ret, const float *__restrict__ adv, __half *__restrict__ xp,
                                float *__restrict__ scr, int P, int S) {
    const size_t rows = (size_t)P * S;
    const size_t total = rows * (TW_NB * 64 + TW_SCF);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t row = i / (TW_NB * 64 + TW_SCF);
        const int f = (int)(i - row * (TW_NB * 64 + TW_SCF));
        const int task = (int)(row / S), s = (int)(row - (size_t)task * S);
        if (f < TW_NB * 64) {
            const float v = f < O ? obs[task * obs_ts + (size_t)s * O + f] : (f == O ? 1.f : 0.f);
            const float h = round11(v);
            __half *dst = xp + row * TW_XROW_HW + (f >> 6) * 128 + (f & 63);
            dst[0] = __float2half_rn(h); dst[64] = __float2half_rn(v - h);
        } else {
            const int k = f - TW_NB * 64;
            float v = 0.f;
            if (k < A) v = action[((size_t)task * S + s) * A + k];
            else if (k == A) v = logp[(size_t)task * S + s];
            else if (k < A + 1 + M) v = vold[task * v_ts + (size_t)s * M + (k - A - 1)];
            else if (k < A + 1 + 2 * M) v = ret[((size_t)task * S + s) * M + (k - A - 1 - M)];
            else if (k == A + 1 + 2 * M) v = adv[(size_t)task * S + s];
            scr[row * TW_SCF + k] = v;
        }
    }
}

// PGM_K3_TRACE builds: clock64 marks of thread 0 (the MMA issuer), optimiser steps 8 and 9 (profiles/k3_tcw_trace.py):
// trace[(cta * 2 + step - 8) * 48 + mark]
#ifdef PGM_K3_TRACE
#define TWT(i) if (trace_on) a.trace[trace_base + (i)] = clock64();
#else
#define TWT(i)
#endif

struct TwExtra {          // wide-path buffers inside the workspace
    const __half *xp;     // [P][S][TW_XROW_HW]
    const float *scr;     // [P][S][TW_SCF]
    __half *w1img;        // [P][2 halves][TW_NB][a1 4096 | a2 4096] halfwords, SWIZZLE_128B block images
    float *pmv;           // [P][2 halves][master | m | v][NHP]
};

template <int O, int A, int M, int RS, bool VU = false>
__global__ void __launch_bounds__(TC_THREADS, 1) k3_tcw_kernel(const K3Args a, const TwExtra x) {
    constexpr int NHP = tw_nhp(O, A);
    constexpr int KHP = 24;                              // head outputs handled per row (A <= 24)
    constexpr int C = 2 * RS;
    static_assert(O % 4 == 0 && O + 1 <= TW_NB * 64 && O > (TW_NB - 1) * 64 && A <= KHP && M <= 8 && A + 2 * M + 2 <= TW_SCF,
                  "k3_tcw: dims outside the wide tensor-core path");
    extern __shared__ __align__(1024) unsigned char smem_raw[];

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = tc::uniform_warp_idx();
    const int r = tid & 127;                             // row of the tile (= TMEM lane) in the epilogues
    const int q = warp & 3, hcol = warp >> 2;            // lane quadrant, column half
    const int task = blockIdx.x / C;
    const unsigned rank = group_rank<2>();
    const int half = (int)rank / RS, rs = (int)rank % RS;
    const bool actor = half == 0;
    const int KH = actor ? A : M;
    const NetLayout &L = a.L;
    const TwSmem sl = tw_smem_layout();
    constexpr int ob1 = H * O, oW2 = ob1 + H, ob2 = oW2 + H * H, oWh = ob2 + H;
    const int obh = oWh + KH * H, ols = obh + KH;
    const int nH = ols + (actor ? A : 0);
    const int n4 = (nH + 3) >> 2;
    // my slice of the half: chunks of 256 float4 go round-robin to the RS CTAs (every CTA gets the same share of each
    // tensor: the W2 / head publishes through DSMEM are the expensive ones); thread tid owns float4 (u RS + rs) 256 + tid
    constexpr int NU = ((NHP / 4 + TC_THREADS - 1) / TC_THREADS + RS - 1) / RS;
    auto slice_i4 = [&](int u) { return (u * RS + rs) * TC_THREADS + tid; };

    unsigned char *S_h1 = smem_raw + sl.H1, *S_h2 = smem_raw + sl.H2, *S_do = smem_raw + sl.DO;
    __half *W2a = (__half *)(smem_raw + sl.W2a), *W2b = (__half *)(smem_raw + sl.W2b);
    __half *Wh1 = (__half *)(smem_raw + sl.Wh1), *Wh2 = (__half *)(smem_raw + sl.Wh2);
    float *SC = (float *)(smem_raw + sl.SC);
    float *FP = (float *)(smem_raw + sl.FP);             // b2 | bh | logstd
    float *DB2 = (float *)(smem_raw + sl.DB2);
    float *GR = (float *)smem_raw;                       // gradient staging (step tail): parameter order, aliases H1 | H2 | ST
    float *GRW2 = GR + NHP;                              // dW2 rows padded to 68 floats (conflict-free row-owner stores)
    constexpr int GW2LD = 68;
    static_assert((NHP + H * GW2LD) * 4 <= 65536 + 2 * (int)TW_STAGE, "gradient staging does not fit");
    float *misc = (float *)(smem_raw + sl.misc);
    float *red = misc + TWM_RED, *part = misc + TWM_PART, *ssqS = misc + TWM_SSQ, *ivS = misc + TWM_IV;
    double *sh_d = (double *)(smem_raw + sl.misc + 2304);
    uint64_t *mbars = (uint64_t *)(smem_raw + sl.misc + 2304 + 32);     // 0 chain, 1-3 forward stages, 4 weight grads, 5-6 G1X pairs, 7 tile done
    uint32_t *tmem_ptr_s = (uint32_t *)(smem_raw + sl.misc + 2304 + 96);
    uint64_t *mbarN = (uint64_t *)(smem_raw + sl.misc + 2304 + 104);    // counts the bytes of the cluster's squared-norm partials
    const float *b2s = FP, *bhs = FP + 64, *lss = FP + 96;

    // global state of my half
    __half *w1g = x.w1img + (size_t)(task * 2 + half) * TW_NB * 8192;
    float *PMg = x.pmv + (size_t)(task * 2 + half) * 3 * NHP, *Mg = PMg + NHP, *Vg = Mg + NHP;

    // ---------------- one-time setup ----------------
    for (int i = tid; i < (int)(sl.total / 16); i += TC_THREADS) reinterpret_cast<float4 *>(smem_raw)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();
    if (warp == 0) tc::tmem_alloc(tmem_ptr_s, 512);
    if (tid == 0) {
        for (int i = 0; i < 8; ++i) tc::mbar_init(mbars + i, 1);
        tc::mbar_init(mbarN, 1);
        tc::fence_mbar_init();
    }
    // publish one parameter / four consecutive parameters (half-local index) to wherever the kernels read them:
    // W1, b1 -> global block images; W2, Wh -> every row-split peer's operand images; b2, bh, logstd -> their FP arrays
    uint32_t peer_base[RS];
#pragma unroll
    for (int k = 0; k < RS; ++k) peer_base[k] = mapa_u32(smem_u32(smem_raw), (uint32_t)(half * RS + k));
    auto put1 = [&](int e, float p) {
        if (e < oW2) {
            const int j = e < ob1 ? e / O : e - ob1, c = e < ob1 ? e - j * O : O;
            __half *img = w1g + (c >> 6) * 8192;
            const int hw = sw128_hw(j, c & 63);
            const float v = p * TC_SW, h = round11(v);
            img[hw] = __float2half_rn(h); img[4096 + hw] = __float2half_rn(v - h);
        } else if (e < ob2 || (e >= oWh && e < obh)) {
            const bool w2 = e < ob2;
            const int rr = w2 ? (e - oW2) >> 6 : (e - oWh) >> 6, k = w2 ? (e - oW2) & 63 : (e - oWh) & 63;
            const uint32_t o1 = (w2 ? sl.W2a : sl.Wh1) + 2u * (uint32_t)sw128_hw(rr, k), o2 = (w2 ? sl.W2b : sl.Wh2) + 2u * (uint32_t)sw128_hw(rr, k);
            const float v = p * TC_SW, h = round11(v);
#pragma unroll
            for (int kk = 0; kk < RS; ++kk) { st_dsmem_h(peer_base[kk] + o1, __float2half_rn(h)); st_dsmem_h(peer_base[kk] + o2, __float2half_rn(v - h)); }
        } else {
            const int fi = e < oWh ? e - ob2 : (e < ols ? 64 + e - obh : 96 + e - ols);
#pragma unroll
            for (int kk = 0; kk < RS; ++kk) st_dsmem1(peer_base[kk] + sl.FP + 4u * (uint32_t)fi, p);
        }
    };
    auto put4 = [&](int e0, float4 p) {
        const bool inW1 = e0 + 3 < ob1, inW2 = e0 >= oW2 && e0 + 3 < ob2, inWh = e0 >= oWh && e0 + 3 < obh;
        if (inW1 || inW2 || inWh) {
            const float w0 = p.x * TC_SW, w1 = p.y * TC_SW, w2 = p.z * TC_SW, w3 = p.w * TC_SW;
            const float h0 = round11(w0), h1 = round11(w1), h2 = round11(w2), h3 = round11(w3);
            const uint2 v1 = make_uint2(pack_h2_ovf(h0, h1), pack_h2_ovf(h2, h3));
            const uint2 v2 = make_uint2(pack_h2_ovf(w0 - h0, w1 - h1), pack_h2_ovf(w2 - h2, w3 - h3));
            if (inW1) {
                const int j = e0 / O, c = e0 - j * O;
                __half *img = w1g + (c >> 6) * 8192;
                const int hw = sw128_hw(j, c & 63);
                *reinterpret_cast<uint2 *>(img + hw) = v1; *reinterpret_cast<uint2 *>(img + 4096 + hw) = v2;
            } else {
                const int eo = inW2 ? e0 - oW2 : e0 - oWh;
                const uint32_t hw2 = 2u * (uint32_t)sw128_hw(eo >> 6, eo & 63);
#pragma unroll
                for (int kk = 0; kk < RS; ++kk) {
                    st_dsmem_u2(peer_base[kk] + (inW2 ? sl.W2a : sl.Wh1) + hw2, v1);
                    st_dsmem_u2(peer_base[kk] + (inW2 ? sl.W2b : sl.Wh2) + hw2, v2);
                }
            }
        } else {
            put1(e0, p.x);
            if (e0 + 1 < nH) put1(e0 + 1, p.y);
            if (e0 + 2 < nH) put1(e0 + 2, p.z);
            if (e0 + 3 < nH) put1(e0 + 3, p.w);
        }
    };
    sync_group<2>();                                     // every CTA of the cluster zeroed its shared memory
    {   // my slice: reference order -> half-local master / moments in the workspace, operand images
        const float *gpar = a.params + (size_t)task * L.n_par;
        for (int u = 0; u < NU; ++u) {
            const int i4 = slice_i4(u);
            if (i4 >= n4) break;
            float pv[4], mv[4], vv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = 4 * i4 + u;
                const bool in = e < nH;
                const size_t gi = (size_t)task * L.n_par + (in ? L.to_global(half, e) : 0);
                pv[u] = in ? __ldg(gpar + L.to_global(half, e)) : 0.f;
                mv[u] = (in && !a.grad_only) ? a.adam_m[gi] : 0.f; vv[u] = (in && !a.grad_only) ? a.adam_v[gi] : 0.f;
            }
            const float4 p4 = make_float4(pv[0], pv[1], pv[2], pv[3]);
            __stcg(reinterpret_cast<float4 *>(PMg) + i4, p4);
            __stcg(reinterpret_cast<float4 *>(Mg) + i4, make_float4(mv[0], mv[1], mv[2], mv[3]));
            __stcg(reinterpret_cast<float4 *>(Vg) + i4, make_float4(vv[0], vv[1], vv[2], vv[3]));
            put4(4 * i4, p4);
        }
    }
    __threadfence();
    tc::fence_async_smem();
    tc::tc_fence_before();
    sync_group<2>();                 // images of every slice are in place (global + peers' shared memory); barriers / TMEM address visible
    tc::tc_fence_after();
    const uint32_t tmem = tc::uniform_u32(*tmem_ptr_s);
    const uint32_t tq = tmem + ((uint32_t)(q * 32) << 16);

    {   // zero the weight-gradient accumulators (each thread: the cells it reads in the step tail)
        float z[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) z[i] = 0.f;
        tc::tmem_st32(tq + TW_GW2 + 32 * hcol, z);
        if (hcol == 0) tc::tmem_st32(tq + TW_GWH, z);
#pragma unroll
        for (int pp = 0; pp < 3; ++pp) tc::tmem_st32(tq + TW_GW1 + 64 * pp + 32 * hcol, z);
        tc::tmem_st_wait();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();

    // ---------------- constants ----------------
    const float clip = (float)a.hy.clip_param;
    const float inv_mb = 1.f / (float)a.mb;
    const float vscale = (float)(a.hy.value_loss_coef * 0.5 / ((double)a.mb * M));
    const float omb1 = (float)(1.0 - a.hy.beta1);
    const float b2f = (float)a.hy.beta2, omb2 = (float)(1.0 - a.hy.beta2);
    const float aeps = (float)a.hy.adam_eps;
    const float ecoef = (float)a.hy.entropy_coef;
    const int step0 = a.grad_only ? 0 : a.adam_step[task];
    double b1pow = pow(a.hy.beta1, (double)step0), b2pow = pow(a.hy.beta2, (double)step0);   // used by thread 0
    const double lr = a.grad_only ? 0.0 : a.lr[task];
    float loss_act = 0.f, loss_val = 0.f, loss_ent = 0.f;

    const int32_t *perm = a.perm + ((a.perm_shared || a.grad_only) ? 0 : (size_t)task * a.E * a.S);
    const __half *xpg = x.xp + (size_t)task * a.S * TW_XROW_HW;
    const float *scg = x.scr + (size_t)task * a.S * TW_SCF;
    const int ntiles_all = (a.mb + 127) >> 7;
    const int ntiles = rs < ntiles_all ? (ntiles_all - rs + RS - 1) / RS : 0;
    uint32_t ph[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};      // mbarrier phase parities
    auto mwait = [&](int b) { tc::mbar_wait(mbars + b, ph[b]); ph[b] ^= 1u; };

    // ---- descriptors (images are [rows][64 halfwords], SWIZZLE_128B; see k3_tc.cuh for the two views) ----
    const uint32_t aH1 = tc::smem_addr(S_h1), aH2 = tc::smem_addr(S_h2), aST = tc::smem_addr(smem_raw + sl.ST), aDO = tc::smem_addr(S_do);
    const uint32_t aW2a = tc::smem_addr(W2a), aW2b = tc::smem_addr(W2b), aWh1 = tc::smem_addr(Wh1), aWh2 = tc::smem_addr(Wh2);
    auto dK = [](uint32_t addr) { return tc::make_desc(addr, 16, 1024, 2); };
    auto dMN = [](uint32_t addr, uint32_t lbo) { return tc::make_desc(addr, lbo, 1024, 2); };
    const uint64_t dH1a_k = dK(aH1), dH1b_k = dK(aH1 + 16384), dH2a_k = dK(aH2), dH2b_k = dK(aH2 + 16384);
    const uint64_t dW2a_k = dK(aW2a), dW2b_k = dK(aW2b), dWh1_k = dK(aWh1), dWh2_k = dK(aWh2);
    const uint64_t dDOa_k = dK(aDO), dDOb_k = dK(aDO + 64);                      // K windows of 32 features: a1 | a2
    const uint64_t dWh1_mn = dMN(aWh1, 16384), dWh2_mn = dMN(aWh2, 16384), dW2a_mn = dMN(aW2a, 16384), dW2b_mn = dMN(aW2b, 16384);
    const uint64_t dH1a_mn = dMN(aH1, 32768), dH1b_mn = dMN(aH1 + 16384, 32768);
    const uint64_t dH2a_mn = dMN(aH2, 32768), dH2b_mn = dMN(aH2 + 16384, 32768);
    const uint64_t dDOa_mn = dMN(aDO, 16384), dDOb_mn = dMN(aDO + 64, 16384);    // N = 32 head columns: a1 | a2
    // backward x slots: slot 0 = H2, slots 1..3 = ST; a pair of slots (2p, 2p + 1) is one M = 128 MN-major operand
    const uint64_t dX0a_mn = dMN(aH2, 32768), dX0b_mn = dMN(aH2 + 16384, 32768);             // slots (0, 1)
    const uint64_t dX2a_mn = dMN(aST + 32768, 32768), dX2b_mn = dMN(aST + 49152, 32768);     // slots (2, 3)
    constexpr uint32_t ID_KK = tc::idesc_f16(128, 64, 0, 0), ID_HEAD = tc::idesc_f16(128, 32, 0, 0), ID_KM = tc::idesc_f16(128, 64, 0, 1);
    constexpr uint32_t ID_GWH = tc::idesc_f16(64, 32, 1, 1), ID_GW2 = tc::idesc_f16(64, 64, 1, 1), ID_GW1 = tc::idesc_f16(128, 64, 1, 1);
    const uint32_t swz = (uint32_t)(r & 7);

    auto sync_all = [&]() { tc::tmem_st_wait(); tc::tmem_ld_wait(); tc::fence_async_smem(); tc::tc_fence_before(); __syncthreads(); };
    auto mma3 = [&](uint32_t d, uint64_t a1, uint64_t a2, uint64_t b1, uint64_t b2, uint32_t id, uint32_t acc) {
        tc::mma_f16(d, a2, b1, id, acc); tc::mma_f16(d, a1, b2, id, 1); tc::mma_f16(d, a1, b1, id, 1);
    };

    // gather of one 64-feature x block of the current tile into an image pair at shared address `dst` (a1 | a2 16 KB apart):
    // item f = tid + 256 k is (row f / 16, 16-byte piece f % 16): 16 consecutive threads read one 256-byte block record
    int ridx[8];
    uint32_t rvalid = 0u;
    auto load_xblock = [&](int b, uint32_t dst) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int row = (tid >> 4) + 16 * k, pc = tid & 15;
            const uint32_t d = dst + (uint32_t)(pc >> 3) * 16384u + (uint32_t)row * 128u + ((uint32_t)((pc & 7) ^ (row & 7)) << 4);
            cp_async16_z(d, xpg + (size_t)ridx[k] * TW_XROW_HW + b * 128 + pc * 8, (rvalid >> k) & 1u);
        }
    };
    auto load_w1block = [&](int b, uint32_t dst) {       // 16 KB, pre-swizzled: plain copy
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int it = tid + TC_THREADS * k;
            cp_async16_z(dst + 16u * (uint32_t)it, w1g + (size_t)b * 8192 + it * 8, true);
        }
    };

    for (int s = 0; s < a.nsteps; ++s) {
#ifdef PGM_K3_TRACE
        const bool trace_on = a.trace && (s == 8 || s == 9) && tid == 0;
        const size_t trace_base = ((size_t)blockIdx.x * 2 + (s - 8)) * 48;
#endif
        if (actor && rs == 0 && tid == 0) {   // entropy with the parameters this step starts from
            float ent = 0.f;
            for (int d = 0; d < A; ++d) ent += 0.5f + 0.91893853320467274178f + lss[d];
            loss_ent += ent;
        }
        for (int i = tid; i < 8 * 48; i += TC_THREADS) part[i] = 0.f;
        DB2[tid] = 0.f;
        if (actor && tid < A) ivS[tid] = expf(-2.f * lss[tid]);
        const int ep = s / a.B, bb = s - ep * a.B;
        const int32_t *pb = perm + (size_t)ep * a.S + (size_t)bb * a.mb;

        for (int t = 0; t < ntiles; ++t) {
            const int row0 = (t * RS + rs) * 128;
            // ---------------- row indices, per-row scalars, first two forward stages ----------------
            rvalid = 0u;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int rowi = row0 + (tid >> 4) + 16 * k;
                const bool ok = rowi < a.mb;
                ridx[k] = ld_nc_s32(pb + (ok ? rowi : 0));
                rvalid |= (ok ? 1u : 0u) << k;
            }
            TWT(0)
            __syncthreads();                                   // everyone is done with the previous tile / step tail (SC, DO, ST)
            if ((tid & 15) < 6) {                              // per-row scalars: pieces 0..5 of the 8 rows this thread gathers
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int row = (tid >> 4) + 16 * k, pc = tid & 15;
                    cp_async16_z(tc::smem_addr(SC) + (uint32_t)(row * 6 + pc) * 16u, scg + (size_t)ridx[k] * TW_SCF + pc * 4, (rvalid >> k) & 1u);
                }
            }
            // three forward stages (x block 32 KB + W1 block 16 KB): the two in ST, and H2 + DO, both idle until E2 / E3
            const uint32_t stX[3] = {aST, aST + TW_STAGE, aH2}, stW[3] = {aST + 32768, aST + TW_STAGE + 32768, aDO};
#pragma unroll
            for (int b = 0; b < 3; ++b) { load_xblock(b, stX[b]); load_w1block(b, stW[b]); cp_async_commit(); }
            TWT(1)
            // ---------------- G1: Z1 = [x | 1] W1^T over six streamed blocks ----------------
#pragma unroll
            for (int b = 0; b < TW_NB; ++b) {
                if (b < TW_NB - 2) cp_async_wait<2>(); else if (b == TW_NB - 2) cp_async_wait<1>(); else cp_async_wait<0>();
                tc::fence_async_smem();
                __syncthreads();
                const int st = b % 3;
                if (warp == 0 && tc::elect_one()) {
                    tc::tc_fence_after();
                    const uint64_t xa = dK(stX[st]), xb = dK(stX[st] + 16384), wa = dK(stW[st]), wb = dK(stW[st] + 8192);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        mma3(tmem + TW_ACC, tc::desc_advance(xa, 32 * ks), tc::desc_advance(xb, 32 * ks),
                             tc::desc_advance(wa, 32 * ks), tc::desc_advance(wb, 32 * ks), ID_KK, (b > 0 || ks > 0) ? 1u : 0u);
                    if (b == TW_NB - 1) tc::mma_commit(mbars + 0);                  // covers every MMA of G1
                    else if (b + 3 < TW_NB) tc::mma_commit(mbars + 1 + st);         // stage st is refilled below
                }
                if (b + 3 < TW_NB) {
                    mwait(1 + st);                             // the MMAs of block b released their stage
                    load_xblock(b + 3, stX[st]); load_w1block(b + 3, stW[st]);
                    cp_async_commit();
                }
                TWT(2 + b)
            }
            // ---------------- E1: h1 = tanh(Z1) -> H1 pair, 1 - h1^2 -> TMEM ----------------
            {
                unsigned char *rowh1 = S_h1 + r * 128;
                mwait(0); tc::tc_fence_after();
                TWT(8)
                // the stages are free: prefetch x blocks 1..3 of the backward pass into slots 1..3
                load_xblock(1, aST); load_xblock(2, aST + 32768); load_xblock(3, aST + 65536);
                cp_async_commit();
                float z[32], dd[32];
                tc::tmem_ld32(tq + TW_ACC + 32 * hcol, z);
                tc::tmem_ld_wait();
#pragma unroll
                for (int k = 0; k < 32; ++k) { z[k] = fast_tanh(z[k] * (1.f / TC_SW)); dd[k] = fmaf(-z[k], z[k], 1.f); z[k] *= TC_SH; }
                tc::tmem_st32(tq + TW_D1 + 32 * hcol, dd);
#pragma unroll
                for (int c = 0; c < 4; ++c) store_pair8(rowh1, (uint32_t)(4 * hcol + c), rowh1 + 16384, (uint32_t)(4 * hcol + c), swz, z + 8 * c);
                TWT(9)
                sync_all();
                if (warp == 0 && tc::elect_one()) {
                    tc::tc_fence_after();
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        mma3(tmem + TW_ACC, tc::desc_advance(dH1a_k, 32 * ks), tc::desc_advance(dH1b_k, 32 * ks),
                             tc::desc_advance(dW2a_k, 32 * ks), tc::desc_advance(dW2b_k, 32 * ks), ID_KK, ks > 0);
                    tc::mma_commit(mbars + 0);
                }
                TWT(10)
            }
            // ---------------- E2: h2 = tanh(Z2 + b2) -> H2 pair, 1 - h2^2 -> TMEM ----------------
            {
                unsigned char *rowh2 = S_h2 + r * 128;
                mwait(0); tc::tc_fence_after();
                TWT(11)
                float z[32], dd[32];
                tc::tmem_ld32(tq + TW_ACC + 32 * hcol, z);
                tc::tmem_ld_wait();
#pragma unroll
                for (int k = 0; k < 32; ++k) z[k] = fmaf(z[k], 1.f / (TC_SH * TC_SW), b2s[32 * hcol + k]);
#pragma unroll
                for (int k = 0; k < 32; ++k) { z[k] = fast_tanh(z[k]); dd[k] = fmaf(-z[k], z[k], 1.f); z[k] *= TC_SH; }
                tc::tmem_st32(tq + TW_D2 + 32 * hcol, dd);
#pragma unroll
                for (int c = 0; c < 4; ++c) store_pair8(rowh2, (uint32_t)(4 * hcol + c), rowh2 + 16384, (uint32_t)(4 * hcol + c), swz, z + 8 * c);
                TWT(12)
                sync_all();
                if (warp == 0 && tc::elect_one()) {
                    tc::tc_fence_after();
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        mma3(tmem + TW_ACC, tc::desc_advance(dH2a_k, 32 * ks), tc::desc_advance(dH2b_k, 32 * ks),
                             tc::desc_advance(dWh1_k, 32 * ks), tc::desc_advance(dWh2_k, 32 * ks), ID_HEAD, ks > 0);
                    tc::mma_commit(mbars + 0);
                }
                TWT(13)
            }
            // ---------------- E3: per-row loss and d loss / d head (warps 0..3: thread = row) ----------------
            mwait(0); tc::tc_fence_after();
            TWT(14)
            if (hcol == 0) {
                float ho[32], dq[32];
                tc::tmem_ld32(tq + TW_ACC, ho);
                const float *sc = SC + r * TW_SCF;
                const bool row_valid = row0 + r < a.mb;
                tc::tmem_ld_wait();
                float gb[KHP], gl[KHP];
#pragma unroll
                for (int d = 0; d < KHP; ++d) { gb[d] = 0.f; gl[d] = 0.f; }
#pragma unroll
                for (int d = 0; d < 32; ++d) dq[d] = 0.f;
                if (actor) {
                    float lp = 0.f, diffv[KHP], ivv[KHP];
#pragma unroll
                    for (int d = 0; d < KHP; ++d) {
                        diffv[d] = 0.f; ivv[d] = 0.f;
                        if (d < A) {
                            const float ls = lss[d];
                            const float iv = ivS[d];
                            const float diff = sc[d] - fmaf(ho[d], 1.f / (TC_SH * TC_SW), bhs[d]);
                            lp += -0.5f * (diff * diff * iv) - ls - 0.91893853320467274178f;
                            diffv[d] = diff; ivv[d] = iv;
                        }
                    }
                    const float ratio = expf(lp - sc[A]);
                    const float adv = sc[A + 1 + 2 * M];
                    const float surr1 = ratio * adv;
                    const float rcl = fminf(fmaxf(ratio, 1.f - clip), 1.f + clip);
                    const float surr2 = rcl * adv;
                    const float w1 = surr1 < surr2 ? 1.f : (surr1 == surr2 ? 0.5f : 0.f);
                    const float inr = (ratio >= 1.f - clip && ratio <= 1.f + clip) ? 1.f : 0.f;
                    const float dmin = w1 * adv + (1.f - w1) * adv * inr;
                    const float dlp = row_valid ? -inv_mb * dmin * ratio : 0.f;
                    if (row_valid) loss_act -= fminf(surr1, surr2);
#pragma unroll
                    for (int d = 0; d < KHP; ++d) {
                        if (d < A) {
                            const float go = dlp * diffv[d] * ivv[d];                 // d loss / d mean
                            gb[d] = go;
                            gl[d] = dlp * (diffv[d] * diffv[d] * ivv[d] - 1.f);
                            dq[d] = go * TC_SD;
                        }
                    }
                } else {
#pragma unroll
                    for (int m = 0; m < M; ++m) {
                        float go = 0.f;
                        const float V = fmaf(ho[m], 1.f / (TC_SH * TC_SW), bhs[m]), vo = sc[A + 1 + m], R = sc[A + 1 + M + m];
                        const float dlt = V - vo;
                        const float vcl = vo + fminf(fmaxf(dlt, -clip), clip);
                        const float ea = V - R, eb = vcl - R;
                        // unclipped value loss (VU): lb = -1 < 0 <= la, so max(la, lb) = la and wa = 1, gradient 2 * ea exactly
                        const float la = ea * ea, lb = VU ? -1.f : eb * eb;
                        const float wa = la > lb ? 1.f : (la == lb ? 0.5f : 0.f);
                        const float pas = (dlt >= -clip && dlt <= clip) ? 1.f : 0.f;
                        if (row_valid) { loss_val += fmaxf(la, lb); go = vscale * (wa * 2.f * ea + (1.f - wa) * 2.f * eb * pas); }
                        gb[m] = go;
                        dq[m] = go * TC_SD;
                    }
                }
                unsigned char *rowd = S_do + r * 128;
#pragma unroll
                for (int c = 0; c < 4; ++c) store_pair8(rowd, (uint32_t)c, rowd, (uint32_t)(4 + c), swz, dq + 8 * c);
                // head bias / logstd gradients: sums over the warp's 32 rows -> this warp's partial slots
                if (actor) {                                   // 2 A <= 32 + 2 values: halving butterfly on 32, plain sums for the rest
                    float v[32];
#pragma unroll
                    for (int d = 0; d < 32; ++d) v[d] = d < A ? gb[d < A ? d : 0] : ((d - A < A) ? gl[(d - A < A) ? d - A : 0] : 0.f);
#pragma unroll
                    for (int off = 16; off >= 1; off >>= 1) {
                        const bool up = (lane & off) != 0;
#pragma unroll
                        for (int i = 0; i < off; ++i) {
                            const float keep = up ? v[i + off] : v[i], send = up ? v[i] : v[i + off];
                            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
                        }
                    }
                    part[warp * 48 + (lane < A ? lane : 24 + lane - A)] += v[0];        // lane l holds value l
#pragma unroll
                    for (int d = 32 - A; d < A; ++d) {                                    // logstd entries that did not fit
                        const float sg = warp_sum(gl[d]);
                        if (lane == 0) part[warp * 48 + 24 + d] += sg;
                    }
                } else {
#pragma unroll
                    for (int d = 0; d < M; ++d) {
                        const float sb = warp_sum(gb[d]);
                        if (lane == 0) part[warp * 48 + d] += sb;
                    }
                }
            }
            TWT(15)
            sync_all();
            if (warp == 0 && tc::elect_one()) {
                tc::tc_fence_after();
#pragma unroll
                for (int ks = 0; ks < 2; ++ks)                                                     // dz2pre = dOut Wh (K = 32 head columns)
                    mma3(tmem + TW_ACC, tc::desc_advance(dDOa_k, 32 * ks), tc::desc_advance(dDOb_k, 32 * ks),
                         tc::desc_advance(dWh1_mn, 2048 * ks), tc::desc_advance(dWh2_mn, 2048 * ks), ID_KM, ks > 0);
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)                                                     // dWh^T += h2^T dOut
                    mma3(tmem + TW_GWH, tc::desc_advance(dH2a_mn, 2048 * ks), tc::desc_advance(dH2b_mn, 2048 * ks),
                         tc::desc_advance(dDOa_mn, 2048 * ks), tc::desc_advance(dDOb_mn, 2048 * ks), ID_GWH, 1);
                tc::mma_commit(mbars + 0);
            }
            TWT(16)
            // ---------------- E4: dz2 = dz2pre (1 - h2^2) -> H2 pair (in place); db2 += column sums ----------------
            {
                unsigned char *rowh2 = S_h2 + r * 128;
                mwait(0); tc::tc_fence_after();
                TWT(17)
                float z[32], dd[32];
                tc::tmem_ld32(tq + TW_ACC + 32 * hcol, z);
                tc::tmem_ld32(tq + TW_D2 + 32 * hcol, dd);
                tc::tmem_ld_wait();
#pragma unroll
                for (int k = 0; k < 32; ++k) z[k] = z[k] * (1.f / TC_SW) * dd[k];           // dz2 (still x 2^12)
#pragma unroll
                for (int c = 0; c < 4; ++c) store_pair8(rowh2, (uint32_t)(4 * hcol + c), rowh2 + 16384, (uint32_t)(4 * hcol + c), swz, z + 8 * c);
                // column sums over the warp's 32 rows: halving butterfly, lane l ends with column 32 hcol + l
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    const bool up = (lane & off) != 0;
#pragma unroll
                    for (int i = 0; i < off; ++i) {
                        const float keep = up ? z[i + off] : z[i], send = up ? z[i] : z[i + off];
                        z[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
                    }
                }
                DB2[warp * 32 + lane] += z[0];
                TWT(18)
                sync_all();
                if (warp == 0 && tc::elect_one()) {
                    tc::tc_fence_after();
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)                                                 // dz1pre = dz2 W2
                        mma3(tmem + TW_ACC, tc::desc_advance(dH2a_k, 32 * ks), tc::desc_advance(dH2b_k, 32 * ks),
                             tc::desc_advance(dW2a_mn, 2048 * ks), tc::desc_advance(dW2b_mn, 2048 * ks), ID_KM, ks > 0);
                    tc::mma_commit(mbars + 0);
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)                                                 // dW2 += dz2^T h1
                        mma3(tmem + TW_GW2, tc::desc_advance(dH2a_mn, 2048 * ks), tc::desc_advance(dH2b_mn, 2048 * ks),
                             tc::desc_advance(dH1a_mn, 2048 * ks), tc::desc_advance(dH1b_mn, 2048 * ks), ID_GW2, 1);
                    tc::mma_commit(mbars + 4);
                }
                TWT(19)
            }
            // ---------------- E5: dz1 = dz1pre (1 - h1^2) -> H1 pair (in place) ----------------
            {
                unsigned char *rowh1 = S_h1 + r * 128;
                mwait(0); tc::tc_fence_after();
                TWT(20)
                float z[32], dd[32];
                tc::tmem_ld32(tq + TW_ACC + 32 * hcol, z);
                tc::tmem_ld32(tq + TW_D1 + 32 * hcol, dd);
                tc::tmem_ld_wait();
#pragma unroll
                for (int k = 0; k < 32; ++k) z[k] = z[k] * (1.f / TC_SW) * dd[k];
                mwait(4);                                      // dW2 MMAs are done reading h1 and dz2: H2 becomes x slot 0
                TWT(21)
                load_xblock(0, aH2);
                cp_async_commit();
#pragma unroll
                for (int c = 0; c < 4; ++c) store_pair8(rowh1, (uint32_t)(4 * hcol + c), rowh1 + 16384, (uint32_t)(4 * hcol + c), swz, z + 8 * c);
                cp_async_wait<0>();
                sync_all();
                TWT(22)
            }
            // ---------------- G1X: dW1^T[feature][j] += x^T dz1, two blocks (M = 128 features) per accumulator ----------------
            if (warp == 0 && tc::elect_one()) {
                tc::tc_fence_after();
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)
                    mma3(tmem + TW_GW1, tc::desc_advance(dX0a_mn, 2048 * ks), tc::desc_advance(dX0b_mn, 2048 * ks),
                         tc::desc_advance(dH1a_mn, 2048 * ks), tc::desc_advance(dH1b_mn, 2048 * ks), ID_GW1, 1);
                tc::mma_commit(mbars + 5);
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)
                    mma3(tmem + TW_GW1 + 64, tc::desc_advance(dX2a_mn, 2048 * ks), tc::desc_advance(dX2b_mn, 2048 * ks),
                         tc::desc_advance(dH1a_mn, 2048 * ks), tc::desc_advance(dH1b_mn, 2048 * ks), ID_GW1, 1);
                tc::mma_commit(mbars + 6);
            }
            TWT(23)
            mwait(5);                                          // slots 0, 1 are free: blocks 4, 5
            TWT(24)
            load_xblock(4, aH2); load_xblock(5, aST);
            cp_async_commit();
            cp_async_wait<0>();
            tc::fence_async_smem();
            __syncthreads();
            TWT(25)
            if (warp == 0 && tc::elect_one()) {
                tc::tc_fence_after();
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)
                    mma3(tmem + TW_GW1 + 128, tc::desc_advance(dX0a_mn, 2048 * ks), tc::desc_advance(dX0b_mn, 2048 * ks),
                         tc::desc_advance(dH1a_mn, 2048 * ks), tc::desc_advance(dH1b_mn, 2048 * ks), ID_GW1, 1);
                tc::mma_commit(mbars + 7);
            }
            TWT(26)
            mwait(6);
            mwait(7);                                          // every MMA of this tile is complete: H1, H2, ST, DO are free
            tc::tc_fence_after();
            TWT(27)
        }   // tiles

        // ================= step tail =================
        // gradients: TMEM -> GR (parameter order; aliases the tile buffers), accumulators handed back zeroed
        __syncthreads();
        TWT(28)
        {
            float gw[32], z[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) z[i] = 0.f;
            tc::tmem_ld32(tq + TW_GW2 + 32 * hcol, gw);
            tc::tmem_ld_wait();
            tc::tmem_st32(tq + TW_GW2 + 32 * hcol, z);
            if (lane < 16) {                               // dW2 rows: (dz2 2^12)^T (h1 2^8)
                float *dst = GRW2 + (16 * q + lane) * GW2LD + 32 * hcol;
#pragma unroll
                for (int i = 0; i < 32; i += 4)
                    *reinterpret_cast<float4 *>(dst + i) = make_float4(gw[i] * (1.f / (TC_SD * TC_SH)), gw[i + 1] * (1.f / (TC_SD * TC_SH)),
                                                                         gw[i + 2] * (1.f / (TC_SD * TC_SH)), gw[i + 3] * (1.f / (TC_SD * TC_SH)));
            }
            if (hcol == 0) {                               // dWh^T rows: (h2 2^8)^T (dOut 2^12)
                tc::tmem_ld32(tq + TW_GWH, gw);
                tc::tmem_ld_wait();
                tc::tmem_st32(tq + TW_GWH, z);
                if (lane < 16) {
                    const int k = 16 * q + lane;
#pragma unroll
                    for (int aa = 0; aa < KHP; ++aa)
                        if (aa < KH) GR[oWh + aa * H + k] = gw[aa] * (1.f / (TC_SD * TC_SH));
                }
            }
#pragma unroll
            for (int pp = 0; pp < 3; ++pp) {               // dW1^T | db1: lane = feature, columns = hidden unit
                tc::tmem_ld32(tq + TW_GW1 + 64 * pp + 32 * hcol, gw);
                tc::tmem_ld_wait();
                tc::tmem_st32(tq + TW_GW1 + 64 * pp + 32 * hcol, z);
                const int f = 128 * pp + 32 * q + lane;
                if (f < O) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) GR[(32 * hcol + i) * O + f] = gw[i] * (1.f / TC_SD);
                } else if (f == O) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) GR[ob1 + 32 * hcol + i] = gw[i] * (1.f / TC_SD);
                }
            }
        }
        if (tid < 64) {                                    // db2: the four quadrant warps of the column half
            const int hc = tid >> 5, l = tid & 31;
            GR[ob2 + tid] = (DB2[(4 * hc + 0) * 32 + l] + DB2[(4 * hc + 1) * 32 + l] + DB2[(4 * hc + 2) * 32 + l] + DB2[(4 * hc + 3) * 32 + l]) * (1.f / TC_SD);
        } else if (tid < 64 + KHP) {                       // head bias, logstd
            const int d = tid - 64;
            if (d < KH) GR[obh + d] = part[0 * 48 + d] + part[1 * 48 + d] + part[2 * 48 + d] + part[3 * 48 + d];
            if (actor && d < A) GR[ols + d] = part[24 + d] + part[48 + 24 + d] + part[96 + 24 + d] + part[144 + 24 + d] - (rs == 0 ? ecoef : 0.f);
        } else if (tid >= 96 && tid < 100 && nH + (tid - 96) < 4 * n4) {
            GR[nH + (tid - 96)] = 0.f;                      // padding of the last float4
        }
        if (tid == 0 && !a.grad_only) {   // Adam scalars of step k = step0 + s + 1, in double
            b1pow *= a.hy.beta1; b2pow *= a.hy.beta2;
            sh_d[0] = lr / (1.0 - b1pow);
            sh_d[1] = 1.0 / sqrt(1.0 - b2pow);
        }
        tc::tmem_st_wait();
        tc::tc_fence_before();
        TWT(29)
        sync_group<2>();                                   // every GR of the cluster is complete
        tc::tc_fence_after();
        TWT(30)

        // my slice: sum over the row-split CTAs of my half in fixed order, keep the sum in my own GR
        uint32_t peerGR[RS];
#pragma unroll
        for (int k = 0; k < RS; ++k) peerGR[k] = peer_base[k];        // GR starts at shared offset 0
        auto gslot = [&](int i4) {                          // float4 slot of half-local float4 index i4 inside GR
            const int e0 = 4 * i4;
            return (e0 >= oW2 && e0 < ob2) ? (NHP + ((e0 - oW2) >> 6) * GW2LD + ((e0 - oW2) & 63)) >> 2 : i4;
        };
        float sq = 0.f;
        constexpr int UB = 4;                               // slice items per batch: all loads of a batch are in flight together
        constexpr int NBATCH = (NU + UB - 1) / UB;
        // master / moment loads are software-pipelined one batch ahead; the first batch is issued here, before the gradient
        // reduction and the norm barrier, so its L2 round trip is hidden completely
        float4 pA[UB], mA[UB], vA[UB], pB[UB], mB[UB], vB[UB];
        auto ld_batch = [&](int u0, float4 *p4, float4 *m4, float4 *v4) {
#pragma unroll
            for (int uu = 0; uu < UB; ++uu) {
                const int i4 = slice_i4(u0 + uu);
                const int ic = (u0 + uu < NU && i4 < n4) ? i4 : 0;
                p4[uu] = ld_cg_f4(reinterpret_cast<const float4 *>(PMg) + ic);
                m4[uu] = ld_cg_f4(reinterpret_cast<const float4 *>(Mg) + ic);
                v4[uu] = ld_cg_f4(reinterpret_cast<const float4 *>(Vg) + ic);
            }
        };
        if (!a.grad_only) ld_batch(0, pA, mA, vA);
#pragma unroll 1
        for (int u0 = 0; u0 < NU; u0 += UB) {
            float4 part4[UB][RS];
#pragma unroll
            for (int uu = 0; uu < UB; ++uu) {
                const int i4 = slice_i4(u0 + uu);
                const int gs = gslot(i4 < n4 ? i4 : 0);
#pragma unroll
                for (int k = 0; k < RS; ++k)
                    part4[uu][k] = (k == rs) ? reinterpret_cast<const float4 *>(GR)[gs] : ld_dsmem4(peerGR[k] + 16u * (uint32_t)gs);
            }
#pragma unroll
            for (int uu = 0; uu < UB; ++uu) {
                const int i4 = slice_i4(u0 + uu);
                if (u0 + uu < NU && i4 < n4) {
                    float4 acc = part4[uu][0];
#pragma unroll
                    for (int k = 1; k < RS; ++k) { acc.x += part4[uu][k].x; acc.y += part4[uu][k].y; acc.z += part4[uu][k].z; acc.w += part4[uu][k].w; }
                    if (a.grad_only) {
                        const float gv[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (4 * i4 + e < nH) a.grad_out[(size_t)task * L.n_par + L.to_global(half, 4 * i4 + e)] = gv[e];
                    }
                    sq = fmaf(acc.x, acc.x, sq); sq = fmaf(acc.y, acc.y, sq); sq = fmaf(acc.z, acc.z, sq); sq = fmaf(acc.w, acc.w, sq);
                    // the sum replaces my own partial: a slot nobody else reads (peers read only THEIR slices of my GR)
                    reinterpret_cast<float4 *>(GR)[gslot(i4)] = acc;
                }
            }
        }
        if (a.grad_only) { sync_group<2>(); break; }        // peers' GRs stay valid until they have been read

        // squared norm: per-warp partials straight into every CTA of the cluster; the barrier is the only synchronisation
        sq = warp_sum(sq);
        float *ssq2 = ssqS + 64 * (s & 1);                  // slots alternate by step parity
        // (round 2) the norm exchange needs no cluster barrier: every partial travels with st.async and completes the
        // RECEIVER's mbarrier (8 warps x C CTAs x 4 bytes per step, the CTA's own partials included); what barrier (2) also
        // separated -- reading the peers' GR slices before, publishing new weights after -- is ordered by barriers (1) and (3)
        if (tid == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbarN)), "r"(32 * C) : "memory");
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < C; ++k)
                asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];"
                             ::"r"(mapa_u32(smem_u32(ssq2 + (int)rank * 8 + warp), (uint32_t)k)), "r"(__float_as_uint(sq)),
                               "r"(mapa_u32(smem_u32(mbarN), (uint32_t)k)) : "memory");
        }
        TWT(31)
        __syncthreads();                                    // sh_d (Adam scalars) written by thread 0
        tc::mbar_wait(mbarN, (uint32_t)(s & 1));
        TWT(32)
        float tot = 0.f;
#pragma unroll
        for (int i = 0; i < 8 * C; ++i) tot += ssq2[i];
        const float coef = fminf(1.f, (float)a.hy.max_grad_norm / (sqrtf(tot) + 1e-6f));
        const float step_size = (float)sh_d[0], ibc2 = (float)sh_d[1];
        auto adam_batch = [&](int u0, float4 *p4, float4 *m4, float4 *v4) {
#pragma unroll
            for (int uu = 0; uu < UB; ++uu) {
                const int i4 = slice_i4(u0 + uu);
                if (u0 + uu < NU && i4 < n4) {
                    const float4 g4 = reinterpret_cast<const float4 *>(GR)[gslot(i4)];
#define TW_ADAM(cc)                                                                         \
                    {                                                                       \
                        const float gq = g4.cc * coef;                                      \
                        m4[uu].cc = fmaf(gq - m4[uu].cc, omb1, m4[uu].cc);                  \
                        v4[uu].cc = fmaf(omb2 * gq, gq, v4[uu].cc * b2f);                   \
                        const float denom = fmaf(fast_sqrt(v4[uu].cc), ibc2, aeps);         \
                        p4[uu].cc -= step_size * __fdividef(m4[uu].cc, denom);              \
                    }
                    TW_ADAM(x) TW_ADAM(y) TW_ADAM(z) TW_ADAM(w)
#undef TW_ADAM
                    __stcg(reinterpret_cast<float4 *>(PMg) + i4, p4[uu]);
                    __stcg(reinterpret_cast<float4 *>(Mg) + i4, m4[uu]);
                    __stcg(reinterpret_cast<float4 *>(Vg) + i4, v4[uu]);
                    put4(4 * i4, p4[uu]);
                }
            }
        };
#pragma unroll 1
        for (int b = 0; b < NBATCH; b += 2) {               // two batches per trip: buffers A and B alternate statically
            if (b + 1 < NBATCH) ld_batch((b + 1) * UB, pB, mB, vB);
            adam_batch(b * UB, pA, mA, vA);
            if (b + 2 < NBATCH) ld_batch((b + 2) * UB, pA, mA, vA);
            if (b + 1 < NBATCH) adam_batch((b + 1) * UB, pB, mB, vB);
        }
        TWT(33)
        __threadfence();
        tc::fence_async_smem();
        tc::tc_fence_before();
        TWT(35)
        sync_group<2>();                                    // new weights are visible everywhere; my GR may be overwritten
        tc::tc_fence_after();
        TWT(34)
    }   // steps

    // ---------------- write back ----------------
    if (!a.grad_only) {
        for (int uq = 0; uq < NU; ++uq)
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = 4 * slice_i4(uq) + u;
                if (e < nH) {
                    const size_t gi = (size_t)task * L.n_par + L.to_global(half, e);
                    a.params[gi] = __ldcg(PMg + e); a.adam_m[gi] = __ldcg(Mg + e); a.adam_v[gi] = __ldcg(Vg + e);
                }
            }
    }
    {
        const float la = block_sum(loss_act, red), lv = block_sum(loss_val, red), le = block_sum(loss_ent, red);
        if (tid == 0) {
            a.lpart[(task * 16 + rank) * 4 + 0] = lv;
            a.lpart[(task * 16 + rank) * 4 + 1] = la;
            a.lpart[(task * 16 + rank) * 4 + 2] = le;
            __threadfence();
        }
    }
    tc::tc_fence_before();
    sync_group<2>();
    if (tid == 0 && rs == 0) {
        float lv = 0.f, la = 0.f, le = 0.f;
        for (int k = 0; k < RS; ++k) {
            lv += __ldcg(a.lpart + (task * 16 + half * RS + k) * 4 + 0);
            la += __ldcg(a.lpart + (task * 16 + half * RS + k) * 4 + 1);
            le += __ldcg(a.lpart + (task * 16 + half * RS + k) * 4 + 2);
        }
        const float ns = (float)a.nsteps;
        if (actor) {
            a.losses[task * 3 + 1] = la * inv_mb / ns;
            a.losses[task * 3 + 2] = le / ns;
            if (!a.grad_only) a.adam_step[task] = step0 + a.nsteps;
        } else {
            a.losses[task * 3 + 0] = lv * 0.5f / ((float)a.mb * M) / ns;
        }
    }
    if (warp == 0) tc::tmem_dealloc(tmem, 512);
}

}  // namespace pgm
