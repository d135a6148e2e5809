// K3 tensor-core path: the PPO minibatch loop (a2c/algo/ppo.py:62-107) on tcgen05 (UMMA kind::f16, FP32 accumulate
// in TMEM). Included by k3_ppo.cu (shares K3Args, k3_pack_kernel, fast_tanh, the DSMEM helpers).
//
// One cluster of 2 * RS CTAs per task: ranks [0, RS) = actor, [RS, 2 RS) = critic (the halves share only the global
// gradient norm); with RS = 2 the row tiles of every minibatch alternate between the two CTAs of a half (small
// populations: twice the SMs per task), which then add their gradients through DSMEM and run Adam redundantly.
// A CTA keeps its half's weights resident in shared memory as UMMA B operands and runs TWO independent 128-thread
// pipelines ("groups"); group g owns the 128-row tiles t = g, g+2, ... of every minibatch, thread = row = TMEM lane.
// While one group waits for its MMAs the other runs its epilogue, which hides the issue->complete latency of the
// dependent GEMM chain.  Per tile:
//   gather (coalesced, 8 lanes per 128-byte record, prefetched one pair ahead) -> x pair to the X image, scalars to smem
//   G1  Z1 = x W1^T (+b1 through a ones column);   E1  h1 = tanh(Z1) -> H1 image pair, 1 - h1^2 -> TMEM
//   G2  Z2 = h1 W2^T;                              E2  h2 = tanh(Z2 + b2) -> H2 image pair, 1 - h2^2 -> TMEM
//   G3  head = h2 Wh^T (N = 16);                   E3  per-row loss, d loss / d head -> X image (thread owns its row)
//   G4  dz2pre = dOut Wh;  GWh  dWh^T += h2^T dOut;  E4  dz2 = dz2pre (1 - h2^2) -> H2 image pair (in place)
//   G5  dz1pre = dz2 W2;   GW2  dW2 += dz2^T h1;     E5  dz1 = dz1pre (1 - h1^2) -> H1 image pair (in place)
//   G1X [dW1 | db1 ; db2] += [dz1 | dz2]^T [x | 1]
// Precision. Every GEMM operand is an FP16 PAIR a = a1 + a2 (a1 = a rounded to 11 significant bits, a2 = fp16(a - a1):
// 22 significant bits), held in power-of-two scaled form so that neither part underflows (activations and weights
// x 2^8, backward signals x 2^12; saturating conversions); a2*b1 + a1*b2 + a1*b1 with FP32 accumulation reproduces the
// FP32 product to ~2^-21 (gradients measured 3e-7 norm-wise against the float64 oracle, like the FP32 FFMA path).
// A pair costs 4 bytes per element, and ONE [row][64 halfwords] SWIZZLE_128B image serves both as a K-major operand
// (contraction over features: G1..G5) and as an MN-major operand (contraction over rows: the weight-gradient GEMMs).
// kind::tf32 cannot do that: its MN-major operands exist only in a special 32-byte-swizzle layout (see tc.cuh).
// Step tail: gradients TMEM -> shared memory in parameter order, squared-norm exchange with the peer CTA through
// DSMEM (one cluster barrier), clip + Adam on FP32 master parameters in shared memory (moments stream through an
// L2-resident workspace), new weights re-split into the operand images.
#pragma once
#include <cuda_fp16.h>

#include "tc.cuh"
#include "tc_pair.cuh"

namespace pgm {

constexpr int TC_THREADS = 256;              // 8 warps = lane quadrant (w & 3) x column half (w >> 2). 16 warps were measured
                                             // no faster: the tanh epilogues are bound by the XU pipe (MUFU ex2/rcp + fp16 packs)
constexpr uint32_t TC_GROUP_BYTES = 81920;   // H1a | H1b | H2a | H2b | X   (16 KB each, [128 rows][64 halfwords])
constexpr uint32_t TC_MISC_BYTES = 1280;
constexpr int TC_NHP = 6144;                 // padded size of one half's parameter vector (floats)

struct TcSmem {   // byte offsets inside dynamic shared memory
    uint32_t grp[2], W2a, W2b, W1, WhA1, WhA2, WhZ, PM, SC, misc, total;
};
__host__ __device__ inline TcSmem tc_smem_layout() {
    TcSmem s; uint32_t o = 0;
    s.grp[0] = o; o += TC_GROUP_BYTES; s.grp[1] = o; o += TC_GROUP_BYTES;
    s.W2a = o; o += 8192; s.W2b = o; o += 8192;               // [64 rows j][64 halfwords k] = W2[j][k] * 2^8 (a1 | a2)
    s.W1 = o; o += 8192;                                      // [64 rows j][features 0..31 a1 | 32..63 a2], column O = bias
    s.WhA1 = o; o += 1024; s.WhA2 = o; o += 1024; s.WhZ = o; o += 1024;   // [8 rows a][64 halfwords k]; Z = zero rows 8..15
    s.PM = o; o += TC_NHP * 4;                                // FP32 master parameters of the half, reference order
    s.SC = o; o += 2 * 128 * 48;                              // per-row scalars of the two tiles in flight (<= 12 floats per row)
    s.misc = o; o += TC_MISC_BYTES; s.total = o;
    return s;
}
// misc (floats): red[40] part[8][16] ssq[32] | at byte 1024: double sh_d[4], mbarriers, tmem ptr
constexpr int TCM_RED = 0, TCM_PART = 40, TCM_SSQ = 168;   // ssq: [2 step parities][2 ranks][8 warps]

// TMEM columns: group g at g*192: D1 [0,64) = 1 - h1^2, D2 [64,128) = 1 - h2^2, ACC [128,192) accumulators;
// weight-gradient accumulators shared by both groups
constexpr uint32_t TC_D1 = 0, TC_D2 = 64, TC_ACC = 128, TC_GSTRIDE = 192, TC_GW2 = 384, TC_G1X = 448, TC_GWH = 480;

// PGM_K3_TRACE builds: clock64 marks of threads r == 0 (MMA issuer) and r == 64 of each group, steps 8 and 9
// (profiles/k3_tc_trace.py): trace[(((cta*2 + group)*2 + who)*2 + step - 8)*48 + mark]
#ifdef PGM_K3_TRACE
#define TCT(i) if (trace_on) a.trace[trace_base + (i)] = clock64();
#else
#define TCT(i)
#endif

template <int O, int A, int M, int RS, bool VU = false>      // RS = CTAs per network half (row split): 1 or 2
__global__ void __launch_bounds__(TC_THREADS, 1) k3_tc_kernel(const K3Args a) {
    constexpr int OP = (O + 3) / 4 * 4;
    constexpr int NK1 = (O + 1 + 15) / 16;           // K steps of layer 1: x, ones column at index O, zero padding
    constexpr int NXC = (O + 1 + 7) / 8;             // 16-byte chunks of x (8 features each) written per row
    constexpr int RSG = (OP + A + 2 * M + 2 + 3) / 4 * 4;
    constexpr int NP = RSG / 4, NPX = OP / 4;        // 16-byte pieces per record; pieces that hold x
    constexpr int NIT = (128 * NP + TC_THREADS - 1) / TC_THREADS;    // gather items per thread per tile
    static_assert(O + 1 <= 24 && A <= 8 && M <= 8 && RSG <= 32 && O % 4 != 0 && RSG - OP <= 12, "k3_tc: dims outside the tensor-core path");
    extern __shared__ __align__(1024) unsigned char smem_raw[];

    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = tc::uniform_warp_idx();         // warp-uniform by construction: MMA operands stay in uniform registers
    const int g = warp >> 2, r = tid & 127;          // group, row inside the tile (= TMEM lane)
    const int q = warp & 3, hcol = warp >> 2;        // lane quadrant, column half used in the step tail
    const int task = blockIdx.x / (2 * RS);
    const unsigned rank = group_rank<2>();
    const int half = (int)rank / RS, rs = (int)rank % RS;
    const bool actor = half == 0;
    const int KH = actor ? A : M;
    const NetLayout &L = a.L;
    const TcSmem sl = tc_smem_layout();
    // half-local parameter offsets (reference order inside the half)
    constexpr int ob1 = H * O, oW2 = ob1 + H, ob2 = oW2 + H * H, oWh = ob2 + H;
    const int obh = oWh + KH * H, ols = obh + KH;
    const int nH = ols + (actor ? A : 0);
    const int n4 = (nH + 3) >> 2;

    unsigned char *sg = smem_raw + sl.grp[g & 1];
    unsigned char *S_h1 = sg, *S_h2 = sg + 32768, *S_x = sg + 65536;     // H1a|H1b, H2a|H2b, X
    __half *W2a = (__half *)(smem_raw + sl.W2a), *W2b = (__half *)(smem_raw + sl.W2b);
    __half *W1i = (__half *)(smem_raw + sl.W1);
    __half *WhA1 = (__half *)(smem_raw + sl.WhA1), *WhA2 = (__half *)(smem_raw + sl.WhA2);
    float *PM = (float *)(smem_raw + sl.PM);
    float *SC = (float *)(smem_raw + sl.SC);                            // [2 tiles][128 rows][12]
    float *GR = (float *)(smem_raw + sl.grp[0]);                         // gradient staging (step tail only), parameter order
    float *GRW2 = GR + TC_NHP;                                           // ... except dW2: rows padded to 68 floats, so that the
    constexpr int GW2LD = 68;                                            // 16 row-owner lanes of a warp store conflict free
    float *misc = (float *)(smem_raw + sl.misc);
    float *red = misc + TCM_RED, *part = misc + TCM_PART, *ssqS = misc + TCM_SSQ;
    double *sh_d = (double *)(smem_raw + sl.misc + 1024);
    uint64_t *mbars = (uint64_t *)(smem_raw + sl.misc + 1024 + 32);     // [0..1] chain (A), [2..3] weight grads (B)
    uint32_t *tmem_ptr_s = (uint32_t *)(smem_raw + sl.misc + 1024 + 64);
    uint64_t *mbarN = (uint64_t *)(smem_raw + sl.misc + 1024 + 72);     // counts the bytes of the peer's 8 squared-norm partials
    const float *b2s = PM + ob2, *bhs = PM + obh, *lss = PM + ols;

    // ---------------- one-time setup ----------------
    for (int i = tid; i < (int)(sl.total / 16); i += TC_THREADS) reinterpret_cast<float4 *>(smem_raw)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();
    if (warp == 0) tc::tmem_alloc(tmem_ptr_s, 512);
    if (tid == 0) {
        for (int i = 0; i < 4; ++i) tc::mbar_init(mbars + i, 1);
        tc::mbar_init(mbarN, 1);
        tc::fence_mbar_init();
    }
    const float *gpar = a.params + (size_t)task * L.n_par;
    // one parameter (half-local index e, value p) -> its operand images
    auto put_param = [&](int e, float p) {
        if (e < ob1) { const int j = e / O, c = e - j * O; put_pair(W1i, sw128_hw(j, c), W1i, sw128_hw(j, 32 + c), p * TC_SW); }
        else if (e < oW2) { const int j = e - ob1; put_pair(W1i, sw128_hw(j, O), W1i, sw128_hw(j, 32 + O), p * TC_SW); }
        else if (e < ob2) { const int j = (e - oW2) >> 6, k = (e - oW2) & 63; put_pair(W2a, sw128_hw(j, k), W2b, sw128_hw(j, k), p * TC_SW); }
        else if (e >= oWh && e < obh) { const int aa = (e - oWh) >> 6, k = (e - oWh) & 63; put_pair(WhA1, sw128_hw(aa, k), WhA2, sw128_hw(aa, k), p * TC_SW); }
    };
    for (int e = tid; e < nH; e += TC_THREADS) {
        const float p = __ldg(gpar + L.to_global(half, e));
        PM[e] = p;
        put_param(e, p);
    }
    // Adam moments: reference order -> half-local order in the workspace
    float *wM = a.mv + ((size_t)((task * 2 + half) * RS + rs) * 2) * TC_NHP, *wV = wM + TC_NHP;   // one copy per CTA
    if (!a.grad_only)
        for (int e = tid; e < 4 * n4; e += TC_THREADS) {
            const bool in = e < nH;
            const size_t gi = (size_t)task * L.n_par + (in ? L.to_global(half, e) : 0);
            wM[e] = in ? a.adam_m[gi] : 0.f; wV[e] = in ? a.adam_v[gi] : 0.f;
        }
    tc::fence_async_smem();
    tc::tc_fence_before();
    sync_group<2>();                 // barrier inits + TMEM address visible; peer CTA is alive before any DSMEM store
    tc::tc_fence_after();
    const uint32_t tmem = tc::uniform_u32(*tmem_ptr_s);
    const uint32_t tq = tmem + ((uint32_t)(q * 32) << 16);          // my lane quadrant
    const uint32_t tg = tq + (uint32_t)g * TC_GSTRIDE;              // + my group's column window

    {   // zero the weight-gradient accumulators (each thread: the cells it will read in the step tail)
        float z[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) z[i] = 0.f;
        tc::tmem_st32(tq + TC_GW2 + 32 * hcol, z);
        tc::tmem_st16(tq + TC_G1X + 16 * hcol, z);
        if (hcol == 0) tc::tmem_st8(tq + TC_GWH, z);
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
    const float *recg = a.rec + (size_t)task * a.S * RSG;
    const int ntiles_all = (a.mb + 127) >> 7;
    const int ntiles = rs < ntiles_all ? (ntiles_all - rs + RS - 1) / RS : 0;    // my tiles: global tile = local * RS + rs
    uint32_t phA[2] = {0u, 0u}, phB[2] = {0u, 0u};    // mbarrier phase parities (per tile of the pair)
    bool pendB[2] = {false, false};

    // ---- descriptors of tile 0 (tile 1: + TC_GROUP_BYTES); images are [rows][64 halfwords], SWIZZLE_128B ----
    // K-major view (M/N = row, K = feature): SBO = 1024 (next 8 rows), +32 B per K step of 16 features.
    // MN-major view (M/N = feature, K = row): LBO = stride to the next 64-feature block, SBO = 1024 (next 8 K rows),
    // +2048 B per K step of 16 rows.
    const uint32_t aH1 = tc::smem_addr(smem_raw + sl.grp[0]), aH2 = aH1 + 32768, aX = aH1 + 65536;
    const uint32_t aW1 = tc::smem_addr(W1i), aW2a = tc::smem_addr(W2a), aW2b = tc::smem_addr(W2b);
    const uint32_t aWh1 = tc::smem_addr(WhA1), aWh2 = tc::smem_addr(WhA2);
    auto dK = [](uint32_t addr) { return tc::make_desc(addr, 16, 1024, 2); };
    auto dMN = [](uint32_t addr, uint32_t lbo) { return tc::make_desc(addr, lbo, 1024, 2); };
    const uint64_t dXa_k = dK(aX), dXb_k = dK(aX + 64), dW1a_k = dK(aW1), dW1b_k = dK(aW1 + 64);
    const uint64_t dH1a_k = dK(aH1), dH1b_k = dK(aH1 + 16384), dH2a_k = dK(aH2), dH2b_k = dK(aH2 + 16384);
    const uint64_t dW2a_k = dK(aW2a), dW2b_k = dK(aW2b);
    // head weights: 8 real rows; rows 8..15 come from the shared zero block (SBO = distance to WhZ)
    const uint64_t dWh1_k = tc::make_desc(aWh1, 16, 2048, 2), dWh2_k = tc::make_desc(aWh2, 16, 1024, 2);
    const uint64_t dWh1_mn = tc::make_desc(aWh1, 16384, 2048, 2), dWh2_mn = tc::make_desc(aWh2, 16384, 1024, 2);
    const uint64_t dXdo_a = dK(aX + 48), dXdo_b = dK(aX + 112);      // K windows that start at dOut a1 / dOut a2
    const uint64_t dW2a_mn = dMN(aW2a, 16384), dW2b_mn = dMN(aW2b, 16384);
    const uint64_t dH1a_mn = dMN(aH1, 32768), dH1b_mn = dMN(aH1 + 16384, 32768);     // [H1 | H2] stacks to M = 128
    const uint64_t dH2a_mn = dMN(aH2, 32768), dH2b_mn = dMN(aH2 + 16384, 32768);
    const uint64_t dXa_mn = dMN(aX, 16384), dXb_mn = dMN(aX + 64, 16384);             // features 0..31 | 32..63
    const uint64_t dXa_do = dMN(aX + 48, 16384), dXb_do = dMN(aX + 112, 16384);       // dOut: 24..31 | 56..63
    constexpr uint32_t ID_KK = tc::idesc_f16(128, 64, 0, 0), ID_HEAD = tc::idesc_f16(128, 16, 0, 0), ID_KM = tc::idesc_f16(128, 64, 0, 1);
    constexpr uint32_t ID_GWH = tc::idesc_f16(64, 8, 1, 1), ID_GW2 = tc::idesc_f16(64, 64, 1, 1), ID_G1X = tc::idesc_f16(128, 32, 1, 1);
    const uint32_t swz = (uint32_t)(r & 7);
    unsigned char *rowx = S_x + r * 128;             // my row of my group's X image (gather, E3)

    // everything I wrote (TMEM, smem images) is complete and ordered before the MMAs issued after the barrier
    auto sync_all = [&]() { tc::tmem_st_wait(); tc::tmem_ld_wait(); tc::fence_async_smem(); tc::tc_fence_before(); __syncthreads(); };
    // 3 MMAs of one K step: a2*b1 + a1*b2 + a1*b1 (small terms first)
    auto mma3 = [&](uint32_t d, uint64_t a1, uint64_t a2, uint64_t b1, uint64_t b2, uint32_t id, uint32_t acc) {
        tc::mma_f16(d, a2, b1, id, acc); tc::mma_f16(d, a1, b2, id, 1); tc::mma_f16(d, a1, b1, id, 1);
    };

    // Record gather, cooperative and coalesced: item f = tid + 256 k of a tile is (row f / NP, 16-byte piece f % NP), so a
    // warp instruction reads whole 128-byte lines. x pieces go straight into the X image (fp16 pair), scalar pieces into
    // SC for the row's owner (E3). The records of the NEXT pair and the row indices of the pair after it are in flight.
    float4 rcv[2][NIT];
    int ridx[2][NIT];
    auto pair_after = [&](int &ss, int &tt) { if (tt + 2 < ntiles) tt += 2; else { ss += 1; tt = 0; } };
    // Loads are issued unconditionally from clamped addresses and masked when CONSUMED: a select on a load's result
    // would make the issuing thread wait for it (8 serialised L2 round trips instead of 8 loads in flight).
    uint32_t vm_idx = 0u, vm_rec = 0u;             // bit (i * NIT + k): item k of tile i is a real row (indices / records in flight)
    auto load_idx = [&](int ss, int tt) {
        const bool sv = ss < a.nsteps;
        const int sc_ = sv ? ss : 0;
        const int ep = sc_ / a.B, bb = sc_ - ep * a.B;
        const int32_t *pb = perm + (size_t)ep * a.S + (size_t)bb * a.mb;
        vm_idx = 0u;
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int k = 0; k < NIT; ++k) {
                const int f = tid + TC_THREADS * k, rowi = ((tt + i) * RS + rs) * 128 + f / NP;
                const bool ok = sv && tt + i < ntiles && f < 128 * NP && rowi < a.mb;
                ridx[i][k] = ld_nc_s32(pb + (ok ? rowi : 0));
                vm_idx |= (ok ? 1u : 0u) << (i * NIT + k);
            }
    };
    auto load_recs = [&]() {
        vm_rec = vm_idx;
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int k = 0; k < NIT; ++k) {
                const int f = tid + TC_THREADS * k;
                rcv[i][k] = ld_nc_f4(reinterpret_cast<const float4 *>(recg + (size_t)ridx[i][k] * RSG) + f % NP);
            }
    };
    load_idx(0, 0);
    load_recs();
    {
        int ss = 0, tt = 0;
        pair_after(ss, tt);
        load_idx(ss, tt);
    }

    for (int s = 0; s < a.nsteps; ++s) {
#ifdef PGM_K3_TRACE
        const bool trace_on = a.trace && (s == 8 || s == 9) && (r == 0 || r == 64);
        const size_t trace_base = ((((size_t)blockIdx.x * 2 + g) * 2 + (r == 64)) * 2 + (s - 8)) * 48;
#endif
        float gbh[8], gls[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { gbh[i] = 0.f; gls[i] = 0.f; }
        if (actor && rs == 0 && tid == 0) {   // entropy with the parameters this step starts from
            float ent = 0.f;
            for (int d = 0; d < A; ++d) ent += 0.5f + 0.91893853320467274178f + lss[d];
            loss_ent += ent;
        }

        // Tiles are processed in PAIRS (tile tp by group 0, tile tp + 1 by group 1 for the per-row phases). The 64-column
        // epilogues of EACH tile are done by all 8 warps (warp = lane quadrant x column half), tile 0 then tile 1, so an
        // epilogue takes half as long and always runs under the other tile's MMAs:
        //   E(0) | issue G(0) | E(1) [G(0) runs] | issue G(1) | next E(0) [G(1) runs] ...
        for (int tp = 0; tp < ntiles; tp += 2) {
            const bool hasB = tp + 1 < ntiles;
            const int nt = hasB ? 2 : 1;
            const bool mine = g < nt;                      // my group's tile tp + g exists
            TCT(0)
#pragma unroll
            for (int i = 0; i < 2; ++i)                    // previous pair's weight-gradient MMAs released X / H1 / H2
                if (pendB[i]) { tc::mbar_wait(mbars + 2 + i, phB[i]); phB[i] ^= 1; pendB[i] = false; }
            tc::tc_fence_after();
            TCT(39)
            // ---------------- records -> X image pair (x, ones column) and SC (per-row scalars) ----------------
            const uint32_t vm_now = vm_rec;
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int k = 0; k < NIT; ++k) {
                    const int f = tid + TC_THREADS * k;
                    if (i < nt && f < 128 * NP) {
                        const int row = f / NP, pc = f % NP;
                        const bool ok = (vm_now >> (i * NIT + k)) & 1u;
                        const float4 v = ok ? rcv[i][k] : make_float4(0.f, 0.f, 0.f, 0.f);
                        if (pc < NPX) {
                            float xv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                            for (int e = 0; e < 4; ++e) if (4 * pc + e >= O) xv[e] = (4 * pc + e == O && ok) ? 1.f : 0.f;
                            const float h0 = round11(xv[0]), h1 = round11(xv[1]), h2 = round11(xv[2]), h3 = round11(xv[3]);
                            unsigned char *xr = smem_raw + sl.grp[i] + 65536 + row * 128 + (pc & 1) * 8;
                            const uint32_t c = (uint32_t)(pc >> 1), sw = (uint32_t)(row & 7);
                            *reinterpret_cast<uint2 *>(xr + ((c ^ sw) << 4)) = make_uint2(pack_h2_ovf(h0, h1), pack_h2_ovf(h2, h3));
                            *reinterpret_cast<uint2 *>(xr + (((c + 4u) ^ sw) << 4)) =
                                make_uint2(pack_h2_ovf(xv[0] - h0, xv[1] - h1), pack_h2_ovf(xv[2] - h2, xv[3] - h3));
                        } else {
                            *reinterpret_cast<float4 *>(SC + (i * 128 + row) * 12 + 4 * (pc - NPX)) = v;
                        }
                    }
                }
            TCT(40)
            // prefetch: records of the next pair (their row indices arrived long ago), row indices of the pair after it
            load_recs();
            TCT(41)
            {
                int ss = s, tt = tp;
                pair_after(ss, tt); pair_after(ss, tt);
                load_idx(ss, tt);
            }
            TCT(42)
            TCT(1)
            sync_all();
            if (warp == 0 && tc::elect_one()) {
                tc::tc_fence_after();
                for (int i = 0; i < nt; ++i) {
                    const uint32_t so = (uint32_t)i * TC_GROUP_BYTES, acc = tmem + (uint32_t)i * TC_GSTRIDE + TC_ACC;
#pragma unroll
                    for (int ks = 0; ks < NK1; ++ks)
                        mma3(acc, tc::desc_advance(dXa_k, so + 32 * ks), tc::desc_advance(dXb_k, so + 32 * ks),
                             tc::desc_advance(dW1a_k, 32 * ks), tc::desc_advance(dW1b_k, 32 * ks), ID_KK, ks > 0);
                    tc::mma_commit(mbars + i);
                }
            }
            TCT(2)
            // ---------------- E1: h1 = tanh(Z1) -> H1 pair, 1 - h1^2 -> TMEM ----------------
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if (i >= nt) break;
                unsigned char *rowh1 = smem_raw + sl.grp[i] + r * 128;
                const uint32_t tt = tq + (uint32_t)i * TC_GSTRIDE;
                tc::mbar_wait(mbars + i, phA[i]); phA[i] ^= 1; tc::tc_fence_after();
                TCT(3 + 3 * i)
                float z[32], dd[32];
                tc::tmem_ld32(tt + TC_ACC + 32 * hcol, z);
                tc::tmem_ld_wait();
#pragma unroll
                for (int k = 0; k < 32; ++k) { z[k] = fast_tanh(z[k] * (1.f / TC_SW)); dd[k] = fmaf(-z[k], z[k], 1.f); z[k] *= TC_SH; }
                tc::tmem_st32(tt + TC_D1 + 32 * hcol, dd);
#pragma unroll
                for (int c = 0; c < 4; ++c) store_pair8(rowh1, (uint32_t)(4 * hcol + c), rowh1 + 16384, (uint32_t)(4 * hcol + c), swz, z + 8 * c);
                TCT(4 + 3 * i)
                sync_all();
                if (warp == 0 && tc::elect_one()) {
                    tc::tc_fence_after();
                    const uint32_t so = (uint32_t)i * TC_GROUP_BYTES, acc = tmem + (uint32_t)i * TC_GSTRIDE + TC_ACC;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        mma3(acc, tc::desc_advance(dH1a_k, so + 32 * ks), tc::desc_advance(dH1b_k, so + 32 * ks),
                             tc::desc_advance(dW2a_k, 32 * ks), tc::desc_advance(dW2b_k, 32 * ks), ID_KK, ks > 0);
                    tc::mma_commit(mbars + i);
                }
                TCT(5 + 3 * i)
            }
            // ---------------- E2: h2 = tanh(Z2 + b2) -> H2 pair, 1 - h2^2 -> TMEM ----------------
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if (i >= nt) break;
                unsigned char *rowh2 = smem_raw + sl.grp[i] + 32768 + r * 128;
                const uint32_t tt = tq + (uint32_t)i * TC_GSTRIDE;
                tc::mbar_wait(mbars + i, phA[i]); phA[i] ^= 1; tc::tc_fence_after();
                TCT(9 + 3 * i)
                float z[32], dd[32];
                tc::tmem_ld32(tt + TC_ACC + 32 * hcol, z);
                tc::tmem_ld_wait();
#pragma unroll
                for (int k = 0; k < 32; k += 4) {
                    const float4 bv = *reinterpret_cast<const float4 *>(b2s + 32 * hcol + k);
                    z[k] = fmaf(z[k], 1.f / (TC_SH * TC_SW), bv.x); z[k + 1] = fmaf(z[k + 1], 1.f / (TC_SH * TC_SW), bv.y);
                    z[k + 2] = fmaf(z[k + 2], 1.f / (TC_SH * TC_SW), bv.z); z[k + 3] = fmaf(z[k + 3], 1.f / (TC_SH * TC_SW), bv.w);
                }
#pragma unroll
                for (int k = 0; k < 32; ++k) { z[k] = fast_tanh(z[k]); dd[k] = fmaf(-z[k], z[k], 1.f); z[k] *= TC_SH; }
                tc::tmem_st32(tt + TC_D2 + 32 * hcol, dd);
#pragma unroll
                for (int c = 0; c < 4; ++c) store_pair8(rowh2, (uint32_t)(4 * hcol + c), rowh2 + 16384, (uint32_t)(4 * hcol + c), swz, z + 8 * c);
                TCT(10 + 3 * i)
                sync_all();
                if (warp == 0 && tc::elect_one()) {
                    tc::tc_fence_after();
                    const uint32_t so = (uint32_t)i * TC_GROUP_BYTES, acc = tmem + (uint32_t)i * TC_GSTRIDE + TC_ACC;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        mma3(acc, tc::desc_advance(dH2a_k, so + 32 * ks), tc::desc_advance(dH2b_k, so + 32 * ks),
                             tc::desc_advance(dWh1_k, 32 * ks), tc::desc_advance(dWh2_k, 32 * ks), ID_HEAD, ks > 0);
                    tc::mma_commit(mbars + i);
                }
                TCT(11 + 3 * i)
            }
            // ---------------- E3: per-row loss and d loss / d head (each group its own tile) ----------------
            if (mine) {
                tc::mbar_wait(mbars + g, g == 0 ? phA[0] : phA[1]); tc::tc_fence_after();
                TCT(15)
                float ho[8], dq[8];
                tc::tmem_ld8(tg + TC_ACC, ho);
                // my row's scalars: action[A] | logp_old | value_old[M] | return[M] | advantage
                float sc[12];
                {
                    const float4 *sp = reinterpret_cast<const float4 *>(SC + (g * 128 + r) * 12);
                    const float4 s0 = sp[0], s1 = sp[1], s2 = sp[2];
                    sc[0] = s0.x; sc[1] = s0.y; sc[2] = s0.z; sc[3] = s0.w; sc[4] = s1.x; sc[5] = s1.y; sc[6] = s1.z; sc[7] = s1.w;
                    sc[8] = s2.x; sc[9] = s2.y; sc[10] = s2.z; sc[11] = s2.w;
                }
                const bool row_valid = ((tp + g) * RS + rs) * 128 + r < a.mb;
                tc::tmem_ld_wait();
                if (actor) {
                    float lp = 0.f, diffv[8], ivv[8];
#pragma unroll
                    for (int d = 0; d < 8; ++d) {
                        diffv[d] = 0.f; ivv[d] = 0.f;
                        if (d < A) {
                            const float ls = lss[d];
                            const float iv = expf(-2.f * ls);
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
                    for (int d = 0; d < 8; ++d) {
                        const float go = dlp * diffv[d] * ivv[d];                 // d loss / d mean
                        gbh[d] += go;
                        gls[d] = fmaf(dlp, diffv[d] * diffv[d] * ivv[d] - (d < A ? 1.f : 0.f), gls[d]);
                        dq[d] = go * TC_SD;
                    }
                } else {
#pragma unroll
                    for (int m = 0; m < 8; ++m) {
                        float go = 0.f;
                        if (m < M) {
                            const float V = fmaf(ho[m], 1.f / (TC_SH * TC_SW), bhs[m]), vo = sc[A + 1 + m], R = sc[A + 1 + M + m];
                            const float dlt = V - vo;
                            const float vcl = vo + fminf(fmaxf(dlt, -clip), clip);
                            const float ea = V - R, eb = vcl - R;
                            // unclipped value loss (VU): lb = -1 < 0 <= la, so max(la, lb) = la and wa = 1, gradient 2 * ea exactly
                            const float la = ea * ea, lb = VU ? -1.f : eb * eb;
                            const float wa = la > lb ? 1.f : (la == lb ? 0.5f : 0.f);
                            const float pas = (dlt >= -clip && dlt <= clip) ? 1.f : 0.f;
                            if (row_valid) { loss_val += fmaxf(la, lb); go = vscale * (wa * 2.f * ea + (1.f - wa) * 2.f * eb * pas); }
                        }
                        gbh[m] += go;
                        dq[m] = go * TC_SD;
                    }
                }
                store_pair8(rowx, 3u, rowx, 7u, swz, dq);          // a1 in features 24..31, a2 in features 56..63
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) if (i < nt) phA[i] ^= 1;   // both head GEMMs are complete once the barrier below is passed
            TCT(16)
            sync_all();
            if (warp == 0 && tc::elect_one()) {
                tc::tc_fence_after();
                for (int i = 0; i < nt; ++i) {
                    const uint32_t so = (uint32_t)i * TC_GROUP_BYTES, acc = tmem + (uint32_t)i * TC_GSTRIDE + TC_ACC;
                    // dz2pre = dOut Wh: K window of 16 X features starting at dOut against [Wh rows 0..7 | zero rows]
                    mma3(acc, tc::desc_advance(dXdo_a, so), tc::desc_advance(dXdo_b, so), dWh1_mn, dWh2_mn, ID_KM, 0);
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)                                                 // dWh^T += h2^T dOut
                        mma3(tmem + TC_GWH, tc::desc_advance(dH2a_mn, so + 2048 * ks), tc::desc_advance(dH2b_mn, so + 2048 * ks),
                             tc::desc_advance(dXa_do, so + 2048 * ks), tc::desc_advance(dXb_do, so + 2048 * ks), ID_GWH, 1);
                    tc::mma_commit(mbars + i);
                }
            }
            TCT(17)
            // ---------------- E4: dz2 = dz2pre (1 - h2^2) -> H2 pair (in place) ----------------
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if (i >= nt) break;
                unsigned char *rowh2 = smem_raw + sl.grp[i] + 32768 + r * 128;
                const uint32_t tt = tq + (uint32_t)i * TC_GSTRIDE;
                tc::mbar_wait(mbars + i, phA[i]); phA[i] ^= 1; tc::tc_fence_after();
                TCT(18 + 3 * i)
                float z[32], dd[32];
                tc::tmem_ld32(tt + TC_ACC + 32 * hcol, z);
                tc::tmem_ld32(tt + TC_D2 + 32 * hcol, dd);
                tc::tmem_ld_wait();
#pragma unroll
                for (int k = 0; k < 32; ++k) z[k] = z[k] * (1.f / TC_SW) * dd[k];           // dz2 (still x 2^12)
#pragma unroll
                for (int c = 0; c < 4; ++c) store_pair8(rowh2, (uint32_t)(4 * hcol + c), rowh2 + 16384, (uint32_t)(4 * hcol + c), swz, z + 8 * c);
                TCT(19 + 3 * i)
                sync_all();
                if (warp == 0 && tc::elect_one()) {
                    tc::tc_fence_after();
                    const uint32_t so = (uint32_t)i * TC_GROUP_BYTES, acc = tmem + (uint32_t)i * TC_GSTRIDE + TC_ACC;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)                                                 // dz1pre = dz2 W2
                        mma3(acc, tc::desc_advance(dH2a_k, so + 32 * ks), tc::desc_advance(dH2b_k, so + 32 * ks),
                             tc::desc_advance(dW2a_mn, 2048 * ks), tc::desc_advance(dW2b_mn, 2048 * ks), ID_KM, ks > 0);
                    tc::mma_commit(mbars + i);
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)                                                 // dW2 += dz2^T h1
                        mma3(tmem + TC_GW2, tc::desc_advance(dH2a_mn, so + 2048 * ks), tc::desc_advance(dH2b_mn, so + 2048 * ks),
                             tc::desc_advance(dH1a_mn, so + 2048 * ks), tc::desc_advance(dH1b_mn, so + 2048 * ks), ID_GW2, 1);
                    tc::mma_commit(mbars + 2 + i);
                }
                TCT(20 + 3 * i)
            }
            // ---------------- E5: dz1 = dz1pre (1 - h1^2) -> H1 pair (in place) ----------------
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if (i >= nt) break;
                unsigned char *rowh1 = smem_raw + sl.grp[i] + r * 128;
                const uint32_t tt = tq + (uint32_t)i * TC_GSTRIDE;
                tc::mbar_wait(mbars + i, phA[i]); phA[i] ^= 1; tc::tc_fence_after();
                TCT(24 + 4 * i)
                float z[32], dd[32];
                tc::tmem_ld32(tt + TC_ACC + 32 * hcol, z);
                tc::tmem_ld32(tt + TC_D1 + 32 * hcol, dd);
                tc::tmem_ld_wait();
#pragma unroll
                for (int k = 0; k < 32; ++k) z[k] = z[k] * (1.f / TC_SW) * dd[k];
                TCT(25 + 4 * i)
                tc::mbar_wait(mbars + 2 + i, phB[i]); phB[i] ^= 1;     // dW2 MMAs are done reading h1
                TCT(26 + 4 * i)
#pragma unroll
                for (int c = 0; c < 4; ++c) store_pair8(rowh1, (uint32_t)(4 * hcol + c), rowh1 + 16384, (uint32_t)(4 * hcol + c), swz, z + 8 * c);
                sync_all();
                if (warp == 0 && tc::elect_one()) {
                    tc::tc_fence_after();
                    const uint32_t so = (uint32_t)i * TC_GROUP_BYTES;
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks)              // [dW1 | db1 ; db2] += [dz1 | dz2]^T [x | 1 | dOut]
                        mma3(tmem + TC_G1X, tc::desc_advance(dH1a_mn, so + 2048 * ks), tc::desc_advance(dH1b_mn, so + 2048 * ks),
                             tc::desc_advance(dXa_mn, so + 2048 * ks), tc::desc_advance(dXb_mn, so + 2048 * ks), ID_G1X, 1);
                    tc::mma_commit(mbars + 2 + i);
                }
                pendB[i] = true;
                TCT(27 + 4 * i)
            }
        }   // tile pairs

        // ================= step tail =================
        // Gradients: TMEM -> GR (shared memory, parameter order); every accumulator cell is handed back zeroed by the thread
        // that read it. GR aliases tile 0's buffers, free once ITS last weight-gradient MMAs are done; the dW2 / dWh
        // accumulators are complete by then (their commits were waited for in E5), so they are drained while tile 1's
        // last GEMM (G1X) is still running.
        if (pendB[0]) { tc::mbar_wait(mbars + 2, phB[0]); phB[0] ^= 1; pendB[0] = false; }
        tc::tc_fence_after();
        TCT(32)
        {
            float gw[32], gh[8], z[32];
            tc::tmem_ld32(tq + TC_GW2 + 32 * hcol, gw);
            if (hcol == 0) tc::tmem_ld8(tq + TC_GWH, gh);
            tc::tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) z[i] = 0.f;
            tc::tmem_st32(tq + TC_GW2 + 32 * hcol, z);
            if (hcol == 0) tc::tmem_st8(tq + TC_GWH, z);
            if (lane < 16) {                               // dW2 rows: (dz2 2^12)^T (h1 2^8)
                float *dst = GRW2 + (16 * q + lane) * GW2LD + 32 * hcol;
#pragma unroll
                for (int i = 0; i < 32; i += 4)
                    *reinterpret_cast<float4 *>(dst + i) = make_float4(gw[i] * (1.f / (TC_SD * TC_SH)), gw[i + 1] * (1.f / (TC_SD * TC_SH)),
                                                                         gw[i + 2] * (1.f / (TC_SD * TC_SH)), gw[i + 3] * (1.f / (TC_SD * TC_SH)));
                if (hcol == 0) {                           // dWh^T rows: (h2 2^8)^T (dOut 2^12)
                    const int k = 16 * q + lane;
#pragma unroll
                    for (int aa = 0; aa < 8; ++aa)
                        if (aa < KH) GR[oWh + aa * H + k] = gh[aa] * (1.f / (TC_SD * TC_SH));
                }
            }
        }
        // head bias / logstd gradients: per-thread row sums -> warp -> CTA
        constexpr int KHM = A > M ? A : M;
#pragma unroll
        for (int i = 0; i < KHM; ++i) gbh[i] = warp_sum(gbh[i]);
        if (actor) {
#pragma unroll
            for (int i = 0; i < A; ++i) gls[i] = warp_sum(gls[i]);
        }
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) { part[warp * 16 + i] = gbh[i]; part[warp * 16 + 8 + i] = gls[i]; }
        }
        if (tid == 0 && !a.grad_only) {   // Adam scalars of step k = step0 + s + 1, in double
            b1pow *= a.hy.beta1; b2pow *= a.hy.beta2;
            sh_d[0] = lr / (1.0 - b1pow);
            sh_d[1] = 1.0 / sqrt(1.0 - b2pow);
        }
        if (pendB[1]) { tc::mbar_wait(mbars + 3, phB[1]); phB[1] ^= 1; pendB[1] = false; }
        tc::tc_fence_after();
        TCT(33)
        {
            float gx[16], z[16];
            tc::tmem_ld16(tq + TC_G1X + 16 * hcol, gx);
            tc::tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) z[i] = 0.f;
            tc::tmem_st16(tq + TC_G1X + 16 * hcol, z);
            if (q < 2) {                                   // dW1 | db1 rows: (dz1 2^12)^T [x | 1]
                const int j = 32 * q + lane;
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const int c = 16 * hcol + i;
                    if (c < O) GR[j * O + c] = gx[i] * (1.f / TC_SD);
                    else if (c == O) GR[ob1 + j] = gx[i] * (1.f / TC_SD);
                }
            } else if (hcol == O / 16) {                   // db2: (dz2 2^12)^T 1
                GR[ob2 + 32 * (q - 2) + lane] = gx[O % 16] * (1.f / TC_SD);
            }
        }
        __syncthreads();
        if (tid < 8) {
            float sb = 0.f, sl_ = 0.f;
#pragma unroll
            for (int w = 0; w < 8; ++w) { sb += part[w * 16 + tid]; sl_ += part[w * 16 + 8 + tid]; }
            if (tid < KH) GR[obh + tid] = sb;
            if (actor && tid < A) GR[ols + tid] = sl_ - (rs == 0 ? ecoef : 0.f);   // d(-ecoef * entropy) / d logstd = -ecoef, once
        }
        if (tid < 4 && nH + tid < 4 * n4) GR[nH + tid] = 0.f;            // padding of the last float4
        __syncthreads();
        TCT(34)

        // row split: the other CTA of my half holds the gradient of the other tiles in ITS GR (same offset)
        uint32_t peerGR = 0;
        if (RS > 1) {
            sync_group<2>();                                   // both GRs complete
            peerGR = mapa_u32(smem_u32(GR), (uint32_t)(half * RS + (rs ^ 1)));
        }
        if (a.grad_only) {
            if (rs == 0)
                for (int e = tid; e < nH; e += TC_THREADS) {
                    const int ge = (e >= oW2 && e < ob2) ? TC_NHP + ((e - oW2) >> 6) * GW2LD + ((e - oW2) & 63) : e;   // staging slot
                    float gsum = GR[ge];
                    if (RS > 1) { float pv; asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(pv) : "r"(peerGR + 4u * (uint32_t)ge) : "memory"); gsum += pv; }
                    a.grad_out[(size_t)task * L.n_par + L.to_global(half, e)] = gsum;
                }
            if (RS > 1) sync_group<2>();                       // the peer's GR stays valid until it has been read
            break;
        }

        // my float4 slices of the half: gradient from GR, moments from the workspace (in flight across the barrier)
        constexpr int NS = (TC_NHP / 4 + TC_THREADS - 1) / TC_THREADS;      // 6
        float4 g4[NS], m4[NS], v4[NS];
        float sq = 0.f;
        {
            float4 pg[NS];
#pragma unroll
            for (int u = 0; u < NS; ++u) {                     // all loads first (shared memory, peer DSMEM, L2), then the sums
                const int i4 = tid + u * TC_THREADS;
                if (i4 < n4) {
                    const int e0 = 4 * i4;
                    const int gi4 = (e0 >= oW2 && e0 < ob2) ? (TC_NHP + ((e0 - oW2) >> 6) * GW2LD + ((e0 - oW2) & 63)) >> 2 : i4;   // staging slot
                    g4[u] = reinterpret_cast<const float4 *>(GR)[gi4];
                    if (RS > 1) pg[u] = ld_dsmem4(peerGR + 16u * (uint32_t)gi4);
                    m4[u] = ld_cg_f4(reinterpret_cast<const float4 *>(wM) + i4);
                    v4[u] = ld_cg_f4(reinterpret_cast<const float4 *>(wV) + i4);
                }
            }
#pragma unroll
            for (int u = 0; u < NS; ++u) {
                const int i4 = tid + u * TC_THREADS;
                if (i4 < n4) {
                    if (RS > 1) {                              // fixed order (rs 0 + rs 1): both CTAs get identical sums
                        const float4 lo4 = rs == 0 ? g4[u] : pg[u], hi4 = rs == 0 ? pg[u] : g4[u];
                        g4[u] = make_float4(lo4.x + hi4.x, lo4.y + hi4.y, lo4.z + hi4.z, lo4.w + hi4.w);
                    }
                    sq = fmaf(g4[u].x, g4[u].x, sq); sq = fmaf(g4[u].y, g4[u].y, sq);
                    sq = fmaf(g4[u].z, g4[u].z, sq); sq = fmaf(g4[u].w, g4[u].w, sq);
                }
            }
        }
        // squared norm: per-warp partials go to my own slots and straight to the peer CTA; the cluster barrier is the
        // only synchronisation, every thread then adds the 16 partials in one fixed order
        sq = warp_sum(sq);
        float *ssq2 = ssqS + 16 * (s & 1);    // slots alternate by step parity: the peer may still be reading the last ones
        // (round 2) no cluster barrier: the partials travel with st.async and complete the PEER's mbarrier (8 x 4 bytes per
        // step); slots alternate by step parity, and a CTA cannot run more than one step ahead of its peer because it needs
        // the peer's partials of every step -- so a slot is never rewritten while it is still being read
        if (tid == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbarN)), "r"(32) : "memory");
        if (lane == 0) {                      // my half's partials -> me and the CTA of the other half with my row-split index
            ssq2[half * 8 + warp] = sq;
            const uint32_t peer = (uint32_t)((1 - half) * RS + rs);
            asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];"
                         ::"r"(mapa_u32(smem_u32(ssq2 + half * 8 + warp), peer)), "r"(__float_as_uint(sq)),
                           "r"(mapa_u32(smem_u32(mbarN), peer)) : "memory");
        }
        TCT(35)
        __syncthreads();                      // my own 8 partials
        tc::mbar_wait(mbarN, (uint32_t)(s & 1));   // the peer's 8 partials
        TCT(36)
        float tot = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) tot += ssq2[i];
        const float coef = fminf(1.f, (float)a.hy.max_grad_norm / (sqrtf(tot) + 1e-6f));
        const float step_size = (float)sh_d[0], ibc2 = (float)sh_d[1];
#pragma unroll
        for (int u = 0; u < NS; ++u) {
            const int i4 = tid + u * TC_THREADS;
            if (i4 < n4) {
                float4 p4 = reinterpret_cast<const float4 *>(PM)[i4];
#define TC_ADAM(cc)                                                                     \
                {                                                                       \
                    const float gq = g4[u].cc * coef;                                   \
                    m4[u].cc = fmaf(gq - m4[u].cc, omb1, m4[u].cc);                     \
                    v4[u].cc = fmaf(omb2 * gq, gq, v4[u].cc * b2f);                     \
                    const float denom = fmaf(fast_sqrt(v4[u].cc), ibc2, aeps);          \
                    p4.cc -= step_size * __fdividef(m4[u].cc, denom);                   \
                }
                TC_ADAM(x) TC_ADAM(y) TC_ADAM(z) TC_ADAM(w)
#undef TC_ADAM
                reinterpret_cast<float4 *>(PM)[i4] = p4;
                __stcg(reinterpret_cast<float4 *>(wM) + i4, m4[u]);
                __stcg(reinterpret_cast<float4 *>(wV) + i4, v4[u]);
                const int e0 = 4 * i4;
                if (e0 >= oW2 && e0 < ob2) {           // W2[j][k0..k0+3]: four consecutive halfwords of each image
                    const int j = (e0 - oW2) >> 6, k0 = (e0 - oW2) & 63;
                    const float w0 = p4.x * TC_SW, w1 = p4.y * TC_SW, w2 = p4.z * TC_SW, w3 = p4.w * TC_SW;
                    const float h0 = round11(w0), h1 = round11(w1), h2 = round11(w2), h3 = round11(w3);
                    const int hw = sw128_hw(j, k0);
                    *reinterpret_cast<uint2 *>(W2a + hw) = make_uint2(pack_h2_ovf(h0, h1), pack_h2_ovf(h2, h3));
                    *reinterpret_cast<uint2 *>(W2b + hw) = make_uint2(pack_h2_ovf(w0 - h0, w1 - h1), pack_h2_ovf(w2 - h2, w3 - h3));
                } else {
                    put_param(e0, p4.x);
                    if (e0 + 1 < nH) put_param(e0 + 1, p4.y);
                    if (e0 + 2 < nH) put_param(e0 + 2, p4.z);
                    if (e0 + 3 < nH) put_param(e0 + 3, p4.w);
                }
            }
        }
        TCT(37)
        tc::tmem_st_wait();
        tc::fence_async_smem();
        tc::tc_fence_before();
        __syncthreads();
        tc::tc_fence_after();
        TCT(38)
    }   // steps

    // ---------------- write back ----------------
    if (!a.grad_only && rs == 0) {
        for (int e = tid; e < nH; e += TC_THREADS) {
            const size_t gi = (size_t)task * L.n_par + L.to_global(half, e);
            a.params[gi] = PM[e];
            a.adam_m[gi] = __ldcg(wM + e); a.adam_v[gi] = __ldcg(wV + e);
        }
    }
    {   // losses: the critic CTA reports the value loss, the actor CTA the action loss and the entropy
        const float la = block_sum(loss_act, red), lv = block_sum(loss_val, red), le = block_sum(loss_ent, red);
        if (tid == 0) {                   // per-CTA sums (each CTA saw its own rows) -> combined by the rs == 0 CTA of the half
            a.lpart[(task * 16 + rank) * 4 + 0] = lv;
            a.lpart[(task * 16 + rank) * 4 + 1] = la;
            a.lpart[(task * 16 + rank) * 4 + 2] = le;
            __threadfence();
        }
    }
    tc::tc_fence_before();
    sync_group<2>();                 // no DSMEM traffic may target an exited CTA; loss partials are published
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
