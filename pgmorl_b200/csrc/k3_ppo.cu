// K3 -- PPO update for the whole population shard in ONE launch.
//
// Replaces PPO.update's minibatch loop (a2c/algo/ppo.py:62-107): evaluate_actions,
// clipped surrogate, clipped (use_clipped_value_loss) or plain vector value loss, autograd
// backward, clip_grad_norm_ and Adam.step, plus the sampler of a2c/storage.py:118-154
// (consumes the host permutation).
//
// Parallel decomposition. A task is a chain of E*B dependent optimiser steps, so the only
// parallelism inside a step is over the minibatch rows and over the two independent networks
// (actor / critic share nothing but the global gradient norm). One thread-block CLUSTER of C
// CTAs owns one task for the whole chain:
//     C == 1 : one CTA runs both halves, all mb rows                     (large populations)
//     C >= 2 : CTAs [0, C/2) = actor, [C/2, C) = critic; each of the G = C/2 CTAs of a half
//              runs mb/G rows                                            (small populations)
// Per step every CTA: gathers its rows' packed records (cp.async, double buffered), runs
// forward + hand-derived backward on 16*TM-row chunks with weights resident in shared memory,
// and takes part in an all-reduce of the half's gradient: reduce-scatter to the G slice owners
// (fixed summation order -> deterministic), norm exchange over all C CTAs, clip + Adam on the
// slice, all-gather of the new parameters. The generic kernel in this file does it through
// L2 scratch slots and three cluster barriers per step (any dims, incl. C == 1); the fast
// kernel for small networks (k3_fast.cuh) keeps everything in (distributed) shared memory and
// runs the exchange as barrier-free dataflow (bulk copies + st.async into mbarriers, TMA
// multicast for the parameters).
//
// FP32 FFMA throughout; Adam bias corrections in double.
#include <cooperative_groups.h>
#include <stdlib.h>

#include "k3_body.cuh"

namespace pgm {

__global__ void k3_pack_kernel(const float *__restrict__ obs, size_t obs_ts, const float *__restrict__ action,
                               const float *__restrict__ logp, const float *__restrict__ vold, size_t v_ts,
                               const float *__restrict__ ret, const float *__restrict__ adv, float *__restrict__ rec,
                               int P, int S, NetLayout L, int RSG) {
    const size_t total = (size_t)P * S * RSG;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int f = (int)(i % RSG);
        const size_t ts = i / RSG;
        const int s = (int)(ts % S);
        const int task = (int)(ts / S);
        const int O = L.O, OP = L.OP, A = L.AC, M = L.M;   // A: action columns
        float v = 0.f;
        if (f < O) v = obs[task * obs_ts + (size_t)s * O + f];
        else if (f < OP) v = 0.f;
        else if (f < OP + A) v = action[((size_t)task * S + s) * A + (f - OP)];
        else if (f == OP + A) v = logp[(size_t)task * S + s];
        else if (f < OP + A + 1 + M) v = vold[task * v_ts + (size_t)s * M + (f - OP - A - 1)];
        else if (f < OP + A + 1 + 2 * M) v = ret[((size_t)task * S + s) * M + (f - OP - A - 1 - M)];
        else if (f == OP + A + 1 + 2 * M) v = adv[(size_t)task * S + s];
        rec[i] = v;
    }
}

template <int C, int TM, int KG1, int NA, bool DB, bool VU = false>
__global__ void __launch_bounds__(NTHREADS, 1) k3_ppo_kernel(const K3Args a) { k3_ppo_body<C, TM, KG1, NA, DB, VU, H>(a); }

template <int HW, int C, int TM, int KG1, int NA, bool DB, bool VU>
__global__ void __launch_bounds__(NTHREADS, 1) k3_ppo_h_kernel(const K3Args a) { k3_ppo_body<C, TM, KG1, NA, DB, VU, HW>(a); }

}  // namespace pgm
#include "k3_fast.cuh"
#include "k3_tc.cuh"
#include "k3_tcw.cuh"
namespace pgm {

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct K3Plan {
    int C, G, TM, KG1, NA, RC, Rg, RSG, RSS, NHP;
    bool DB, fast, tc, tcw;
    bool vu;      // unclipped value loss (PGM_PPO_VALUE_UNCLIPPED): the VU = true instantiation of the chosen kernel
    int hidden;   // hidden width: 64, or 32 / 128 (generic kernel k3_ppo_h_kernel only)
    bool cat;     // Categorical head: the generic kernel k3_ppo_cat_kernel (k3_cat.cu) at every width
    int tail;     // fast path step tail (k3_fast.cuh): 0 three cluster barriers, 1 redundant Adam, 2 TMA multicast broadcast
    int rs;
    int stage_floats;
    size_t smem;
    size_t off_rec, off_gpart, off_ssq, off_lpart, off_trace, off_mv, total;
    size_t off_xp, off_scr, off_w1img, off_pmv;      // wide tensor-core path (k3_tcw.cuh)
};

static size_t k3_smem_bytes(const NetLayout &L, int C, int TM, bool DB, int RSS, int hw = H) {
    const int RC = 16 * TM;
    const int ldo = ((L.A > L.M ? L.A : L.M) | 1);
    const size_t i0 = halfnet_smem_floats(L, 0, hw), i1 = halfnet_smem_floats(L, 1, hw);
    size_t f = 0;
    if (C == 1) f += i0 + i1;
    else f += i0 > i1 ? i0 : i1;
    f += 3 * (size_t)RC * (hw + 4) + 2 * (size_t)round_up(RC * ldo, 4);
    f += (size_t)(DB ? 2 : 1) * RC * RSS;
    return f * sizeof(float);
}

// shapes the tensor-core kernel is instantiated for (Walker2d / HalfCheetah and Hopper-v3, SURVEY section 8)
static bool k3_tc_dims(int O, int A, int M) { return (O == 17 && A == 6 && M == 2) || (O == 11 && A == 3 && M == 3); }
static size_t k3_tc_mv_bytes(int P) { return (size_t)P * 2 * 2 * 2 * TC_NHP * sizeof(float); }   // [P][half][rs <= 2][m|v]
constexpr int K3_CLUSTER_TC = 32;   // `cluster` values that select the tensor-core path explicitly: 32 = 2 CTAs per task,
constexpr int K3_CLUSTER_TC2 = 64;  // 64 = 4 CTAs per task (row tiles split over two CTAs per network half)
constexpr int K3_CLUSTER_TC4 = 128; // 128 = 8 CTAs per task (wide-observation kernel only)
// shape the wide-observation tensor-core kernel (k3_tcw.cuh) is instantiated for: Humanoid (SURVEY section 8)
static bool k3_tcw_dims(int O, int A, int M) { return O == 376 && A == 17 && M == 2; }
static size_t k3_tcw_bytes(int P, int S, int O, int A, size_t *oxp, size_t *oscr, size_t *ow1, size_t *opmv) {
    size_t off = 0;
    auto seg = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t a0 = seg((size_t)P * S * TW_XROW_HW * sizeof(__half));
    const size_t a1 = seg((size_t)P * S * TW_SCF * sizeof(float));
    const size_t a2 = seg((size_t)P * 2 * TW_NB * 8192 * sizeof(__half));
    const size_t a3 = seg((size_t)P * 2 * 3 * tw_nhp(O, A) * sizeof(float));
    if (oxp) { *oxp = a0; *oscr = a1; *ow1 = a2; *opmv = a3; }
    return off;
}

// Clusters of 2*rs CTAs of the wide kernel that the device keeps resident at once (a cluster has to fit one GPC, so this
// is less than SMs / cluster size); -1 when it cannot be queried (no device: workspace sizing on a build machine).
static int k3_tcw_resident_clusters(int rs) {
    static int cache[5] = {-2, -2, -2, -2, -2};
    if (cache[rs] != -2) return cache[rs];
    const void *kern = rs == 4 ? (const void *)k3_tcw_kernel<376, 17, 2, 4>
                               : (rs == 2 ? (const void *)k3_tcw_kernel<376, 17, 2, 2> : (const void *)k3_tcw_kernel<376, 17, 2, 1>);
    const size_t smem = tw_smem_layout().total;
    int n = -1;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2 * rs * 64); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2 * rs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) n = -1;
    }
    if (n < 0) (void)cudaGetLastError();
    return cache[rs] = n;
}

// Step tails of the FFMA cluster kernel (k3_fast.cuh, template parameter TAIL); every variant performs the same arithmetic
// in the same order, so results are bit-identical (tests/test_gpu_kernels.py::test_k3_step_tails_bit_identical). Same-box
// A/B at the headline configuration (6 tasks x 16 CTAs, profiles/r02/README.md), ms per MOPG iteration:
//   tail 0  3.876  three cluster barriers: partial images pulled through ld.shared::cluster, parameters pushed (round 1)
//   tail 1  4.04   two barriers: register tiles pushed to the slice owner, whole-half Adam in every CTA
//   tail 2  3.734  parameter broadcast by TMA bulk copy with cluster multicast, third barrier gone
//   tail 3  3.839  tail 2 + gradient exchange through L2 scratch slots
//   tail 4  3.712  tail 2 + gradient reduce-scatter pushed by cp.async.bulk shared::cta -> shared::cluster, first barrier gone
//   tail 5  3.575  tail 4 + norm partials by st.async with mbarrier completion: no cluster barrier left in the step (default)
//   tail 6  3.557* tail 5 + the W2-only gradient slices pushed right after the {dW2, dz1} phase (*same box: tail 5 3.525;
//                  the mid-phase proxy fence costs more than the early transfer saves)
// A tail can be forced per call by OR-ing a flag into `cluster` (tests, A/B) or per process with PGM_K3_TAIL=0..5.
constexpr int K3_DEFAULT_TAIL = 5;
constexpr int K3_CLUSTER_TAIL2 = 0x100;    // tail 1
constexpr int K3_CLUSTER_TAILMC = 0x200;   // tail 2
constexpr int K3_CLUSTER_TAILGL = 0x400;   // tail 3
constexpr int K3_CLUSTER_TAIL0 = 0x800;    // tail 0
constexpr int K3_CLUSTER_TAILBP = 0x1000;  // tail 4
constexpr int K3_CLUSTER_TAILNB = 0x2000;  // tail 5
constexpr int K3_CLUSTER_TAILEP = 0x4000;  // tail 6
constexpr int K3_CLUSTER_FLAGS = K3_CLUSTER_TAIL2 | K3_CLUSTER_TAILMC | K3_CLUSTER_TAILGL | K3_CLUSTER_TAIL0 | K3_CLUSTER_TAILBP |
                                 K3_CLUSTER_TAILNB | K3_CLUSTER_TAILEP | PGM_PPO_VALUE_UNCLIPPED;

static int k3_plan(K3Plan &pl, int P, int S, int mb, int O, int A, int M, int cluster, int sms, int hidden, int dist) {
    NetLayout L(O, A, M, hidden, dist);
    const bool cat = dist == PGM_DIST_CATEGORICAL;
    const bool tail2 = (cluster & K3_CLUSTER_TAIL2) != 0, tailmc = (cluster & K3_CLUSTER_TAILMC) != 0;
    const bool tailgl = (cluster & K3_CLUSTER_TAILGL) != 0, tail0 = (cluster & K3_CLUSTER_TAIL0) != 0;
    const bool tailbp = (cluster & K3_CLUSTER_TAILBP) != 0, tailnb = (cluster & K3_CLUSTER_TAILNB) != 0;
    const bool tailep = (cluster & K3_CLUSTER_TAILEP) != 0;
    pl.vu = (cluster & PGM_PPO_VALUE_UNCLIPPED) != 0;
    cluster &= ~K3_CLUSTER_FLAGS;
    pl.tc = false; pl.tcw = false; pl.tail = 0; pl.off_mv = 0; pl.hidden = hidden; pl.cat = cat;
    // Categorical heads run on the generic cluster kernel only, at every hidden width
    if (cat) {
        PGM_REQUIRE(A >= 1 && A <= CAT_MAX, "ppo: a categorical head has 1..%d categories, got %d", CAT_MAX, A);
        PGM_REQUIRE(cluster != K3_CLUSTER_TC && cluster != K3_CLUSTER_TC2 && cluster != K3_CLUSTER_TC4,
                    "ppo: the tensor-core paths (cluster 32, 64, 128) are built for Gaussian heads, got a categorical head");
        PGM_REQUIRE(cluster != 1, "ppo: cluster 1 (both halves in one CTA) is built for Gaussian heads, got a categorical "
                    "head (use cluster 0, 2, 4, 8 or 16)");
    }
    // the tensor-core kernels, the fast cluster kernel and cluster = 1 are built for hidden width 64; other widths run on
    // the generic cluster kernel at 2..16 CTAs per task
    if (hidden != H) {
        PGM_REQUIRE(cluster != K3_CLUSTER_TC && cluster != K3_CLUSTER_TC2 && cluster != K3_CLUSTER_TC4,
                    "ppo: the tensor-core paths (cluster 32, 64, 128) are built for hidden width 64, got hidden width %d", hidden);
        PGM_REQUIRE(cluster != 1, "ppo: cluster 1 (both halves in one CTA) is built for hidden width 64, got hidden width %d "
                    "(use cluster 0, 2, 4, 8 or 16)", hidden);
    }
    // wide observations (Humanoid): the streamed tensor-core kernel; row split over as many CTAs per half as fill the SMs
    if (hidden == H && !cat && k3_tcw_dims(O, A, M) && (cluster == 0 || cluster == K3_CLUSTER_TC || cluster == K3_CLUSTER_TC2 || cluster == K3_CLUSTER_TC4)) {
        const int tiles = (mb + 127) / 128;
        if (cluster == 0) {
            // most CTAs per task whose clusters are all resident at once (a second wave of clusters doubles the step)
            auto fits = [&](int rs) {
                const int res = k3_tcw_resident_clusters(rs);
                return tiles >= rs && 2 * rs * P <= sms && (res < 0 || P <= res);
            };
            pl.rs = fits(4) ? 4 : (fits(2) ? 2 : 1);
        }
        else pl.rs = cluster == K3_CLUSTER_TC4 ? 4 : (cluster == K3_CLUSTER_TC2 ? 2 : 1);
        pl.tc = true; pl.tcw = true; pl.C = 2 * pl.rs; pl.G = 1; pl.TM = 0; pl.KG1 = 0; pl.NA = 0; pl.RC = 128; pl.Rg = 0;
        pl.RSG = 0; pl.RSS = 0; pl.NHP = 64; pl.DB = false; pl.fast = false; pl.stage_floats = 0;
        pl.smem = tw_smem_layout().total;
        size_t off = 0;
        auto seg = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
        pl.off_rec = 0;
        pl.off_gpart = seg((size_t)P * 2 * pl.G * pl.NHP * sizeof(float));
        pl.off_ssq = seg((size_t)P * 16 * sizeof(float));
        pl.off_lpart = seg((size_t)P * 16 * 4 * sizeof(float));
#ifdef PGM_K3_TRACE
        pl.off_trace = seg((size_t)P * 8 * 2 * 48 * sizeof(long long));
#else
        pl.off_trace = 0;
#endif
        const size_t base = off;
        off += k3_tcw_bytes(P, S, O, A, &pl.off_xp, &pl.off_scr, &pl.off_w1img, &pl.off_pmv);
        pl.off_xp += base; pl.off_scr += base; pl.off_w1img += base; pl.off_pmv += base;
        pl.total = off;
        return PGM_OK;
    }
    // auto: the tensor-core path wins as soon as the FFMA path can no longer give every task a 16-CTA cluster (measured on
    // a B200, profiles/k3_sweep.py: 1.2x at P = 8, 2.4x at 16, 3.3x from 37 tasks on; below 8 tasks FFMA is 6 % faster)
    if (hidden == H && !cat && cluster == 0 && k3_tc_dims(O, A, M) && P >= 8) {
        // 4 CTAs per task (row tiles split over two CTAs per half) while they fit in one wave: 4-CTA clusters tile the 148
        // SMs less densely than pairs (measured: 32 clusters run in one wave, 37 need two)
        cluster = (mb > 128 && 4 * P <= sms - 20) ? K3_CLUSTER_TC2 : K3_CLUSTER_TC;
    }
    pl.rs = 1;
    if (cluster == K3_CLUSTER_TC || cluster == K3_CLUSTER_TC2) {
        pl.rs = cluster == K3_CLUSTER_TC2 ? 2 : 1;
        PGM_REQUIRE(k3_tc_dims(O, A, M), "ppo: the tensor-core path is built for (O,A,M) = (17,6,2) and (11,3,3), got (%d,%d,%d)", O, A, M);
        pl.tc = true; pl.C = 2 * pl.rs; pl.G = 1; pl.TM = 0; pl.KG1 = 0; pl.NA = 0; pl.RC = 128; pl.Rg = 0;
        pl.RSG = rec_stride(L); pl.RSS = 0; pl.NHP = 64; pl.DB = false; pl.fast = false; pl.stage_floats = 0;
        pl.smem = tc_smem_layout().total;
        size_t off = 0;
        auto seg = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
        pl.off_rec = seg((size_t)P * S * pl.RSG * sizeof(float));
        pl.off_gpart = seg((size_t)P * 2 * pl.G * pl.NHP * sizeof(float));
        pl.off_ssq = seg((size_t)P * 16 * sizeof(float));
        pl.off_lpart = seg((size_t)P * 16 * 4 * sizeof(float));
        pl.off_mv = seg(k3_tc_mv_bytes(P));
#ifdef PGM_K3_TRACE
        pl.off_trace = seg((size_t)P * 16 * 4 * 16 * 2 * sizeof(long long));
#else
        pl.off_trace = 0;
#endif
        pl.total = off;
        return PGM_OK;
    }
    PGM_REQUIRE(O >= 1 && O <= 384 && A >= 1 && A <= 32 && M >= 1 && M <= 16,
                "ppo: unsupported dims O=%d A=%d M=%d (O<=384, A<=32, M<=16)", O, A, M);
    PGM_REQUIRE(cluster == 0 || cluster == 1 || cluster == 2 || cluster == 4 || cluster == 8 || cluster == 16,
                "ppo: cluster must be 0 (auto), 1, 2, 4, 8, 16 (FP32 FFMA paths), 32, 64 (tensor-core paths) or 128 (wide tensor-core path) (got %d)", cluster);
    int C = cluster;
    if (C == 0) {   // fill the SMs: double the cluster while every task still gets its CTAs resident at once
        C = 2;      // one CTA per network half is the throughput configuration (large populations)
        // 16-CTA clusters are non-portable and at most one fits a GPC (ncu: launch__cluster_max_active = 7 with
        // this kernel's shared-memory footprint): use them only when every task's cluster is resident at once
        const int cmax = (P <= 7) ? 16 : 8;
        while (C < cmax && (long long)P * C * 2 <= sms && mb / C >= 32) C *= 2;
    }
    const bool big = (L.OP > 64) || (A > 16) || (M > 16);
    pl.C = C; pl.G = C == 1 ? 1 : C / 2;
    // dW1 k lanes: 16 (64 features per KG1 group) at hidden width 64 and 128, 32 (128 per group) at 32; head rows: 16 per
    // NA at 64 and 128, 32 at 32. At 128 the wide variant stops at KG1 = 2 (OP <= 128): its dW1 tile then stays in
    // registers next to the 64 dW2 accumulators (KG1 = 3 spills); at 32, KG1 = 3 covers Humanoid's 376 features
    if (hidden == H) { pl.KG1 = big ? 6 : 1; pl.NA = big ? 2 : 1; }
    else if (hidden == 128) { pl.KG1 = big ? 2 : 1; pl.NA = big ? 2 : 1; }
    else { pl.KG1 = big ? 3 : 1; pl.NA = 1; }
    const int rows = (mb + pl.G - 1) / pl.G;          // rows per CTA per step
    pl.TM = big ? 2 : (rows <= 32 ? 2 : 4);
    pl.RC = 16 * pl.TM;
    pl.Rg = round_up(rows, pl.RC);
    pl.RSG = rec_stride(L);
    pl.RSS = stride4odd(pl.RSG);
    {
        const int i0 = halfnet_smem_floats(L, 0, hidden), i1 = halfnet_smem_floats(L, 1, hidden);
        pl.NHP = round_up(i0 > i1 ? i0 : i1, 64);   // covers both the reference-order half and its padded image
    }
    pl.DB = (C > 1) && !big;
    pl.fast = hidden == H && !cat && (C > 1) && !big && L.OP <= 48 && pl.RC * (pl.RSG / 4) <= 4 * NTHREADS;
    pl.stage_floats = 0;
    if (pl.fast) {
        const int s0 = k3_fast_stage_floats(L.OP, A), s1 = k3_fast_stage_floats(L.OP, M);
        pl.stage_floats = s0 > s1 ? s0 : s1;
        // step tail: default from K3_DEFAULT_TAIL; others on request (cluster flags, or PGM_K3_TAIL=0|1|2 in the
        // environment for whole-program A/B runs)
        static const int env_tail = [] { const char *e = getenv("PGM_K3_TAIL"); return (e && e[0] >= '0' && e[0] <= '6') ? e[0] - '0' : -1; }();
        const int want = tail0 ? 0 : (tail2 ? 1 : (tailmc ? 2 : (tailgl ? 3 : (tailbp ? 4 : (tailnb ? 5 : (tailep ? 6 : (env_tail >= 0 ? env_tail : K3_DEFAULT_TAIL)))))));
        // one CTA per half (C = 2) keeps a whole half resident: with TM = 4 that exceeds 227 KB at wider shapes (Ant,
        // (27,8,2): 237 664 B). Fall back to TM = 2, then to the generic double-buffered kernel below.
        for (;;) {
            pl.tail = want;
            if (pl.tail == 1 && !(pl.G >= 2 && k3_fast_smem_bytes(L, pl.TM, pl.RSS, pl.NHP, pl.stage_floats, pl.G, true) <= 227 * 1024))
                pl.tail = 0;
            if (pl.tail >= 2 && pl.G < 2) pl.tail = 0;
            if (pl.tail >= 4 && k3_fast_smem_bytes(L, pl.TM, pl.RSS, pl.NHP, pl.stage_floats, pl.G, false, false, true) > 227 * 1024)
                pl.tail = 2;
            pl.smem = k3_fast_smem_bytes(L, pl.TM, pl.RSS, pl.NHP, pl.stage_floats, pl.G, pl.tail == 1, pl.tail == 3, pl.tail >= 4);
            if (pl.smem <= 227 * 1024 || pl.TM == 2) break;
            pl.TM = 2; pl.RC = 32; pl.Rg = round_up(rows, pl.RC);
        }
        if (pl.smem > 227 * 1024) { pl.fast = false; pl.stage_floats = 0; pl.tail = 0; }
    }
    if (!pl.fast) pl.smem = k3_smem_bytes(L, C, pl.TM, pl.DB, pl.RSS, hidden);
    PGM_REQUIRE(pl.smem <= 227 * 1024, "ppo: configuration needs %zu B of shared memory (O=%d, cluster=%d, hidden width %d)",
                pl.smem, O, C, hidden);
    PGM_REQUIRE(L.OP <= (hidden == 32 ? 128 : 64) * pl.KG1, "ppo: obs dim %d exceeds the dW1 tile at hidden width %d", O, hidden);
    size_t off = 0;
    auto seg = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    pl.off_rec = seg((size_t)P * S * pl.RSG * sizeof(float));
    pl.off_gpart = seg((size_t)P * 2 * (pl.G + 1) * pl.NHP * sizeof(float));      // + one staging row per half (pstage)
    pl.off_ssq = seg((size_t)P * 16 * sizeof(float));
    pl.off_lpart = seg((size_t)P * 16 * 4 * sizeof(float));
#ifdef PGM_K3_TRACE
    pl.off_trace = seg((size_t)P * 16 * 4 * 16 * 2 * sizeof(long long));
#else
    pl.off_trace = 0;
#endif
    pl.total = off;
    return PGM_OK;
}

template <typename Kern>
static int k3_launch_k(Kern kern, int C, const K3Args &a, const K3Plan &pl, int P, cudaStream_t st) {
    PGM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    if (C > 8) PGM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(P * C); cfg.blockDim = dim3(pl.tc ? TC_THREADS : NTHREADS); cfg.dynamicSmemBytes = pl.smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = C > 1 ? 1 : 0;
    PGM_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
    return PGM_OK;
}

template <int C, bool VU>
static int k3_launch_c(const K3Args &a, const K3Plan &pl, int P, cudaStream_t st) {
    if constexpr (C > 1) {
        if (pl.fast) {
            if (pl.tail == 1)
                return pl.TM == 2 ? k3_launch_k(k3_ppo_fast_kernel<C, 2, 1, VU>, C, a, pl, P, st)
                                  : k3_launch_k(k3_ppo_fast_kernel<C, 4, 1, VU>, C, a, pl, P, st);
            if (pl.tail == 2)
                return pl.TM == 2 ? k3_launch_k(k3_ppo_fast_kernel<C, 2, 2, VU>, C, a, pl, P, st)
                                  : k3_launch_k(k3_ppo_fast_kernel<C, 4, 2, VU>, C, a, pl, P, st);
            if (pl.tail == 3)
                return pl.TM == 2 ? k3_launch_k(k3_ppo_fast_kernel<C, 2, 3, VU>, C, a, pl, P, st)
                                  : k3_launch_k(k3_ppo_fast_kernel<C, 4, 3, VU>, C, a, pl, P, st);
            if (pl.tail == 4)
                return pl.TM == 2 ? k3_launch_k(k3_ppo_fast_kernel<C, 2, 4, VU>, C, a, pl, P, st)
                                  : k3_launch_k(k3_ppo_fast_kernel<C, 4, 4, VU>, C, a, pl, P, st);
            if (pl.tail == 5)
                return pl.TM == 2 ? k3_launch_k(k3_ppo_fast_kernel<C, 2, 5, VU>, C, a, pl, P, st)
                                  : k3_launch_k(k3_ppo_fast_kernel<C, 4, 5, VU>, C, a, pl, P, st);
            if (pl.tail == 6)
                return pl.TM == 2 ? k3_launch_k(k3_ppo_fast_kernel<C, 2, 6, VU>, C, a, pl, P, st)
                                  : k3_launch_k(k3_ppo_fast_kernel<C, 4, 6, VU>, C, a, pl, P, st);

            return pl.TM == 2 ? k3_launch_k(k3_ppo_fast_kernel<C, 2, 0, VU>, C, a, pl, P, st)
                              : k3_launch_k(k3_ppo_fast_kernel<C, 4, 0, VU>, C, a, pl, P, st);
        }
        if (pl.KG1 == 6) return k3_launch_k(k3_ppo_kernel<C, 2, 6, 2, false, VU>, C, a, pl, P, st);
        return pl.TM == 2 ? k3_launch_k(k3_ppo_kernel<C, 2, 1, 1, true, VU>, C, a, pl, P, st)
                          : k3_launch_k(k3_ppo_kernel<C, 4, 1, 1, true, VU>, C, a, pl, P, st);
    } else {
        if (pl.KG1 == 6) return k3_launch_k(k3_ppo_kernel<1, 2, 6, 2, false, VU>, 1, a, pl, P, st);
        return pl.TM == 2 ? k3_launch_k(k3_ppo_kernel<1, 2, 1, 1, false, VU>, 1, a, pl, P, st)
                          : k3_launch_k(k3_ppo_kernel<1, 4, 1, 1, false, VU>, 1, a, pl, P, st);
    }
}

// hidden width 32 / 128: the generic kernel at 2..16 CTAs per task
template <int HW, int C, bool VU>
static int k3_launch_hc(const K3Args &a, const K3Plan &pl, int P, cudaStream_t st) {
    constexpr int KGB = HW == 128 ? 2 : 3, NAB = HW == 128 ? 2 : 1;   // the wide ("big") instantiation, k3_plan
    if (pl.KG1 > 1) return k3_launch_k(k3_ppo_h_kernel<HW, C, 2, KGB, NAB, false, VU>, C, a, pl, P, st);
    return pl.TM == 2 ? k3_launch_k(k3_ppo_h_kernel<HW, C, 2, 1, 1, true, VU>, C, a, pl, P, st)
                      : k3_launch_k(k3_ppo_h_kernel<HW, C, 4, 1, 1, true, VU>, C, a, pl, P, st);
}

template <int HW, bool VU>
static int k3_launch_h(const K3Args &a, const K3Plan &pl, int P, cudaStream_t st) {
    switch (pl.C) {
        case 2: return k3_launch_hc<HW, 2, VU>(a, pl, P, st);
        case 4: return k3_launch_hc<HW, 4, VU>(a, pl, P, st);
        case 8: return k3_launch_hc<HW, 8, VU>(a, pl, P, st);
        case 16: return k3_launch_hc<HW, 16, VU>(a, pl, P, st);
    }
    set_error("ppo: bad cluster %d at hidden width %d", pl.C, HW);
    return PGM_ERR_ARG;
}

template <typename Kern>
static int k3_launch_w(Kern kern, const K3Args &a, const TwExtra &x, const K3Plan &pl, int P, cudaStream_t st) {
    PGM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(P * pl.C); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = pl.smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = pl.C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    PGM_CUDA(cudaLaunchKernelEx(&cfg, kern, a, x));
    return PGM_OK;
}

template <bool VU>
static int k3_launch(const K3Args &a, const K3Plan &pl, int P, cudaStream_t st) {
    if (pl.cat) return k3_launch_cat(a, pl.hidden, pl.C, pl.TM, pl.KG1 > 1, VU, pl.smem, P, st);
    if (pl.hidden == 32) return k3_launch_h<32, VU>(a, pl, P, st);
    if (pl.hidden == 128) return k3_launch_h<128, VU>(a, pl, P, st);
    if (pl.tc) {
        if (a.L.O == 17) return pl.rs == 2 ? k3_launch_k(k3_tc_kernel<17, 6, 2, 2, VU>, pl.C, a, pl, P, st)
                                           : k3_launch_k(k3_tc_kernel<17, 6, 2, 1, VU>, pl.C, a, pl, P, st);
        return pl.rs == 2 ? k3_launch_k(k3_tc_kernel<11, 3, 3, 2, VU>, pl.C, a, pl, P, st)
                          : k3_launch_k(k3_tc_kernel<11, 3, 3, 1, VU>, pl.C, a, pl, P, st);
    }
    switch (pl.C) {
        case 1: return k3_launch_c<1, VU>(a, pl, P, st);
        case 2: return k3_launch_c<2, VU>(a, pl, P, st);
        case 4: return k3_launch_c<4, VU>(a, pl, P, st);
        case 8: return k3_launch_c<8, VU>(a, pl, P, st);
        case 16: return k3_launch_c<16, VU>(a, pl, P, st);
    }
    set_error("ppo: bad cluster %d", pl.C);
    return PGM_ERR_ARG;
}

template <bool VU>
static int k3_launch_tcw(const K3Args &a, const TwExtra &x, const K3Plan &pl, int P, cudaStream_t st) {
    if (pl.rs == 4) return k3_launch_w(k3_tcw_kernel<376, 17, 2, 4, VU>, a, x, pl, P, st);
    if (pl.rs == 2) return k3_launch_w(k3_tcw_kernel<376, 17, 2, 2, VU>, a, x, pl, P, st);
    return k3_launch_w(k3_tcw_kernel<376, 17, 2, 1, VU>, a, x, pl, P, st);
}

static int sm_count(int &sms) {
    int dev = 0;
    PGM_CUDA(cudaGetDevice(&dev));
    PGM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    return PGM_OK;
}

}  // namespace pgm

using namespace pgm;

#ifdef PGM_K3_TRACE
static size_t g_last_trace_offset = 0;
// instrumented builds only (libpgmorl_b200_trace.so): byte offset of the clock marks inside the workspace of the last launch
extern "C" size_t pgm_ppo_last_trace_offset() { return g_last_trace_offset; }
#endif

extern "C" size_t pgm_ppo_workspace_bytes_x(int P, int S, int O, int A, int M, int cluster, int hidden, int dist) {
    // upper bound over every plan the launcher may choose for these dims (cluster 0 = auto)
    if (!hidden_supported(hidden) || !dist_supported(dist)) return 0;
    const bool cat = dist == PGM_DIST_CATEGORICAL;
    NetLayout L(O, A, M, hidden, dist);
    cluster &= ~K3_CLUSTER_FLAGS;
    const int G = cluster == 0 ? 8 : (cluster == 1 ? 1 : cluster / 2);
    const int i0 = halfnet_smem_floats(L, 0, hidden), i1 = halfnet_smem_floats(L, 1, hidden);
    const int NHP = round_up(i0 > i1 ? i0 : i1, 64);
    size_t t = 0;
    auto seg = [&](size_t b) { t += (b + 255) / 256 * 256; };
    seg((size_t)P * S * rec_stride(L) * sizeof(float));
    seg((size_t)P * 2 * (G + 1) * NHP * sizeof(float));
    seg((size_t)P * 16 * sizeof(float));
    seg((size_t)P * 64 * sizeof(float));
    if (hidden == H && !cat && k3_tc_dims(O, A, M)) seg(k3_tc_mv_bytes(P));
    if (hidden == H && !cat && k3_tcw_dims(O, A, M)) seg(k3_tcw_bytes(P, S, O, A, nullptr, nullptr, nullptr, nullptr) + 1024);
#ifdef PGM_K3_TRACE
    seg((size_t)P * 16 * 4 * 16 * 2 * sizeof(long long));
#endif
    return t;
}

extern "C" size_t pgm_ppo_workspace_bytes_h(int P, int S, int O, int A, int M, int cluster, int hidden) {
    return pgm_ppo_workspace_bytes_x(P, S, O, A, M, cluster, hidden, PGM_DIST_GAUSSIAN);
}

extern "C" size_t pgm_ppo_workspace_bytes(int P, int S, int O, int A, int M, int cluster) {
    return pgm_ppo_workspace_bytes_h(P, S, O, A, M, cluster, H);
}

static int ppo_common(float *params, float *adam_m, float *adam_v, int32_t *adam_step, const double *lr,
                      const float *obs, size_t obs_ts, const float *action, const float *logp_old,
                      const float *value_old, size_t v_ts, const float *returns, const float *adv,
                      const int32_t *perm, int perm_shared, int E, int B, int mb, const pgm_ppo_hyper *hy,
                      float *losses, float *grad_out, void *workspace, size_t wbytes, int cluster, int P, int S,
                      int O, int A, int M, int hidden, int dist, cudaStream_t st) {
    PGM_REQUIRE(params && obs && action && logp_old && value_old && returns && adv && perm && hy && losses && workspace,
                "ppo: null pointer argument");
    PGM_REQUIRE(hidden_supported(hidden), "ppo: hidden width %d is not one of {32, 64, 128}", hidden);
    PGM_REQUIRE(dist_supported(dist), "ppo: unknown action head %d", dist);
    PGM_REQUIRE(P > 0 && S > 0 && mb > 0 && mb <= S, "ppo: bad sizes P=%d S=%d mb=%d", P, S, mb);
    PGM_REQUIRE(((uintptr_t)workspace & 255) == 0, "ppo: workspace must be 256-byte aligned");
    int sms = 148;
    if (int rc = sm_count(sms)) return rc;
    K3Plan pl;
    if (int rc = k3_plan(pl, P, S, mb, O, A, M, cluster, sms, hidden, dist)) return rc;
    if (pl.total > wbytes) {
        set_error("ppo: workspace too small: need %zu bytes, got %zu", pl.total, wbytes);
        return PGM_ERR_WORKSPACE;
    }
    char *ws = (char *)workspace;
    K3Args a;
    a.params = params; a.adam_m = adam_m; a.adam_v = adam_v; a.adam_step = adam_step; a.lr = lr;
    a.rec = (const float *)(ws + pl.off_rec); a.perm = perm; a.losses = losses;
    a.gpart = (float *)(ws + pl.off_gpart); a.pstage = a.gpart + (size_t)P * 2 * pl.G * pl.NHP; a.ssq = (float *)(ws + pl.off_ssq); a.lpart = (float *)(ws + pl.off_lpart);
#ifdef PGM_K3_TRACE
    a.trace = (long long *)(ws + pl.off_trace);
    g_last_trace_offset = pl.off_trace;
#else
    a.trace = nullptr;
#endif
    a.mv = (float *)(ws + pl.off_mv);
    a.grad_out = grad_out; a.perm_shared = perm_shared; a.E = E; a.B = B; a.mb = mb; a.S = S;
    a.grad_only = grad_out != nullptr; a.nsteps = a.grad_only ? 1 : E * B;
    a.Rg = pl.Rg; a.RSG = pl.RSG; a.RSS = pl.RSS; a.NHP = pl.NHP; a.stage_floats = pl.stage_floats; a.rs = pl.rs; a.hy = *hy; a.L = NetLayout(O, A, M, hidden, dist);
    if (pl.tcw) {
        TwExtra x;
        x.xp = (const __half *)(ws + pl.off_xp); x.scr = (const float *)(ws + pl.off_scr);
        x.w1img = (__half *)(ws + pl.off_w1img); x.pmv = (float *)(ws + pl.off_pmv);
        const size_t total = (size_t)P * S * (TW_NB * 64 + TW_SCF);
        int blocks = (int)((total + 255) / 256);
        if (blocks > sms * 16) blocks = sms * 16;
        k3w_pack_kernel<376, 17, 2><<<blocks, 256, 0, st>>>(obs, obs_ts, action, logp_old, value_old, v_ts, returns, adv,
                                                            (__half *)(ws + pl.off_xp), (float *)(ws + pl.off_scr), P, S);
        PGM_CUDA(cudaGetLastError());
        // features O+1 .. 383 of the last W1 block image are never written by the kernel: they must be zero, not stale bytes
        PGM_CUDA(cudaMemsetAsync(ws + pl.off_w1img, 0, (size_t)P * 2 * TW_NB * 8192 * sizeof(__half), st));
        return pl.vu ? k3_launch_tcw<true>(a, x, pl, P, st) : k3_launch_tcw<false>(a, x, pl, P, st);
    }
    {
        const size_t total = (size_t)P * S * pl.RSG;
        int blocks = (int)((total + 255) / 256);
        if (blocks > sms * 16) blocks = sms * 16;
        k3_pack_kernel<<<blocks, 256, 0, st>>>(obs, obs_ts, action, logp_old, value_old, v_ts, returns, adv,
                                               (float *)(ws + pl.off_rec), P, S, a.L, pl.RSG);
        PGM_CUDA(cudaGetLastError());
    }
    // padding entries of the gradient slots are never written by the kernel: keep them zero
    PGM_CUDA(cudaMemsetAsync(ws + pl.off_gpart, 0, (size_t)P * 2 * (pl.G + 1) * pl.NHP * sizeof(float), st));
    return pl.vu ? k3_launch<true>(a, pl, P, st) : k3_launch<false>(a, pl, P, st);
}

extern "C" int pgm_ppo_update_x_f32(float *params, float *adam_m, float *adam_v, int32_t *adam_step, const double *lr,
                                    const float *obs, size_t obs_task_stride, const float *action,
                                    const float *logp_old, const float *value_old, size_t value_task_stride,
                                    const float *returns, const float *adv, const int32_t *perm, int perm_shared,
                                    int E, int B, const pgm_ppo_hyper *hyper_host, float *losses, void *workspace,
                                    size_t workspace_bytes, int cluster, int P, int S, int O, int A, int M, int hidden,
                                    int dist, void *stream) {
    PGM_REQUIRE(adam_m && adam_v && adam_step && lr, "pgm_ppo_update_f32: null optimizer state");
    PGM_REQUIRE(E > 0 && B > 0 && S / B > 0, "pgm_ppo_update_f32: bad E=%d B=%d for S=%d", E, B, S);
    // the reference's BatchSampler(drop_last=True) yields S // (S // B) minibatches per epoch (a2c/storage.py:133-137), which
    // is B only when the remainder S % B is smaller than one minibatch; otherwise it would take more than E*B steps
    PGM_REQUIRE(S / (S / B) == B, "pgm_ppo_update_f32: S=%d samples in B=%d minibatches of %d leave a remainder of %d >= one "
                "minibatch: the reference would run %d minibatches per epoch; choose S, B with S %% B < S / B", S, B, S / B, S % B, S / (S / B));
    return ppo_common(params, adam_m, adam_v, adam_step, lr, obs, obs_task_stride, action, logp_old, value_old,
                      value_task_stride, returns, adv, perm, perm_shared, E, B, S / B, hyper_host, losses, nullptr,
                      workspace, workspace_bytes, cluster, P, S, O, A, M, hidden, dist, (cudaStream_t)stream);
}

extern "C" int pgm_ppo_update_h_f32(float *params, float *adam_m, float *adam_v, int32_t *adam_step, const double *lr,
                                    const float *obs, size_t obs_task_stride, const float *action,
                                    const float *logp_old, const float *value_old, size_t value_task_stride,
                                    const float *returns, const float *adv, const int32_t *perm, int perm_shared,
                                    int E, int B, const pgm_ppo_hyper *hyper_host, float *losses, void *workspace,
                                    size_t workspace_bytes, int cluster, int P, int S, int O, int A, int M, int hidden,
                                    void *stream) {
    return pgm_ppo_update_x_f32(params, adam_m, adam_v, adam_step, lr, obs, obs_task_stride, action, logp_old, value_old,
                                value_task_stride, returns, adv, perm, perm_shared, E, B, hyper_host, losses, workspace,
                                workspace_bytes, cluster, P, S, O, A, M, hidden, PGM_DIST_GAUSSIAN, stream);
}

extern "C" int pgm_ppo_update_f32(float *params, float *adam_m, float *adam_v, int32_t *adam_step, const double *lr,
                                  const float *obs, size_t obs_task_stride, const float *action,
                                  const float *logp_old, const float *value_old, size_t value_task_stride,
                                  const float *returns, const float *adv, const int32_t *perm, int perm_shared,
                                  int E, int B, const pgm_ppo_hyper *hyper_host, float *losses, void *workspace,
                                  size_t workspace_bytes, int cluster, int P, int S, int O, int A, int M,
                                  void *stream) {
    return pgm_ppo_update_h_f32(params, adam_m, adam_v, adam_step, lr, obs, obs_task_stride, action, logp_old, value_old,
                                value_task_stride, returns, adv, perm, perm_shared, E, B, hyper_host, losses, workspace,
                                workspace_bytes, cluster, P, S, O, A, M, H, stream);
}

extern "C" int pgm_ppo_grad_x_f32(const float *params, const float *obs, size_t obs_task_stride, const float *action,
                                  const float *logp_old, const float *value_old, size_t value_task_stride,
                                  const float *returns, const float *adv, const int32_t *idx, int mb,
                                  const pgm_ppo_hyper *hyper_host, float *grad, float *losses, void *workspace,
                                  size_t workspace_bytes, int cluster, int P, int S, int O, int A, int M, int hidden,
                                  int dist, void *stream) {
    PGM_REQUIRE(grad, "pgm_ppo_grad_f32: null grad");
    return ppo_common(const_cast<float *>(params), nullptr, nullptr, nullptr, nullptr, obs, obs_task_stride, action,
                      logp_old, value_old, value_task_stride, returns, adv, idx, 1, 1, 1, mb, hyper_host, losses, grad,
                      workspace, workspace_bytes, cluster, P, S, O, A, M, hidden, dist, (cudaStream_t)stream);
}

extern "C" int pgm_ppo_grad_h_f32(const float *params, const float *obs, size_t obs_task_stride, const float *action,
                                  const float *logp_old, const float *value_old, size_t value_task_stride,
                                  const float *returns, const float *adv, const int32_t *idx, int mb,
                                  const pgm_ppo_hyper *hyper_host, float *grad, float *losses, void *workspace,
                                  size_t workspace_bytes, int cluster, int P, int S, int O, int A, int M, int hidden,
                                  void *stream) {
    return pgm_ppo_grad_x_f32(params, obs, obs_task_stride, action, logp_old, value_old, value_task_stride, returns, adv,
                              idx, mb, hyper_host, grad, losses, workspace, workspace_bytes, cluster, P, S, O, A, M, hidden,
                              PGM_DIST_GAUSSIAN, stream);
}

extern "C" int pgm_ppo_grad_f32(const float *params, const float *obs, size_t obs_task_stride, const float *action,
                                const float *logp_old, const float *value_old, size_t value_task_stride,
                                const float *returns, const float *adv, const int32_t *idx, int mb,
                                const pgm_ppo_hyper *hyper_host, float *grad, float *losses, void *workspace,
                                size_t workspace_bytes, int cluster, int P, int S, int O, int A, int M, void *stream) {
    return pgm_ppo_grad_h_f32(params, obs, obs_task_stride, action, logp_old, value_old, value_task_stride, returns, adv,
                              idx, mb, hyper_host, grad, losses, workspace, workspace_bytes, cluster, P, S, O, A, M, H,
                              stream);
}
