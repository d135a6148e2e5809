// K3's generic cluster kernel body (k3_ppo_body) and what it shares with the other K3 kernels: the argument block, the
// record layout, the cluster helpers. Included by k3_ppo.cu (Gaussian heads, every kernel family) and k3_cat.cu
// (Categorical heads), so that the two translation units compile in parallel.
#pragma once
#include "net.cuh"

namespace pgm {

struct K3Args {
    float *params, *adam_m, *adam_v;
    int32_t *adam_step;
    const double *lr;
    const float *rec;       // packed records [P][S][RSG]
    const int32_t *perm;    // [P or 1][E][S]  (update)  or  [mb] (grad mode)
    float *losses;          // [P][3]
    float *gpart;           // scratch: partial / reduced gradients [P][2][G][NHP]
    float *pstage;          // scratch: updated parameters on their way to the TMA multicast [P][2][NHP] (fast path, TAIL >= 2)
    float *ssq;             // scratch: squared-norm partials       [P][16]
    float *lpart;           // scratch: loss partial sums           [P][16][4]
    float *grad_out;        // grad mode only: [P][n_par]
    float *mv;              // tensor-core path: Adam moments per half in reference order [P][2 halves][m|v][TC_NHP]
    long long *trace;       // PGM_K3_TRACE builds only: [CTA][4 steps][16 marks] clock64 / globaltimer
    int perm_shared, E, B, mb, S, nsteps, grad_only;
    int Rg;                 // rows per CTA per step (multiple of the chunk size)
    int RSG, RSS, NHP;      // record stride in global / shared memory; padded half size
    int stage_floats;       // fast path: staging floats for row-split partials
    int rs;                 // tensor-core path: CTAs per network half (row split), 1 or 2
    pgm_ppo_hyper hy;
    NetLayout L;
};

// record field offsets (floats): x[0,OP) act[OP,OP+AC) logp_old v_old[M] ret[M] adv; AC = action columns (1 for a
// Categorical head: the category index)
__host__ __device__ inline int rec_stride(const NetLayout &L) { return round_up(L.OP + L.AC + 2 * L.M + 2, 4); }

#ifdef PGM_K3_TRACE
#define PGM_TR(ph)                                                                                   \
    if (a.trace && tid == 0 && s >= 8 && s < 12) {                                                   \
        long long gt_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_));                       \
        a.trace[(((size_t)blockIdx.x * 4 + (s - 8)) * 16 + (ph)) * 2] = clock64();                   \
        a.trace[(((size_t)blockIdx.x * 4 + (s - 8)) * 16 + (ph)) * 2 + 1] = gt_;                     \
    }
#else
#define PGM_TR(ph)
#endif

template <int C>
__device__ __forceinline__ void sync_group() {
    if (C == 1) {
        __syncthreads();
    } else {
        asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
        asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
    }
}

template <int C>
__device__ __forceinline__ unsigned group_rank() {
    if (C == 1) return 0;
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
    return r;
}

// half-local flat parameter index -> offset inside the padded shared-memory image of the half
template <int HW = H>
__device__ __forceinline__ int half_img_off(const HalfNet &n, const NetLayout &L, int e) {
    constexpr int LD = RowTile<HW>::LD, LOG2 = RowTile<HW>::LOG2;
    const int O = L.O;
    if (e < HW * O) { const int j = e / O; return j * L.ldw1 + (e - j * O); }
    e -= HW * O;
    if (e < HW) return (int)(n.b1 - n.W1) + e;
    e -= HW;
    if (e < HW * HW) return (int)(n.W2 - n.W1) + (e >> LOG2) * LD + (e & (HW - 1));
    e -= HW * HW;
    if (e < HW) return (int)(n.b2 - n.W1) + e;
    e -= HW;
    if (e < n.KH * HW) return (int)(n.Wh - n.W1) + (e >> LOG2) * LD + (e & (HW - 1));
    e -= n.KH * HW;
    if (e < n.KH) return (int)(n.bh - n.W1) + e;
    return (int)(n.ls - n.W1) + (e - n.KH);
}

__device__ __forceinline__ float fast_sqrt(float x) { float r; asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

// C: CTAs per task; TM: rows per thread per chunk (chunk = 16*TM rows);
// KG1: 4-column groups of dW1 per thread (OP <= 64*KG1); NA: head rows per thread (A,M <= 16*NA);
// DB: double-buffered record gather; VU: unclipped value loss (every kernel family takes it as a template parameter, so the
// clipped instantiations are the code they were before the option existed).
// HW: hidden width (net.cuh RowTile). A thread's dW2 tile is CG x KQ2 quads by 4x4, its dW1 tile KG1 x CG; at HW = 32
// the 32 k lanes cover OP <= 128 * KG1, at 64 and 128 the 16 k lanes cover OP <= 64 * KG1.
// Generic path (any supported dims, incl. wide observations and C == 1): each CTA updates a 1/G
// slice of its half in global memory and all CTAs reload the parameters (three barriers per step).
// Small networks on C >= 2 take the fast path in k3_fast.cuh instead (hidden width 64).
// The body is shared by k3_ppo_kernel (HW = 64) and k3_ppo_h_kernel (HW = 32, 128).
// CAT: Categorical head (k3_ppo_cat_kernel in k3_cat.cu, every width): the actor head emits A = n logits, the record holds
// one action column (the category index), there is no logstd; the entropy term enters the logits' gradient and the
// reported entropy is the mean over rows and steps.
template <int C, int TM, int KG1, int NA, bool DB, bool VU, int HW, bool CAT = false>
__device__ __forceinline__ void k3_ppo_body(const K3Args &a) {
    using T = RowTile<HW>;
    constexpr int RC = 16 * TM;
    constexpr int RT = T::RT, CT = T::CT, CG = T::CG, LD = T::LD, RPT = RC / RT;
    constexpr int KQ2 = (HW / 4 + RT - 1) / RT;          // k quads of dW2 per thread
    constexpr int NHALF = (C == 1) ? 2 : 1;
    constexpr int G = (C == 1) ? 1 : C / 2;
    static_assert(!(DB && NHALF == 2), "double-buffered gather needs one half per CTA");
    static_assert(RC % RT == 0, "chunk rows must be a multiple of the row lanes");
    extern __shared__ __align__(16) float smem[];
    __shared__ float red[34];
    __shared__ double sh_d[4];

    const NetLayout &L = a.L;
    const int tid = threadIdx.x, tr = tid & (RT - 1), tc = tid >> T::RT_LOG2;
    const int task = blockIdx.x / C;
    const unsigned rank = group_rank<C>();
    const int half0 = (C == 1) ? 0 : (int)(rank / G);
    const int g = (C == 1) ? 0 : (int)(rank % G);
    const int O = L.O, OP = L.OP, A = L.A, M = L.M;
    const int AC = CAT ? 1 : A;   // action columns of a record
    const int ldo = ((A > M ? A : M) | 1);
    const int RSS = a.RSS, RSG = a.RSG;
    const int nchunk = a.Rg / RC;

    // ---- shared memory carve ----
    HalfNet net[NHALF];
    float *p = smem;
#pragma unroll
    for (int hh = 0; hh < NHALF; ++hh) p = halfnet_carve<HW>(net[hh], p, L, half0 + hh);
    float *h1 = p; p += RC * LD;
    float *h2 = p; p += RC * LD;
    float *dz = p; p += RC * LD;
    float *ho = p; p += round_up(RC * ldo, 4);
    float *els = p; p += round_up(RC * ldo, 4);
    float *recb = p;   // [DB ? 2 : 1][RC][RSS]

    float *gparams = a.params + (size_t)task * L.n_par;
#pragma unroll
    for (int hh = 0; hh < NHALF; ++hh) halfnet_load<false, HW, !CAT>(net[hh], gparams, L, half0 + hh);

    const float clip = (float)a.hy.clip_param;
    const float inv_mb = 1.f / (float)a.mb;
    const float vscale = (float)(a.hy.value_loss_coef * 0.5 / ((double)a.mb * M));
    const float omb1 = (float)(1.0 - a.hy.beta1);
    const float b2f = (float)a.hy.beta2, omb2 = (float)(1.0 - a.hy.beta2);
    const float aeps = (float)a.hy.adam_eps;
    const float ecoef = (float)a.hy.entropy_coef;
    const int step0 = a.grad_only ? 0 : a.adam_step[task];
    double b1pow = pow(a.hy.beta1, (double)step0), b2pow = pow(a.hy.beta2, (double)step0);   // thread 0 uses them
    const double lr = a.grad_only ? 0.0 : a.lr[task];

    float loss_act = 0.f, loss_val = 0.f, loss_ent = 0.f;   // running sums (per thread)

    const int32_t *perm = a.perm + ((a.perm_shared || a.grad_only) ? 0 : (size_t)task * a.E * a.S);
    const float *recg = a.rec + (size_t)task * a.S * RSG;
    const int q4 = RSG / 4;

    // gather chunk `ci` (flat index over steps x chunks) into buffer `buf`
    auto gather = [&](int ci, int buf) {
        const int s = ci / nchunk, c = ci - s * nchunk;
        const int e = s / a.B, b = s - e * a.B;
        const int row0 = g * a.Rg + c * RC;                       // first row of this chunk inside the minibatch
        const int32_t *pb = perm + (size_t)e * a.S + (size_t)b * a.mb;
        float *dst = recb + buf * RC * RSS;
        for (int i = tid; i < RC * q4; i += NTHREADS) {
            const int r = i / q4, q = i - r * q4;
            float *d = dst + r * RSS + 4 * q;
            if (row0 + r < a.mb) {
                const int idx = __ldg(pb + row0 + r);
                cp_async16(d, recg + (size_t)idx * RSG + 4 * q);
            } else {
                sts4(d, make_float4(0.f, 0.f, 0.f, 0.f));
            }
        }
        cp_async_commit();
    };

    const int total_chunks = a.nsteps * nchunk;
    if (DB) gather(0, 0);
    __syncthreads();

    for (int s = 0; s < a.nsteps; ++s) {
        PGM_TR(0)
#pragma unroll
        for (int hh = 0; hh < NHALF; ++hh) {
            const int half = half0 + hh;
            const HalfNet &n = net[hh];
            const int KH = n.KH;
            // gradient accumulators (registers, persist over the chunks of this step)
            float gW2[CG][KQ2][4][4], gb2[CG][4], gW1[KG1][CG][4][4], gb1[CG][4], gWh[NA][CG][4], gbh[NA], gls[NA];
#pragma unroll
            for (int jg = 0; jg < CG; ++jg)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                gb2[jg][i] = 0.f; gb1[jg][i] = 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
#pragma unroll
                    for (int kq = 0; kq < KQ2; ++kq) gW2[jg][kq][i][j] = 0.f;
#pragma unroll
                    for (int q = 0; q < KG1; ++q) gW1[q][jg][i][j] = 0.f;
                }
            }
#pragma unroll
            for (int ia = 0; ia < NA; ++ia) {
                gbh[ia] = 0.f; gls[ia] = 0.f;
#pragma unroll
                for (int jg = 0; jg < CG; ++jg) gWh[ia][jg][0] = gWh[ia][jg][1] = gWh[ia][jg][2] = gWh[ia][jg][3] = 0.f;
            }

            for (int c = 0; c < nchunk; ++c) {
                const int ci = s * nchunk + c;
                const float *x;
                if (DB) {
                    cp_async_wait<0>();
                    __syncthreads();            // chunk ci landed; every thread is done with chunk ci-1
                    if (ci + 1 < total_chunks) gather(ci + 1, (ci + 1) & 1);
                    x = recb + (ci & 1) * RC * RSS;
                } else {
                    __syncthreads();            // previous users of recb are done
                    gather(ci, 0);
                    cp_async_wait<0>();
                    __syncthreads();
                    x = recb;
                }
                const int row0 = g * a.Rg + c * RC;

                PGM_TR(1)
                // ---------------- forward ----------------
                half_forward<TM, HW>(x, RSS, n, L, h1, h2, ho, ldo, tr, tc);

                PGM_TR(2)
                // ---------------- loss + d(loss)/d(head output), thread per row ----------------
                if (tid < RC) {
                    const int r = tid;
                    const bool valid = row0 + r < a.mb;
                    const float *rp = x + r * RSS;
                    if (half == 0) {
                        float lp = 0.f, lse = 0.f, ent = 0.f;
                        int act = 0;
                        if (CAT) {      // log-softmax of the logits, log-prob of the taken category, entropy of the row
                            const float *z = ho + r * ldo;
                            act = min(max((int)rp[OP], 0), A - 1);
                            float mx = z[0];
                            for (int j = 1; j < A; ++j) mx = fmaxf(mx, z[j]);
                            float se = 0.f;
                            for (int j = 0; j < A; ++j) se += expf(z[j] - mx);
                            lse = mx + logf(se);
                            for (int j = 0; j < A; ++j) { const float lpj = z[j] - lse; ent -= expf(lpj) * lpj; }
                            lp = z[act] - lse;
                        } else {
                            for (int d = 0; d < A; ++d) {
                                const float ls = n.ls[d], sd = expf(ls);
                                const float diff = rp[OP + d] - ho[r * ldo + d];
                                lp += -(diff * diff) / (2.f * sd * sd) - ls - 0.91893853320467274178f;
                            }
                        }
                        const float ratio = expf(lp - rp[OP + AC]);
                        const float adv = rp[OP + AC + 1 + 2 * M];
                        const float surr1 = ratio * adv;
                        const float rcl = fminf(fmaxf(ratio, 1.f - clip), 1.f + clip);
                        const float surr2 = rcl * adv;
                        const float w1 = surr1 < surr2 ? 1.f : (surr1 == surr2 ? 0.5f : 0.f);
                        const float inr = (ratio >= 1.f - clip && ratio <= 1.f + clip) ? 1.f : 0.f;
                        const float dmin = w1 * adv + (1.f - w1) * adv * inr;
                        const float dlp = valid ? -inv_mb * dmin * ratio : 0.f;
                        if (valid) loss_act -= fminf(surr1, surr2);
                        if (CAT) {
                            // d logp / dz_j = [j = a] - p_j;  d(-ecoef * mean_i H_i) / dz_j = ecoef / mb * p_j (log p_j + H)
                            const float ec = valid ? ecoef * inv_mb : 0.f;
                            if (valid) loss_ent += ent;
                            for (int j = 0; j < A; ++j) {
                                const float lpj = ho[r * ldo + j] - lse, pj = expf(lpj);
                                ho[r * ldo + j] = dlp * ((j == act ? 1.f : 0.f) - pj) + ec * pj * (lpj + ent);
                            }
                        } else {
                            for (int d = 0; d < A; ++d) {
                                const float sd = expf(n.ls[d]);
                                const float iv = 1.f / (sd * sd);
                                const float diff = rp[OP + d] - ho[r * ldo + d];
                                ho[r * ldo + d] = dlp * diff * iv;
                                els[r * ldo + d] = dlp * (diff * diff * iv - 1.f);
                            }
                        }
                    } else {
                        for (int m = 0; m < M; ++m) {
                            const float V = ho[r * ldo + m];
                            const float vo = rp[OP + AC + 1 + m];
                            const float R = rp[OP + AC + 1 + M + m];
                            const float d = V - vo;
                            const float vcl = vo + fminf(fmaxf(d, -clip), clip);
                            const float ea = V - R, eb = vcl - R;
                            // unclipped value loss (VU): lb = -1 < 0 <= la, so max(la, lb) = la and wa = 1, gradient 2 * ea exactly
                            const float la = ea * ea, lb = VU ? -1.f : eb * eb;
                            const float wa = la > lb ? 1.f : (la == lb ? 0.5f : 0.f);
                            const float pas = (d >= -clip && d <= clip) ? 1.f : 0.f;
                            if (valid) loss_val += fmaxf(la, lb);
                            ho[r * ldo + m] = valid ? vscale * (wa * 2.f * ea + (1.f - wa) * 2.f * eb * pas) : 0.f;
                        }
                    }
                }
                __syncthreads();

                PGM_TR(3)
                // ---------------- phase A: head weight grads, dz2 ----------------
                {
                    const int kg = tid & (CT - 1), a0 = tid >> T::CT_LOG2;
#pragma unroll
                    for (int ia = 0; ia < NA; ++ia) {
                        const int aa = a0 + RT * ia;
                        if (aa < KH) {
#pragma unroll 4
                            for (int r = 0; r < RC; ++r) {
                                const float sv = ho[r * ldo + aa];
#pragma unroll
                                for (int jg = 0; jg < CG; ++jg) {
                                    const float4 hv = lds4(h2 + r * LD + 4 * (kg + CT * jg));
                                    float *gw = gWh[ia][jg];
                                    gw[0] = fmaf(sv, hv.x, gw[0]); gw[1] = fmaf(sv, hv.y, gw[1]);
                                    gw[2] = fmaf(sv, hv.z, gw[2]); gw[3] = fmaf(sv, hv.w, gw[3]);
                                }
                                if (kg == 0) gbh[ia] += sv;
                                if (!CAT && half == 0 && kg == 1) gls[ia] += els[r * ldo + aa];
                            }
                        }
                    }
                    float acc[RPT][CG][4];
#pragma unroll
                    for (int i = 0; i < RPT; ++i)
#pragma unroll
                        for (int jg = 0; jg < CG; ++jg) acc[i][jg][0] = acc[i][jg][1] = acc[i][jg][2] = acc[i][jg][3] = 0.f;
                    for (int aa = 0; aa < KH; ++aa) {
#pragma unroll
                        for (int jg = 0; jg < CG; ++jg) {
                            const float4 w = lds4(n.Wh + aa * LD + 4 * (tc + CT * jg));
#pragma unroll
                            for (int i = 0; i < RPT; ++i) {
                                const float sv = ho[(tr + RT * i) * ldo + aa];
                                float *ac = acc[i][jg];
                                ac[0] = fmaf(sv, w.x, ac[0]); ac[1] = fmaf(sv, w.y, ac[1]);
                                ac[2] = fmaf(sv, w.z, ac[2]); ac[3] = fmaf(sv, w.w, ac[3]);
                            }
                        }
                    }
#pragma unroll
                    for (int i = 0; i < RPT; ++i)
#pragma unroll
                    for (int jg = 0; jg < CG; ++jg) {
                        const int o = (tr + RT * i) * LD + 4 * (tc + CT * jg);
                        const float4 hv = lds4(h2 + o);
                        const float *ac = acc[i][jg];
                        sts4(dz + o, make_float4(ac[0] * (1.f - hv.x * hv.x), ac[1] * (1.f - hv.y * hv.y),
                                                 ac[2] * (1.f - hv.z * hv.z), ac[3] * (1.f - hv.w * hv.w)));
                    }
                }
                __syncthreads();

                PGM_TR(4)
                // ---------------- phase B: dW2, db2, dz1 (into the h2 buffer) ----------------
                {
                    const int tj = tid & (CT - 1), tk = tid >> T::CT_LOG2;
#pragma unroll 4
                    for (int r = 0; r < RC; ++r) {
#pragma unroll
                        for (int jg = 0; jg < CG; ++jg) {
                            const float4 dv = lds4(dz + r * LD + 4 * (tj + CT * jg));
                            const float dd[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
                            for (int kq = 0; kq < KQ2; ++kq) {
                                if (4 * RT * KQ2 > HW && 4 * (tk + RT * kq) >= HW) continue;   // idle k lanes at HW = 32
                                const float4 hv = lds4(h1 + r * LD + 4 * (tk + RT * kq));
#pragma unroll
                                for (int jj = 0; jj < 4; ++jj) {
                                    float *gw = gW2[jg][kq][jj];
                                    gw[0] = fmaf(dd[jj], hv.x, gw[0]); gw[1] = fmaf(dd[jj], hv.y, gw[1]);
                                    gw[2] = fmaf(dd[jj], hv.z, gw[2]); gw[3] = fmaf(dd[jj], hv.w, gw[3]);
                                }
                            }
                            if (tk == 0) { gb2[jg][0] += dv.x; gb2[jg][1] += dv.y; gb2[jg][2] += dv.z; gb2[jg][3] += dv.w; }
                        }
                    }
                    float acc[RPT][CG][4];
#pragma unroll
                    for (int i = 0; i < RPT; ++i)
#pragma unroll
                        for (int jg = 0; jg < CG; ++jg) acc[i][jg][0] = acc[i][jg][1] = acc[i][jg][2] = acc[i][jg][3] = 0.f;
#pragma unroll 2
                    for (int j = 0; j < HW; j += 4) {
                        float4 av[RPT], bv[CG][4];
#pragma unroll
                        for (int i = 0; i < RPT; ++i) av[i] = lds4(dz + (tr + RT * i) * LD + j);
#pragma unroll
                        for (int jg = 0; jg < CG; ++jg)
#pragma unroll
                            for (int jj = 0; jj < 4; ++jj) bv[jg][jj] = lds4(n.W2 + (j + jj) * LD + 4 * (tc + CT * jg));
#pragma unroll
                        for (int i = 0; i < RPT; ++i) {
                            const float aa[4] = {av[i].x, av[i].y, av[i].z, av[i].w};
#pragma unroll
                            for (int jg = 0; jg < CG; ++jg)
#pragma unroll
                            for (int jj = 0; jj < 4; ++jj) {
                                float *ac = acc[i][jg];
                                ac[0] = fmaf(aa[jj], bv[jg][jj].x, ac[0]); ac[1] = fmaf(aa[jj], bv[jg][jj].y, ac[1]);
                                ac[2] = fmaf(aa[jj], bv[jg][jj].z, ac[2]); ac[3] = fmaf(aa[jj], bv[jg][jj].w, ac[3]);
                            }
                        }
                    }
#pragma unroll
                    for (int i = 0; i < RPT; ++i)
#pragma unroll
                    for (int jg = 0; jg < CG; ++jg) {
                        const int o = (tr + RT * i) * LD + 4 * (tc + CT * jg);
                        const float4 hv = lds4(h1 + o);
                        const float *ac = acc[i][jg];
                        sts4(h2 + o, make_float4(ac[0] * (1.f - hv.x * hv.x), ac[1] * (1.f - hv.y * hv.y),
                                                 ac[2] * (1.f - hv.z * hv.z), ac[3] * (1.f - hv.w * hv.w)));
                    }
                }
                __syncthreads();

                PGM_TR(5)
                // ---------------- phase C: dW1, db1 ----------------
                {
                    const int tj = tid & (CT - 1), tk = tid >> T::CT_LOG2;
#pragma unroll
                    for (int q = 0; q < KG1; ++q) {
                        const int k0 = 4 * (tk + RT * q);
                        if (k0 < OP) {
#pragma unroll 4
                            for (int r = 0; r < RC; ++r) {
#pragma unroll
                                for (int jg = 0; jg < CG; ++jg) {
                                    const float4 dv = lds4(h2 + r * LD + 4 * (tj + CT * jg));
                                    const float4 xv = lds4(x + r * RSS + k0);
                                    const float dd[4] = {dv.x, dv.y, dv.z, dv.w};
#pragma unroll
                                    for (int jj = 0; jj < 4; ++jj) {
                                        float *gw = gW1[q][jg][jj];
                                        gw[0] = fmaf(dd[jj], xv.x, gw[0]); gw[1] = fmaf(dd[jj], xv.y, gw[1]);
                                        gw[2] = fmaf(dd[jj], xv.z, gw[2]); gw[3] = fmaf(dd[jj], xv.w, gw[3]);
                                    }
                                    if (q == 0 && tk == 0) { gb1[jg][0] += dv.x; gb1[jg][1] += dv.y; gb1[jg][2] += dv.z; gb1[jg][3] += dv.w; }
                                }
                            }
                        }
                    }
                }
                // no barrier needed here: the next chunk's forward (or the barrier below) orders
                // the reuse of h2 / x behind every thread's phase C
            }

            PGM_TR(6)
            // ---- write this CTA's partial gradient of `half` to its scratch slot ----
            {
                float *gp = a.gpart + ((size_t)(task * 2 + half) * G + g) * a.NHP;
                const int tj = tid & (CT - 1), tk = tid >> T::CT_LOG2;
                const int lb1 = HW * O, lW2 = lb1 + HW, lb2 = lW2 + HW * HW, lWh = lb2 + HW, lbh = lWh + KH * HW, lls = lbh + KH;
#pragma unroll
                for (int q = 0; q < KG1; ++q)
#pragma unroll
                    for (int jg = 0; jg < CG; ++jg)
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj)
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const int k = 4 * (tk + RT * q) + kk;
                            if (k < O) gp[(4 * (tj + CT * jg) + jj) * O + k] = gW1[q][jg][jj][kk];
                        }
#pragma unroll
                for (int jg = 0; jg < CG; ++jg)
#pragma unroll
                    for (int kq = 0; kq < KQ2; ++kq) {
                        if (4 * RT * KQ2 > HW && 4 * (tk + RT * kq) >= HW) continue;
#pragma unroll
                        for (int jj = 0; jj < 4; ++jj) {
                            const float *gw = gW2[jg][kq][jj];
                            sts4(gp + lW2 + (4 * (tj + CT * jg) + jj) * HW + 4 * (tk + RT * kq), make_float4(gw[0], gw[1], gw[2], gw[3]));
                        }
                    }
                if (tk == 0) {
#pragma unroll
                    for (int jg = 0; jg < CG; ++jg) {
                        sts4(gp + lb1 + 4 * (tj + CT * jg), make_float4(gb1[jg][0], gb1[jg][1], gb1[jg][2], gb1[jg][3]));
                        sts4(gp + lb2 + 4 * (tj + CT * jg), make_float4(gb2[jg][0], gb2[jg][1], gb2[jg][2], gb2[jg][3]));
                    }
                }
                const int kg = tid & (CT - 1), a0 = tid >> T::CT_LOG2;
#pragma unroll
                for (int ia = 0; ia < NA; ++ia) {
                    const int aa = a0 + RT * ia;
                    if (aa < KH) {
#pragma unroll
                        for (int jg = 0; jg < CG; ++jg)
                            sts4(gp + lWh + aa * HW + 4 * (kg + CT * jg), make_float4(gWh[ia][jg][0], gWh[ia][jg][1], gWh[ia][jg][2], gWh[ia][jg][3]));
                        if (kg == 0) gp[lbh + aa] = gbh[ia];
                        if (!CAT && half == 0 && kg == 1) gp[lls + aa] = gls[ia];
                    }
                }
            }
            if (!CAT && half == 0 && g == 0 && tid == 0) {   // entropy with the parameters this step started from
                float ent = 0.f;
                for (int d = 0; d < A; ++d) ent += 0.5f + 0.91893853320467274178f + n.ls[d];
                loss_ent += ent;
            }
        }   // halves

        PGM_TR(7)
        sync_group<C>();   // (1) all partial gradients of this task are in L2
        PGM_TR(8)

        // ---- reduce my slice over the G partials, squared-norm partial ----
        float sq = 0.f;
#pragma unroll
        for (int hh = 0; hh < NHALF; ++hh) {
            const int half = half0 + hh;
            const int nH = L.half_size<CAT>(half, HW);
            const int per = round_up((nH + G - 1) / G, 4);
            const int s0 = g * per, s1 = min(nH, s0 + per);
            float *slot0 = a.gpart + (size_t)(task * 2 + half) * G * a.NHP;
            const int lls = L.n_base + L.head_dim(half) * HW + L.head_dim(half);
            for (int e = s0 + tid; e < s1; e += NTHREADS) {
                float gs = 0.f;
#pragma unroll
                for (int gg = 0; gg < G; ++gg) gs += __ldcg(slot0 + (size_t)gg * a.NHP + e);
                if (!CAT && half == 0 && e >= lls) gs -= ecoef;      // d(-ecoef * entropy)/d logstd
                sq = fmaf(gs, gs, sq);
                if (a.grad_only) a.grad_out[(size_t)task * L.n_par + L.to_global(half, e)] = gs;
                else slot0[(size_t)g * a.NHP + e] = gs;   // keep the reduced value in my own slot (only I read it)
            }
        }
        sq = block_sum(sq, red);
        if (tid == 0) a.ssq[task * 16 + rank] = sq;
        if (a.grad_only) break;

        if (tid == 0) {   // Adam scalars of step k = step0 + s + 1, in double
            b1pow *= a.hy.beta1; b2pow *= a.hy.beta2;
            sh_d[0] = lr / (1.0 - b1pow);            // step_size
            sh_d[1] = 1.0 / sqrt(1.0 - b2pow);       // 1 / bias_correction2_sqrt
        }
        sync_group<C>();   // (2) squared-norm partials visible

        float tot = 0.f;
#pragma unroll
        for (int rr = 0; rr < C; ++rr) tot += __ldcg(a.ssq + task * 16 + rr);
        const float coef = fminf(1.f, (float)a.hy.max_grad_norm / (sqrtf(tot) + 1e-6f));
        const float step_size = (float)sh_d[0], ibc2 = (float)sh_d[1];
#pragma unroll
        for (int hh = 0; hh < NHALF; ++hh) {
            const int half = half0 + hh;
            const int nH = L.half_size<CAT>(half, HW);
            const int per = round_up((nH + G - 1) / G, 4);
            const int s0 = g * per, s1 = min(nH, s0 + per);
            const float *mine = a.gpart + ((size_t)(task * 2 + half) * G + g) * a.NHP;
            for (int e = s0 + tid; e < s1; e += NTHREADS) {
                const size_t gi = (size_t)task * L.n_par + L.to_global(half, e);
                const float gr = __ldcg(mine + e) * coef;
                float m = a.adam_m[gi], v = a.adam_v[gi], pw = a.params[gi];
                m = fmaf(gr - m, omb1, m);                 // exp_avg.lerp_(grad, 1 - beta1)
                v = fmaf(omb2 * gr, gr, v * b2f);          // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
                const float denom = sqrtf(v) * ibc2 + aeps;
                pw -= step_size * (m / denom);
                a.adam_m[gi] = m; a.adam_v[gi] = v; a.params[gi] = pw;
            }
        }
        sync_group<C>();   // (3) new parameters of this task are in L2
#pragma unroll
        for (int hh = 0; hh < NHALF; ++hh) halfnet_load<true, HW, !CAT>(net[hh], gparams, L, half0 + hh);
        __syncthreads();
    }

    // ---- losses: per-CTA partial sums -> rank 0 combines in fixed order ----
    {
        const float la = block_sum(loss_act, red), lv = block_sum(loss_val, red), le = block_sum(loss_ent, red);
        if (tid == 0) {
            a.lpart[(task * 16 + rank) * 4 + 0] = lv;
            a.lpart[(task * 16 + rank) * 4 + 1] = la;
            a.lpart[(task * 16 + rank) * 4 + 2] = le;
        }
        sync_group<C>();
        if (rank == 0 && tid == 0) {
            float sv = 0.f, sa = 0.f, se = 0.f;
            for (int rr = 0; rr < C; ++rr) {
                sv += __ldcg(a.lpart + (task * 16 + rr) * 4 + 0);
                sa += __ldcg(a.lpart + (task * 16 + rr) * 4 + 1);
                se += __ldcg(a.lpart + (task * 16 + rr) * 4 + 2);
            }
            const float ns = (float)a.nsteps;
            a.losses[task * 3 + 0] = sv * 0.5f / ((float)a.mb * M) / ns;
            a.losses[task * 3 + 1] = sa * inv_mb / ns;
            a.losses[task * 3 + 2] = CAT ? se * inv_mb / ns : se / ns;   // Categorical: se sums the rows' entropies
            if (!a.grad_only) a.adam_step[task] = step0 + a.nsteps;
        }
    }
}

// Launch of the generic kernel for a Categorical head (k3_cat.cu): hidden width, CTAs per task, chunk rows / 16, the wide
// variant (OP > 64 or n > 16) and the unclipped value loss as planned by k3_plan.
int k3_launch_cat(const K3Args &a, int hidden, int C, int TM, bool wide, bool vu, size_t smem, int P, cudaStream_t st);

}  // namespace pgm
