// K3 fast path: small networks (OP <= 48, A, M <= 16) on a cluster of C >= 2 CTAs.
// Included by k3_ppo.cu (shares K3Args, sync_group, half_img_off, PGM_TR).
//
// Per CTA: one network half (parameters + Adam moments + reduced gradient resident in shared
// memory in one padded "image" layout), RC = 16*TM minibatch rows per chunk.
// Chunk pipeline (each arrow is one __syncthreads):
//   records landed -> L1 fwd -> [issue next gather] L2 fwd -> head + per-element loss terms
//   -> per-row loss (actor) -> dz2 -> dW2, db2, dz1 -> {dW1 | dWh} on disjoint thread groups
// Step tail = all-reduce of the half's gradient + Adam, template parameter TAIL (all variants bit-identical; A/B table in
// k3_ppo.cu). Default (TAIL = 5), no cluster barrier inside the step:
//   combine row-split partials -> partial gradient image in OWN smem -> 8 threads issue one cp.async.bulk per slice owner
//   (smem -> the owner's per-source slot, completing the owner's mbarrier R) -> owner adds its G slots in fixed order,
//   sends its squared-norm partial to every CTA with st.async (mbarrier N) -> clip + Adam on the slice (moments of the slice
//   live in smem for the whole launch) -> updated slice to an L2 staging row, ONE TMA bulk copy with cluster multicast lands
//   it in every resident image of the half (mbarrier S).
// TAIL = 0 is the round-1 form: three barrier.cluster, partials pulled with ld.shared::cluster, parameters pushed with
// st.shared::cluster.
#pragma once

namespace pgm {


__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t cta) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta)); return r;
}
__device__ __forceinline__ float4 ld_dsmem4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void st_dsmem4(uint32_t addr, float4 v) {
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_dsmem2x64(uint32_t addr, ulonglong2 v) {
    asm volatile("st.shared::cluster.v2.b64 [%0], {%1, %2};" ::"r"(addr), "l"(v.x), "l"(v.y) : "memory");
}
__device__ __forceinline__ void st_dsmem1(uint32_t addr, float v) {
    asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}

// ---- packed FP32x2 FMA (Blackwell FFMA2): two FMAs per lane per issue slot -----------------------
typedef unsigned long long u64;
__device__ __forceinline__ u64 ffma2(u64 a, u64 b, u64 c) {       // (a.lo*b.lo + c.lo, a.hi*b.hi + c.hi)
    u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d;
}
__device__ __forceinline__ u64 ffma2_s(float s, u64 b, u64 c) {   // (s*b.lo + c.lo, s*b.hi + c.hi); ptxas folds the
    u64 d;                                                        // broadcast into the FFMA2 .F32 operand form
    asm("{ .reg .b64 t; mov.b64 t, {%1, %1}; fma.rn.f32x2 %0, t, %2, %3; }" : "=l"(d) : "f"(s), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ float2 unpack2(u64 v) { float2 r; asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v)); return r; }
__device__ __forceinline__ u64 pack2(float lo, float hi) { u64 d; asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi)); return d; }
__device__ __forceinline__ ulonglong2 lds2x64(const float *p) { return *reinterpret_cast<const ulonglong2 *>(p); }

struct K3FastPlan {       // how phase C splits the 16 thread slots (slot = tid >> 4)
    int nkg, nrs1, nW1;   // dW1: k-groups, row splits, slots used
    int nWh, nrsH, nA;    // dWh: slots, row splits, distinct head rows per pass
};

__host__ __device__ inline K3FastPlan k3_fast_plan(int OP, int KH) {
    K3FastPlan f;
    f.nkg = OP / 4;
    f.nrs1 = 12 / f.nkg; if (f.nrs1 < 1) f.nrs1 = 1;
    f.nW1 = f.nkg * f.nrs1;
    f.nWh = 16 - f.nW1;
    f.nrsH = f.nWh / KH; if (f.nrsH < 1) f.nrsH = 1;
    f.nA = f.nWh / f.nrsH;
    return f;
}
// staging floats needed to combine row-split partials of dW1/db1 and dWh/dbh/dls
__host__ __device__ inline int k3_fast_stage_floats(int OP, int KH) {
    const K3FastPlan f = k3_fast_plan(OP, KH);
    return (f.nrs1 - 1) * (H * OP + H) + (f.nrsH - 1) * KH * (H + 4);
}

template <int TM, int KU>
__device__ __forceinline__ void layer_fwd_fast(const float *__restrict__ in, int ldi, const float *__restrict__ W,
                                               int ldw, const float *__restrict__ bias, int K,
                                               float *__restrict__ out, int tr, int tc) {
    // acc[i][c] holds (sum over even k, sum over odd k) of in[r_i][k] * W[j_c][k]
    u64 acc[TM][4];
#pragma unroll
    for (int i = 0; i < TM; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0ull;
    const float *ip = in + tr * ldi;
    const float *wp = W + 4 * tc * ldw;
    // KU k-blocks unrolled: with two warps per scheduler only independent loads of later k-blocks hide the LDS latency
#pragma unroll(KU)
    for (int k = 0; k < K; k += 4) {
        ulonglong2 av[TM], b[4];
#pragma unroll
        for (int i = 0; i < TM; ++i) av[i] = lds2x64(ip + i * 16 * ldi + k);
#pragma unroll
        for (int c = 0; c < 4; ++c) b[c] = lds2x64(wp + c * ldw + k);
#pragma unroll
        for (int i = 0; i < TM; ++i)
#pragma unroll
            for (int c = 0; c < 4; ++c) { acc[i][c] = ffma2(av[i].x, b[c].x, acc[i][c]); acc[i][c] = ffma2(av[i].y, b[c].y, acc[i][c]); }
    }
    const float4 bv = lds4(bias + 4 * tc);
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        const float2 s0 = unpack2(acc[i][0]), s1 = unpack2(acc[i][1]), s2 = unpack2(acc[i][2]), s3 = unpack2(acc[i][3]);
        sts4(out + (tr + 16 * i) * LDH + 4 * tc,
             make_float4(fast_tanh(bv.x + (s0.x + s0.y)), fast_tanh(bv.y + (s1.x + s1.y)),
                         fast_tanh(bv.z + (s2.x + s2.y)), fast_tanh(bv.w + (s3.x + s3.y))));
    }
}

// Step tails (all bit-identical):
// TAIL = 0  : sliced Adam, three cluster barriers per step (partials pulled from the peers' images, new parameters pushed).
// TAIL = 1  : (RA) partial gradient tiles go straight from registers into the slice OWNER's per-source slots, the owner adds its
//             G slots in fixed order and pushes the reduced slice to every CTA of the half, and every CTA runs Adam on the whole
//             half redundantly (moments of the whole half resident) -- two cluster barriers per step, nothing is pulled.
//             Same operations in the same order as RA = false: results are bit-identical.
// TAIL = 2  : as TAIL = 0, but the parameter broadcast goes through the TMA: every CTA stores its updated slice to an
//             L2-resident staging row and issues ONE bulk copy with cluster multicast (cp.async.bulk ... .multicast::cluster)
//             that lands the slice in the resident image of every CTA of the half; an mbarrier per CTA counts the bytes of
//             the G slices, so the third cluster barrier disappears. Bit-identical results.
// TAIL = 3  : as TAIL = 2, and the gradient exchange goes through L2 instead of distributed shared memory: every CTA stores
//             its partial gradient image to its scratch slot in global memory, and after barrier (1) the slice owners read the
//             G partials with ld.global.cg (L2 bandwidth per SM is several times the SM-to-SM network's ~17 B/clk).
// TAIL = 4  : as TAIL = 2, and the gradient reduce-scatter is PUSHED by the bulk-copy engine: every CTA writes its partial
//             image to its own shared memory as before, then 8 threads issue one cp.async.bulk shared::cta -> shared::cluster
//             per slice owner into that owner's per-source slot; the owner's mbarrier counts the bytes of its G incoming
//             slices, so barrier (1) disappears as well and nothing is pulled through ld.shared::cluster. The owner adds
//             its G local slots in the same fixed order. One cluster barrier per step is left (the norm exchange).
// TAIL = 5  : as TAIL = 4, and the squared-norm partials travel with st.async ... mbarrier::complete_tx into every CTA's
//             mbarrier: NO cluster barrier is left inside the step, the optimiser step is pure dataflow over three mbarriers
//             (gradient slices in, norm partials in, parameter slices in). Ordering argument in DESIGN.md section 4.
// TAIL = 6  : as TAIL = 5, and the slices that hold only dW2 (5 of 8 at Walker2d dims, 70 % of the bytes) leave EARLY: dW2 is
//             final after the {dW2, dz1} phase of the step's last chunk, so its tiles are written to the image there and the
//             bulk copies of the W2-only slices fly under phase C, the row-split combine and the rest of the image write.
template <int C, int TM, int TAIL, bool VU = false>
__global__ void __launch_bounds__(NTHREADS, 1) k3_ppo_fast_kernel(const K3Args a) {
    constexpr bool RA = TAIL == 1, MC = TAIL >= 2, GL = TAIL == 3, BP = TAIL >= 4, NB = TAIL >= 5, EP = TAIL == 6;
    constexpr int RC = 16 * TM;
    constexpr int G = C / 2;
    constexpr int NU = 4;                 // gather items per thread (RC * RSG/4 <= NU * 256, checked on host)
    static_assert(C >= 2, "fast path needs one CTA per network half");
    extern __shared__ __align__(16) float smem[];
    __shared__ float red[34];
    __shared__ double sh_d[4];
    __shared__ float ssqS[16];            // squared-norm partials of all C CTAs (same offset in every CTA)
    __shared__ __align__(8) unsigned long long mbarS;   // TAIL >= 2: counts the bytes of the G multicast parameter slices
    __shared__ __align__(8) unsigned long long mbarR;   // TAIL >= 4: counts the bytes of the G incoming gradient slices
    __shared__ __align__(8) unsigned long long mbarN;   // TAIL = 5: counts the bytes of the C incoming squared-norm partials

    const NetLayout &L = a.L;
    const int tid = threadIdx.x, tr = tid & 15, tc = tid >> 4;
    const int task = blockIdx.x / C;
    const unsigned rank = group_rank<C>();
    const int half = (int)(rank / G);
    const int g = (int)(rank % G);
    const int OP = L.OP, A = L.A, M = L.M;
    const int ldo = ((A > M ? A : M) | 1);
    const int RSS = a.RSS, RSG = a.RSG;
    const int nchunk = a.Rg / RC;

    // ---- shared memory carve ----
    HalfNet n;
    float *p = halfnet_carve(n, smem, L, half);
    const int KH = n.KH;
    const int NIMG = halfnet_smem_floats(L, half);
    float *h1 = p; p += RC * LDH;
    float *h2 = p; p += RC * LDH;
    float *dz = p; p += RC * LDH;
    float *d1 = p; p += RC * LDH;
    float *ho = p; p += round_up(RC * ldo, 4);
    float *els = p; p += round_up(RC * ldo, 4);
    float *lpe = p; p += round_up(RC * ldo, 4);
    float *dlpS = p; p += RC;
    float *stg = p; p += round_up(a.stage_floats, 4);
    float *recb = p; p += 2 * RC * RSS;
    const int n4 = NIMG >> 2;                       // float4s in the image
    const int per4 = (n4 + G - 1) / G;              // float4s per slice
    const int sl0 = g * per4, sl1 = min(n4, sl0 + per4);   // my slice [sl0, sl1) in float4 units
    // RA = false: gP = this CTA's partial gradient (image layout), read by peers; moments + reduced gradient of my slice
    // RA = true : gP = G per-source slots of my slice (written by the peers), gS = reduced gradient of the whole half
    //             (written by the slice owners), mS / vS = moments of the whole half
    float *gP = p; p += RA ? G * 4 * per4 : (GL ? 0 : a.NHP);
    float *gPg = a.gpart + ((size_t)(task * 2 + half) * G + g) * a.NHP;      // TAIL = 3: my partial image in global memory
    float *slotB = p; p += BP ? G * 4 * per4 : 0;                            // TAIL = 4: G per-source slots of my slice
    float *gS = p; p += RA ? G * 4 * per4 : 4 * per4;
    const int nmom = RA ? NIMG : 4 * per4;
    float *mS = p, *vS = p + nmom;
    const uint32_t magic = (uint32_t)((0x100000000ull + (unsigned)per4 - 1) / (unsigned)per4);   // i4 / per4 == umulhi(i4, magic)

    if (MC && tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbarS)));
        if (BP) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbarR)));
        if (NB) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbarN)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");     // visible to the peers' multicasts: barrier (1)
    }                                                                          // and (2) of step 0 come before the first one
    if (BP) sync_group<C>();     // no barrier precedes the first remote signal in these tails: publish the mbarrier inits now
    float *gparams = a.params + (size_t)task * L.n_par;
    halfnet_load<false>(n, gparams, L, half);
    for (int i = tid; i < nmom; i += NTHREADS) { mS[i] = 0.f; vS[i] = 0.f; }
    for (int i = tid; i < (RA ? G * 4 * per4 : (GL ? 0 : a.NHP)); i += NTHREADS) gP[i] = 0.f;   // padding entries stay zero for the whole launch
    if (RA) for (int i = tid; i < G * 4 * per4; i += NTHREADS) gS[i] = 0.f;
    for (int i = tid; i < RC; i += NTHREADS) dlpS[i] = 1.f;       // the critic never rewrites it
    __syncthreads();
    if (!a.grad_only) {
        const int nH = L.half_size(half);
        for (int e = tid; e < nH; e += NTHREADS) {
            const int io = half_img_off(n, L, e);
            if (RA || (io >= 4 * sl0 && io < 4 * sl1)) {
                const size_t gi = (size_t)task * L.n_par + L.to_global(half, e);
                mS[io - (RA ? 0 : 4 * sl0)] = a.adam_m[gi];
                vS[io - (RA ? 0 : 4 * sl0)] = a.adam_v[gi];
            }
        }
    }
    const float clip = (float)a.hy.clip_param;
    const float inv_mb = 1.f / (float)a.mb;
    const float vscale = (float)(a.hy.value_loss_coef * 0.5 / ((double)a.mb * M));
    const float omb1 = (float)(1.0 - a.hy.beta1);
    const float b2f = (float)a.hy.beta2, omb2 = (float)(1.0 - a.hy.beta2);
    const float aeps = (float)a.hy.adam_eps;
    const float ecoef = (float)a.hy.entropy_coef;
    const int step0 = a.grad_only ? 0 : a.adam_step[task];
    double b1pow = pow(a.hy.beta1, (double)step0), b2pow = pow(a.hy.beta2, (double)step0);
    const double lr = a.grad_only ? 0.0 : a.lr[task];
    float loss_act = 0.f, loss_val = 0.f, loss_ent = 0.f;

    const int32_t *perm = a.perm + ((a.perm_shared || a.grad_only) ? 0 : (size_t)task * a.E * a.S);
    const float *recg = a.rec + (size_t)task * a.S * RSG;
    const int q4 = RSG / 4;
    const int nitems = RC * q4;

    // record gather, split in two so that the index loads fly while the CTA computes
    int gidx[NU];
    auto gather_idx = [&](int ci) {
        const int s = ci / nchunk, c = ci - s * nchunk;
        const int e = s / a.B, b = s - e * a.B;
        const int row0 = g * a.Rg + c * RC;
        const int32_t *pb = perm + (size_t)e * a.S + (size_t)b * a.mb;
#pragma unroll
        for (int u = 0; u < NU; ++u) {
            const int i = tid + u * NTHREADS;
            const int r = i / q4;
            gidx[u] = (i < nitems && row0 + r < a.mb) ? __ldg(pb + row0 + r) : -1;
        }
    };
    auto gather_issue = [&](int buf) {
        float *dst = recb + buf * RC * RSS;
#pragma unroll
        for (int u = 0; u < NU; ++u) {
            const int i = tid + u * NTHREADS;
            if (i < nitems) {
                const int r = i / q4, q = i - r * q4;
                float *d = dst + r * RSS + 4 * q;
                if (gidx[u] >= 0) cp_async16(d, recg + (size_t)gidx[u] * RSG + 4 * q);
                else sts4(d, make_float4(0.f, 0.f, 0.f, 0.f));
            }
        }
        cp_async_commit();
    };

    // phase C thread roles (uniform per CTA)
    const K3FastPlan fp = k3_fast_plan(OP, KH);
    const int slot = tid >> 4, l16 = tid & 15;
    const bool isW1 = slot < fp.nW1;
    const int kg1 = isW1 ? slot % fp.nkg : 0, rs1 = isW1 ? slot / fp.nkg : 0;
    const int sh = slot - fp.nW1;
    const int aslot = isW1 ? 0 : sh / fp.nrsH, rsh = isW1 ? 0 : sh % fp.nrsH;
    const bool isWh = !isW1 && aslot < fp.nA;
    const int r1lo = rs1 * RC / fp.nrs1, r1hi = (rs1 + 1) * RC / fp.nrs1;
    const int rhlo = rsh * RC / fp.nrsH, rhhi = (rsh + 1) * RC / fp.nrsH;

    const int total_chunks = a.nsteps * nchunk;
    gather_idx(0);
    gather_issue(0);
    __syncthreads();

    for (int s = 0; s < a.nsteps; ++s) {
        PGM_TR(0)
        // weight-gradient tiles as packed pairs: g*[row][0] = cols (0,1), g*[row][1] = cols (2,3)
        u64 gW2[4][2], gW1[4][2], gWh[4][2];
        float gb2[4], gb1[4], gbh[4], gls[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            gb2[i] = gb1[i] = gbh[i] = gls[i] = 0.f;
            gW2[i][0] = gW2[i][1] = gW1[i][0] = gW1[i][1] = gWh[i][0] = gWh[i][1] = 0ull;
        }

        for (int c = 0; c < nchunk; ++c) {
            const int ci = s * nchunk + c;
            cp_async_wait<0>();
            __syncthreads();                       // chunk ci landed; everyone is done with chunk ci-1
            const float *x = recb + (ci & 1) * RC * RSS;
            const bool more = ci + 1 < total_chunks;
            if (more) gather_idx(ci + 1);          // index loads in flight during layer 1
            const int row0 = g * a.Rg + c * RC;
            PGM_TR(1)

            // ---------------- forward ----------------
            layer_fwd_fast<TM, (TM == 2 ? 4 : 2)>(x, RSS, n.W1, L.ldw1, n.b1, OP, h1, tr, tc);
            if (more) gather_issue((ci + 1) & 1);  // async copies overlap layer 2 .. backward
            __syncthreads();
            layer_fwd_fast<TM, (TM == 2 ? H / 4 : 2)>(h1, LDH, n.W2, LDH, n.b2, H, h2, tr, tc);
            __syncthreads();

            // ---------------- head + per-element loss terms: item = (head row aa, batch row r) ----------------
            for (int i = tid; i < RC * KH; i += NTHREADS) {
                const int aa = i / RC, r = i - aa * RC;
                const float *hp = h2 + r * LDH, *wp = n.Wh + aa * LDH;
                u64 ac0 = 0ull, ac1 = 0ull;
#pragma unroll
                for (int k = 0; k < H; k += 4) {
                    const ulonglong2 hv = lds2x64(hp + k), wv = lds2x64(wp + k);
                    ac0 = ffma2(hv.x, wv.x, ac0); ac1 = ffma2(hv.y, wv.y, ac1);
                }
                const float2 q0 = unpack2(ac0), q1 = unpack2(ac1);
                const float acc = n.bh[aa] + ((q0.x + q0.y) + (q1.x + q1.y));
                const float *rp = x + r * RSS;
                if (half == 0) {
                    const float ls = n.ls[aa];
                    const float iv = expf(-2.f * ls);
                    const float diff = rp[OP + aa] - acc;
                    const float t = diff * diff * iv;
                    ho[r * ldo + aa] = diff * iv;                                 // d logp / d mean
                    els[r * ldo + aa] = t - 1.f;                                  // d logp / d logstd
                    lpe[r * ldo + aa] = -0.5f * t - ls - 0.91893853320467274178f;  // log N(a | mean, std)
                } else {
                    const bool valid = row0 + r < a.mb;
                    const float V = acc, vo = rp[OP + A + 1 + aa], R = rp[OP + A + 1 + M + aa];
                    const float dlt = V - vo;
                    const float vcl = vo + fminf(fmaxf(dlt, -clip), clip);
                    const float ea = V - R, eb = vcl - R;
                    // unclipped value loss (VU): lb = -1 < 0 <= la, so max(la, lb) = la and wa = 1, gradient 2 * ea exactly
                    const float la = ea * ea, lb = VU ? -1.f : eb * eb;
                    const float wa = la > lb ? 1.f : (la == lb ? 0.5f : 0.f);
                    const float pas = (dlt >= -clip && dlt <= clip) ? 1.f : 0.f;
                    if (valid) loss_val += fmaxf(la, lb);
                    ho[r * ldo + aa] = valid ? vscale * (wa * 2.f * ea + (1.f - wa) * 2.f * eb * pas) : 0.f;
                }
            }
            __syncthreads();
            PGM_TR(2)
            // ---------------- per-row surrogate (actor): d loss / d logp ----------------
            if (half == 0) {
                if (tid < RC) {
                    const int r = tid;
                    const bool valid = row0 + r < a.mb;
                    const float *rp = x + r * RSS;
                    float lp = 0.f;
                    for (int d = 0; d < A; ++d) lp += lpe[r * ldo + d];
                    const float ratio = expf(lp - rp[OP + A]);
                    const float adv = rp[OP + A + 1 + 2 * M];
                    const float surr1 = ratio * adv;
                    const float rcl = fminf(fmaxf(ratio, 1.f - clip), 1.f + clip);
                    const float surr2 = rcl * adv;
                    const float w1 = surr1 < surr2 ? 1.f : (surr1 == surr2 ? 0.5f : 0.f);
                    const float inr = (ratio >= 1.f - clip && ratio <= 1.f + clip) ? 1.f : 0.f;
                    const float dmin = w1 * adv + (1.f - w1) * adv * inr;
                    dlpS[r] = valid ? -inv_mb * dmin * ratio : 0.f;
                    if (valid) loss_act -= fminf(surr1, surr2);
                }
                __syncthreads();
            }
            PGM_TR(3)

            // ---------------- dz2 = dlp * (u . Wh) * (1 - h2^2) ----------------
            {
                u64 acc[TM][2];
#pragma unroll
                for (int i = 0; i < TM; ++i) acc[i][0] = acc[i][1] = 0ull;
                for (int aa = 0; aa < KH; ++aa) {
                    const ulonglong2 w = lds2x64(n.Wh + aa * LDH + 4 * tc);
#pragma unroll
                    for (int i = 0; i < TM; ++i) {
                        const float sv = ho[(tr + 16 * i) * ldo + aa];
                        acc[i][0] = ffma2_s(sv, w.x, acc[i][0]); acc[i][1] = ffma2_s(sv, w.y, acc[i][1]);
                    }
                }
#pragma unroll
                for (int i = 0; i < TM; ++i) {
                    const int r = tr + 16 * i;
                    const float sc = dlpS[r];
                    const float4 hv = lds4(h2 + r * LDH + 4 * tc);
                    const float2 a0 = unpack2(acc[i][0]), a1 = unpack2(acc[i][1]);
                    sts4(dz + r * LDH + 4 * tc,
                         make_float4(sc * a0.x * (1.f - hv.x * hv.x), sc * a0.y * (1.f - hv.y * hv.y),
                                     sc * a1.x * (1.f - hv.z * hv.z), sc * a1.y * (1.f - hv.w * hv.w)));
                }
            }
            __syncthreads();
            PGM_TR(4)

            // ---------------- dW2, db2, dz1 -> d1 ----------------
            {
                const int tj = tid & 15, tk = tid >> 4;
#pragma unroll 8
                for (int r = 0; r < RC; ++r) {
                    const float4 dv = lds4(dz + r * LDH + 4 * tj);
                    const ulonglong2 hv = lds2x64(h1 + r * LDH + 4 * tk);
                    gW2[0][0] = ffma2_s(dv.x, hv.x, gW2[0][0]); gW2[0][1] = ffma2_s(dv.x, hv.y, gW2[0][1]);
                    gW2[1][0] = ffma2_s(dv.y, hv.x, gW2[1][0]); gW2[1][1] = ffma2_s(dv.y, hv.y, gW2[1][1]);
                    gW2[2][0] = ffma2_s(dv.z, hv.x, gW2[2][0]); gW2[2][1] = ffma2_s(dv.z, hv.y, gW2[2][1]);
                    gW2[3][0] = ffma2_s(dv.w, hv.x, gW2[3][0]); gW2[3][1] = ffma2_s(dv.w, hv.y, gW2[3][1]);
                    if (tk == 0) { gb2[0] += dv.x; gb2[1] += dv.y; gb2[2] += dv.z; gb2[3] += dv.w; }
                }
                if (EP && c == nchunk - 1) {      // dW2 of this step is complete: its tiles go to the image now
                    const int oW2e = (int)(n.W2 - n.W1);
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj)
                        *reinterpret_cast<ulonglong2 *>(gP + oW2e + (4 * tj + jj) * LDH + 4 * tk) = make_ulonglong2(gW2[jj][0], gW2[jj][1]);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                }
                u64 acc[TM][2];
#pragma unroll
                for (int i = 0; i < TM; ++i) acc[i][0] = acc[i][1] = 0ull;
#pragma unroll(TM == 2 ? 4 : 2)
                for (int j = 0; j < H; j += 4) {
                    float4 av[TM];
                    ulonglong2 bv[4];
#pragma unroll
                    for (int i = 0; i < TM; ++i) av[i] = lds4(dz + (tr + 16 * i) * LDH + j);
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) bv[jj] = lds2x64(n.W2 + (j + jj) * LDH + 4 * tc);
#pragma unroll
                    for (int i = 0; i < TM; ++i) {
                        acc[i][0] = ffma2_s(av[i].x, bv[0].x, acc[i][0]); acc[i][1] = ffma2_s(av[i].x, bv[0].y, acc[i][1]);
                        acc[i][0] = ffma2_s(av[i].y, bv[1].x, acc[i][0]); acc[i][1] = ffma2_s(av[i].y, bv[1].y, acc[i][1]);
                        acc[i][0] = ffma2_s(av[i].z, bv[2].x, acc[i][0]); acc[i][1] = ffma2_s(av[i].z, bv[2].y, acc[i][1]);
                        acc[i][0] = ffma2_s(av[i].w, bv[3].x, acc[i][0]); acc[i][1] = ffma2_s(av[i].w, bv[3].y, acc[i][1]);
                    }
                }
#pragma unroll
                for (int i = 0; i < TM; ++i) {
                    const float4 hv = lds4(h1 + (tr + 16 * i) * LDH + 4 * tc);
                    const float2 a0 = unpack2(acc[i][0]), a1 = unpack2(acc[i][1]);
                    sts4(d1 + (tr + 16 * i) * LDH + 4 * tc,
                         make_float4(a0.x * (1.f - hv.x * hv.x), a0.y * (1.f - hv.y * hv.y),
                                     a1.x * (1.f - hv.z * hv.z), a1.y * (1.f - hv.w * hv.w)));
                }
            }
            __syncthreads();
            if (EP && c == nchunk - 1) {          // W2-only slices -> their owners' slots, under phase C and the image write
                if (tid == 0)
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                                 ::"r"(smem_u32(&mbarR)), "r"(G * 16 * (sl1 - sl0)) : "memory");
                if (tid < G) {
                    const int o0 = tid * per4, o1 = min(n4, o0 + per4);
                    const int w0 = (int)(n.W2 - n.W1) >> 2, w1 = (int)(n.b2 - n.W1) >> 2;
                    if (o1 > o0 && o0 >= w0 && o1 <= w1) {
                        const uint32_t dst = mapa_u32(smem_u32(slotB) + 16u * (uint32_t)(g * per4), (uint32_t)(half * G + tid));
                        const uint32_t mb = mapa_u32(smem_u32(&mbarR), (uint32_t)(half * G + tid));
                        asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                     ::"r"(dst), "r"(smem_u32(gP) + 16u * (uint32_t)o0), "r"(16 * (o1 - o0)), "r"(mb) : "memory");
                    }
                }
            }
            PGM_TR(5)

            // ---------------- phase C: dW1/db1 on slots [0, nW1), dWh/dbh/dls on the rest ----------------
            if (isW1) {
#pragma unroll 8
                for (int r = r1lo; r < r1hi; ++r) {
                    const float4 dv = lds4(d1 + r * LDH + 4 * l16);
                    const ulonglong2 xv = lds2x64(x + r * RSS + 4 * kg1);
                    gW1[0][0] = ffma2_s(dv.x, xv.x, gW1[0][0]); gW1[0][1] = ffma2_s(dv.x, xv.y, gW1[0][1]);
                    gW1[1][0] = ffma2_s(dv.y, xv.x, gW1[1][0]); gW1[1][1] = ffma2_s(dv.y, xv.y, gW1[1][1]);
                    gW1[2][0] = ffma2_s(dv.z, xv.x, gW1[2][0]); gW1[2][1] = ffma2_s(dv.z, xv.y, gW1[2][1]);
                    gW1[3][0] = ffma2_s(dv.w, xv.x, gW1[3][0]); gW1[3][1] = ffma2_s(dv.w, xv.y, gW1[3][1]);
                    if (kg1 == 0) { gb1[0] += dv.x; gb1[1] += dv.y; gb1[2] += dv.z; gb1[3] += dv.w; }
                }
            } else if (isWh) {
#pragma unroll
                for (int ia = 0; ia < 4; ++ia) {
                    const int aa = aslot + ia * fp.nA;
                    if (aa < KH) {
#pragma unroll 8
                        for (int r = rhlo; r < rhhi; ++r) {
                            const float sv = ho[r * ldo + aa] * dlpS[r];
                            const ulonglong2 hv = lds2x64(h2 + r * LDH + 4 * l16);
                            gWh[ia][0] = ffma2_s(sv, hv.x, gWh[ia][0]); gWh[ia][1] = ffma2_s(sv, hv.y, gWh[ia][1]);
                            if (l16 == 0) gbh[ia] += sv;
                            if (half == 0 && l16 == 1) gls[ia] = fmaf(els[r * ldo + aa], dlpS[r], gls[ia]);
                        }
                    }
                }
            }
            PGM_TR(6)
            // the next chunk's first barrier (or the combine barrier below) orders buffer reuse
        }

        // ---- combine row-split partials through the staging buffer ----
        {
            float *s1 = stg;                                         // [(nrs1-1)][H*OP + H]
            float *sH = stg + (fp.nrs1 - 1) * (H * OP + H);          // [(nrsH-1)][KH][H + 4]
            if (isW1 && rs1 > 0) {
                float *b = s1 + (rs1 - 1) * (H * OP + H);
#pragma unroll
                for (int jj = 0; jj < 4; ++jj)
                    *reinterpret_cast<ulonglong2 *>(b + (4 * l16 + jj) * OP + 4 * kg1) = make_ulonglong2(gW1[jj][0], gW1[jj][1]);
                if (kg1 == 0) sts4(b + H * OP + 4 * l16, make_float4(gb1[0], gb1[1], gb1[2], gb1[3]));
            }
            if (isWh && rsh > 0 && aslot < KH) {       // row splits only exist when nA >= KH (one pass)
                float *b = sH + ((rsh - 1) * KH + aslot) * (H + 4);
                *reinterpret_cast<ulonglong2 *>(b + 4 * l16) = make_ulonglong2(gWh[0][0], gWh[0][1]);
                if (l16 == 0) b[H] = gbh[0];
                if (l16 == 1) b[H + 1] = gls[0];
            }
            __syncthreads();
            if (isW1 && rs1 == 0) {
                for (int q = 1; q < fp.nrs1; ++q) {
                    const float *b = s1 + (q - 1) * (H * OP + H);
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const float4 t = lds4(b + (4 * l16 + jj) * OP + 4 * kg1);
                        const float2 c0 = unpack2(gW1[jj][0]), c1 = unpack2(gW1[jj][1]);
                        gW1[jj][0] = pack2(c0.x + t.x, c0.y + t.y); gW1[jj][1] = pack2(c1.x + t.z, c1.y + t.w);
                    }
                    if (kg1 == 0) { const float4 t = lds4(b + H * OP + 4 * l16); gb1[0] += t.x; gb1[1] += t.y; gb1[2] += t.z; gb1[3] += t.w; }
                }
            }
            if (isWh && rsh == 0 && aslot < KH) {
                for (int q = 1; q < fp.nrsH; ++q) {
                    const float *b = sH + ((q - 1) * KH + aslot) * (H + 4);
                    const float4 t = lds4(b + 4 * l16);
                    const float2 c0 = unpack2(gWh[0][0]), c1 = unpack2(gWh[0][1]);
                    gWh[0][0] = pack2(c0.x + t.x, c0.y + t.y); gWh[0][1] = pack2(c1.x + t.z, c1.y + t.w);
                    if (l16 == 0) gbh[0] += b[H];
                    if (l16 == 1) gls[0] += b[H + 1];
                }
            }
        }

        // ---- partial gradient of this CTA: RA = false -> its own smem image (peers read it through DSMEM);
        //      RA = true -> straight from registers into slot g of each piece's slice owner (st.shared::cluster) ----
        {
            const uint32_t gP_u = smem_u32(gP);
            auto emit16 = [&](int io, ulonglong2 v) {            // io: float offset in the image, multiple of 4
                if (RA) {
                    const uint32_t i4 = (uint32_t)io >> 2, ow = __umulhi(i4, magic);
                    const uint32_t loc = gP_u + 16u * ((uint32_t)g * (uint32_t)per4 + (i4 - ow * (uint32_t)per4));
                    st_dsmem2x64(mapa_u32(loc, (uint32_t)(half * G) + ow), v);
                } else if (GL) {
                    *reinterpret_cast<ulonglong2 *>(gPg + io) = v;
                } else {
                    *reinterpret_cast<ulonglong2 *>(gP + io) = v;
                }
            };
            auto emit1 = [&](int io, float v) {
                if (RA) {
                    const uint32_t ow = __umulhi((uint32_t)io >> 2, magic);
                    const uint32_t loc = gP_u + 4u * ((uint32_t)g * 4u * (uint32_t)per4 + ((uint32_t)io - 4u * ow * (uint32_t)per4));
                    st_dsmem1(mapa_u32(loc, (uint32_t)(half * G) + ow), v);
                } else if (GL) {
                    gPg[io] = v;
                } else {
                    gP[io] = v;
                }
            };
            const int tj = tid & 15, tk = tid >> 4;
            const int ob1 = (int)(n.b1 - n.W1), oW2 = (int)(n.W2 - n.W1), ob2 = (int)(n.b2 - n.W1);
            const int oWh = (int)(n.Wh - n.W1), obh = (int)(n.bh - n.W1), ols = (int)(n.ls - n.W1);
            if (!EP) {
#pragma unroll
                for (int jj = 0; jj < 4; ++jj)
                    emit16(oW2 + (4 * tj + jj) * LDH + 4 * tk, make_ulonglong2(gW2[jj][0], gW2[jj][1]));
            }
            if (tk == 0) emit16(ob2 + 4 * tj, make_ulonglong2(pack2(gb2[0], gb2[1]), pack2(gb2[2], gb2[3])));
            if (isW1 && rs1 == 0) {
#pragma unroll
                for (int jj = 0; jj < 4; ++jj)
                    emit16((4 * l16 + jj) * L.ldw1 + 4 * kg1, make_ulonglong2(gW1[jj][0], gW1[jj][1]));
                if (kg1 == 0) emit16(ob1 + 4 * l16, make_ulonglong2(pack2(gb1[0], gb1[1]), pack2(gb1[2], gb1[3])));
            }
            if (isWh && rsh == 0) {
#pragma unroll
                for (int ia = 0; ia < 4; ++ia) {
                    const int aa = aslot + ia * fp.nA;
                    if (aa < KH) {
                        emit16(oWh + aa * LDH + 4 * l16, make_ulonglong2(gWh[ia][0], gWh[ia][1]));
                        if (l16 == 0) emit1(obh + aa, gbh[ia]);
                        if (half == 0 && l16 == 1) emit1(ols + aa, gls[ia]);
                    }
                }
            }
        }
        if (half == 0 && g == 0 && tid == 0) {   // entropy with the parameters this step started from
            float ent = 0.f;
            for (int d = 0; d < A; ++d) ent += 0.5f + 0.91893853320467274178f + n.ls[d];
            loss_ent += ent;
        }
        PGM_TR(7)
        if (BP) {
            // my partial image -> the per-source slot of every slice owner, by the bulk-copy engine; no barrier (1)
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // my st.shared, before the async proxy reads them
            __syncthreads();
            if (!EP && tid == 0)
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                             ::"r"(smem_u32(&mbarR)), "r"(G * 16 * (sl1 - sl0)) : "memory");
            if (tid < G) {
                const int o0 = tid * per4, o1 = min(n4, o0 + per4);
                const int w0 = (int)(n.W2 - n.W1) >> 2, w1 = (int)(n.b2 - n.W1) >> 2;
                if (o1 > o0 && !(EP && o0 >= w0 && o1 <= w1)) {      // (TAIL = 6: the W2-only slices left after phase B)
                    const uint32_t dst = mapa_u32(smem_u32(slotB) + 16u * (uint32_t)(g * per4), (uint32_t)(half * G + tid));
                    const uint32_t mb = mapa_u32(smem_u32(&mbarR), (uint32_t)(half * G + tid));
                    asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                 ::"r"(dst), "r"(smem_u32(gP) + 16u * (uint32_t)o0), "r"(16 * (o1 - o0)), "r"(mb) : "memory");
                }
            }
            uint32_t done = 0;      // the G partial slices of my slice have landed in my slots
            while (!done)
                asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                             : "=r"(done) : "r"(smem_u32(&mbarR)), "r"(s & 1) : "memory");
        } else {
            sync_group<C>();   // (1) every CTA's partial gradient image is complete
        }
        PGM_TR(8)

        // ---- reduce my slice over the G CTAs of my half (fixed order), squared-norm partial ----
        {
            const uint32_t gP_u = smem_u32(gP);
            uint32_t peer[G];
#pragma unroll
            for (int gg = 0; gg < G; ++gg) peer[gg] = mapa_u32(RA ? smem_u32(gS) : gP_u, (uint32_t)(half * G + gg));
            const int ls4 = (int)(n.ls - n.W1) >> 2;
            float sq = 0.f;
            for (int i4 = sl0 + tid; i4 < sl1; i4 += NTHREADS) {
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int gg = 0; gg < G; ++gg) {
                    // RA: slot gg of my slice (local, filled by CTA gg of my half); else CTA gg's image through DSMEM
                    const float4 t = RA ? lds4(gP + 4 * (gg * per4 + (i4 - sl0)))
                                   : BP ? lds4(slotB + 4 * (gg * per4 + (i4 - sl0)))
                                   : (GL ? __ldcg(reinterpret_cast<const float4 *>(a.gpart + ((size_t)(task * 2 + half) * G + gg) * a.NHP) + i4)
                                         : ld_dsmem4(peer[gg] + 16u * (uint32_t)i4));
                    acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
                }
                if (ecoef != 0.f && half == 0 && i4 >= ls4) {   // d(-ecoef * entropy)/d logstd
                    const int e0 = 4 * (i4 - ls4);
                    if (e0 + 0 < A) acc.x -= ecoef;
                    if (e0 + 1 < A) acc.y -= ecoef;
                    if (e0 + 2 < A) acc.z -= ecoef;
                    if (e0 + 3 < A) acc.w -= ecoef;
                }
                sq = fmaf(acc.x, acc.x, sq); sq = fmaf(acc.y, acc.y, sq);
                sq = fmaf(acc.z, acc.z, sq); sq = fmaf(acc.w, acc.w, sq);
                if (RA) {
#pragma unroll
                    for (int gg = 0; gg < G; ++gg) st_dsmem4(peer[gg] + 16u * (uint32_t)i4, acc);   // reduced slice -> every CTA of the half
                } else {
                    sts4(gS + 4 * (i4 - sl0), acc);
                }
            }
            sq = block_sum(sq, red);
            PGM_TR(9)
            if (NB) {       // my partial -> every CTA's slot, signalling that CTA's mbarrier (4 bytes each)
                if (tid == 0)
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&mbarN)), "r"(4 * C) : "memory");
                if (tid < C)
                    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];"
                                 ::"r"(mapa_u32(smem_u32(ssqS + rank), (uint32_t)tid)), "r"(__float_as_uint(sq)),
                                   "r"(mapa_u32(smem_u32(&mbarN), (uint32_t)tid)) : "memory");
            } else if (tid < C) {
                st_dsmem1(mapa_u32(smem_u32(ssqS + rank), (uint32_t)tid), sq);   // my partial -> every CTA
            }
        }
        if (a.grad_only) {
            if (NB) {               // every st.async aimed at this CTA must have landed before it may exit
                uint32_t done = 0;
                while (!done)
                    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                                 : "=r"(done) : "r"(smem_u32(&mbarN)), "r"(s & 1) : "memory");
            }
            sync_group<C>();
            const int nH = L.half_size(half);
            for (int e = tid; e < nH; e += NTHREADS) {
                const int io = half_img_off(n, L, e);
                if (io >= 4 * sl0 && io < 4 * sl1)
                    a.grad_out[(size_t)task * L.n_par + L.to_global(half, e)] = gS[io - (RA ? 0 : 4 * sl0)];
            }
            break;
        }
        if (tid == 0) {   // Adam scalars of step k = step0 + s + 1, in double
            b1pow *= a.hy.beta1; b2pow *= a.hy.beta2;
            sh_d[0] = lr / (1.0 - b1pow);            // step_size
            sh_d[1] = 1.0 / sqrt(1.0 - b2pow);       // 1 / bias_correction2_sqrt
        }
        if (NB) {
            __syncthreads();        // sh_d (Adam scalars) written by thread 0
            uint32_t done = 0;      // all C squared-norm partials have landed in ssqS
            while (!done)
                asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                             : "=r"(done) : "r"(smem_u32(&mbarN)), "r"(s & 1) : "memory");
        } else {
            sync_group<C>();   // (2) all squared-norm partials have landed in ssqS
        }
        PGM_TR(10)
        {
            float tot = 0.f;
#pragma unroll
            for (int rr = 0; rr < C; ++rr) tot += ssqS[rr];
            const float coef = fminf(1.f, (float)a.hy.max_grad_norm / (sqrtf(tot) + 1e-6f));
            const float step_size = (float)sh_d[0], ibc2 = (float)sh_d[1];
            float *pimg = n.W1;
#define PGM_ADAM1(cc)                                                                                  \
                {                                                                                      \
                    const float gr = g4.cc * coef;                                                     \
                    m4.cc = fmaf(gr - m4.cc, omb1, m4.cc);          /* exp_avg.lerp_(grad, 1 - beta1) */ \
                    v4.cc = fmaf(omb2 * gr, gr, v4.cc * b2f);       /* exp_avg_sq.mul_(b2).addcmul_() */ \
                    const float denom = fmaf(fast_sqrt(v4.cc), ibc2, aeps);                            \
                    p4.cc -= step_size * __fdividef(m4.cc, denom);                                     \
                }
            if (RA) {   // the whole half, redundantly in every CTA of the half: nothing to publish, no third barrier
                for (int i4 = tid; i4 < n4; i4 += NTHREADS) {
                    const float4 g4 = lds4(gS + 4 * i4);
                    float4 m4 = lds4(mS + 4 * i4), v4 = lds4(vS + 4 * i4), p4 = lds4(pimg + 4 * i4);
                    PGM_ADAM1(x) PGM_ADAM1(y) PGM_ADAM1(z) PGM_ADAM1(w)
                    sts4(mS + 4 * i4, m4); sts4(vS + 4 * i4, v4); sts4(pimg + 4 * i4, p4);
                }
                // the next step's first __syncthreads orders these writes before any read of the parameters
            } else {
                const uint32_t pimg_u = smem_u32(pimg);
                uint32_t peer[G];
#pragma unroll
                for (int gg = 0; gg < G; ++gg) peer[gg] = mapa_u32(pimg_u, (uint32_t)(half * G + gg));
                float *pst = a.pstage + (size_t)(task * 2 + half) * a.NHP;      // TAIL >= 2: L2-resident staging row of the half
                for (int i4 = sl0 + tid; i4 < sl1; i4 += NTHREADS) {
                    const int j4 = i4 - sl0;
                    const float4 g4 = lds4(gS + 4 * j4);
                    float4 m4 = lds4(mS + 4 * j4), v4 = lds4(vS + 4 * j4), p4 = lds4(pimg + 4 * i4);
                    PGM_ADAM1(x) PGM_ADAM1(y) PGM_ADAM1(z) PGM_ADAM1(w)
                    sts4(mS + 4 * j4, m4); sts4(vS + 4 * j4, v4);
                    if (MC) {
                        *reinterpret_cast<float4 *>(pst + 4 * i4) = p4;
                    } else {
#pragma unroll
                        for (int gg = 0; gg < G; ++gg) st_dsmem4(peer[gg] + 16u * (uint32_t)i4, p4);   // incl. my own image
                    }
                }
                if (MC) {
                    asm volatile("fence.proxy.async.global;" ::: "memory");     // my stores, before the async proxy reads them
                    __syncthreads();
                    if (tid == 0) {
                        const uint32_t mb = smem_u32(&mbarS);
                        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(16 * n4) : "memory");
                        if (sl1 > sl0) {
                            const unsigned short mask = (unsigned short)(((1u << G) - 1u) << (half * G));
                            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster "
                                         "[%0], [%1], %2, [%3], %4;"
                                         ::"r"(pimg_u + 16u * (uint32_t)sl0), "l"(pst + 4 * sl0), "r"(16 * (sl1 - sl0)), "r"(mb), "h"(mask)
                                         : "memory");
                        }
                    }
                    uint32_t done = 0;      // all G slices of my half have landed in my resident image
                    while (!done)
                        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                                     : "=r"(done) : "r"(smem_u32(&mbarS)), "r"(s & 1) : "memory");
                }
            }
#undef PGM_ADAM1
        }
        if (!RA && !MC) sync_group<C>();   // (3) every resident image holds the new parameters
        PGM_TR(11)
    }

    if (!a.grad_only) {   // final state back to global memory (reference order); moments by slice owner
        const int nH = L.half_size(half);
        for (int e = tid; e < nH; e += NTHREADS) {
            const size_t gi = (size_t)task * L.n_par + L.to_global(half, e);
            const int io = half_img_off(n, L, e);
            if (g == 0) a.params[gi] = n.W1[io];
            if (RA ? g == 0 : (io >= 4 * sl0 && io < 4 * sl1)) {
                a.adam_m[gi] = mS[io - (RA ? 0 : 4 * sl0)];
                a.adam_v[gi] = vS[io - (RA ? 0 : 4 * sl0)];
            }
        }
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
            a.losses[task * 3 + 2] = se / ns;
            if (!a.grad_only) a.adam_step[task] = step0 + a.nsteps;
        }
    }
}

__host__ inline size_t k3_fast_smem_bytes(const NetLayout &L, int TM, int RSS, int NHP, int stage_floats, int G, bool ra, bool gl = false,
                                          bool bp = false) {
    const int RC = 16 * TM;
    const int ldo = ((L.A > L.M ? L.A : L.M) | 1);
    const int img = halfnet_smem_floats(L, 0) > halfnet_smem_floats(L, 1) ? halfnet_smem_floats(L, 0) : halfnet_smem_floats(L, 1);
    // image + activations + loss arrays + staging + records + partial-gradient image + slice buffers (G >= 1)
    const size_t per = 4 * (size_t)((img / 4 + G - 1) / G);
    size_t f = img + 4 * (size_t)RC * LDH + 3 * (size_t)round_up(RC * ldo, 4) + RC + round_up(stage_floats, 4) +
               2 * (size_t)RC * RSS + (ra ? 2 * G * per + 2 * (size_t)img : (gl ? 0 : (size_t)NHP) + 3 * per + (bp ? G * per : 0));
    return f * sizeof(float);
}

}  // namespace pgm
