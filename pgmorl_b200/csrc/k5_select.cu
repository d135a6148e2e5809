// K5 -- Pareto filtering, exact 2-D / 3-D hypervolume, sparsity and the greedy candidate pick of the
// prediction-guided selection, in FLOAT64 and bit-exact with the reference.
//
// Replaces (paths relative to the reference's morl/):
//   utils.get_ep_indices / check_dominated   utils.py:24-39      -> k5_dominance / k5_rank kernels
//   utils.update_ep                          utils.py:42-65      -> device fn update_front_3d
//   Population.compute_hypervolume/sparsity  population_2d.py:185-202 -> score_2d
//   InnerHyperVolume (3 objectives)          hypervolume.py:41-153    -> k5_score3d_kernel
//   utils.compute_sparsity                   utils.py:87-100          -> k5_score3d_kernel
//   evaluate_hv / evaluate_sparsity / greedy loop  population_2d.py:207-224,264-302,
//                                                  population_3d.py:206-214,294-331
//
// Bit-exactness: every sum is accumulated in the reference's order with separate IEEE multiply and
// add (__dmul_rn / __dadd_rn: no FMA contraction), so hv, sparsity and therefore every arg-max agree
// with the CPU reference to the last bit. Parallelism comes from the candidates (one thread per
// candidate in 2-D, one CTA per candidate in 3-D with one thread per z-slice), never from
// re-associating a sum.
#include <climits>

#include "common.cuh"

namespace pgm {

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }

// Python round(x, 4) for x >= 0: correctly rounded decimal rounding (ties to even), as float.__round__.
__device__ inline double round4(double x) {
    const double t = x * 10000.0;
    if (!(fabs(t) < 4.0e15)) return x;                 // already an integer multiple at this magnitude
    double r0 = floor(t);
    // sign of the exact x*1e4 - (r0 + 0.5): one rounding in fma, so the sign is exact unless it is a true tie
    double e = fma(x, 10000.0, -(r0 + 0.5));
    if (e < -1.0) { r0 -= 1.0; e = fma(x, 10000.0, -(r0 + 0.5)); }      // t was rounded up across an integer
    else if (e >= 1.0) { r0 += 1.0; e = fma(x, 10000.0, -(r0 + 0.5)); }
    double r;
    if (e > 0.0) r = r0 + 1.0;
    else if (e < 0.0) r = r0;
    else r = (fmod(r0, 2.0) == 0.0) ? r0 : r0 + 1.0;
    return r / 10000.0;
}

// ------------------------------------------------------------------------------------------------
// get_ep_indices
// ------------------------------------------------------------------------------------------------
template <int M>
__global__ void k5_dominance_kernel(const double *__restrict__ objs, int n, int *__restrict__ kept) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    __shared__ double tile[256 * M];
    double p[M];
    bool valid = i < n;
    if (valid)
        for (int m = 0; m < M; ++m) { p[m] = objs[(size_t)i * M + m]; }
    bool nonneg = valid, dominated = false;
    if (valid)
        for (int m = 0; m < M; ++m) nonneg = nonneg && (p[m] >= 0.0);
    for (int j0 = 0; j0 < n; j0 += 256) {
        const int nj = min(256, n - j0);
        __syncthreads();
        for (int t = threadIdx.x; t < nj * M; t += blockDim.x) tile[t] = objs[(size_t)j0 * M + t];
        __syncthreads();
        if (valid && !dominated)
            for (int j = 0; j < nj; ++j) {
                bool ge = true, gt = false;
                for (int m = 0; m < M; ++m) { const double q = tile[j * M + m]; ge = ge && (q >= p[m]); gt = gt || (q > p[m]); }
                if (ge && gt) { dominated = true; break; }
            }
    }
    if (valid) kept[i] = (nonneg && !dominated) ? 1 : 0;
}

template <int M>
__global__ void k5_rank_kernel(const double *__restrict__ objs, int n, const int *__restrict__ kept,
                               int32_t *__restrict__ keep_idx, int32_t *__restrict__ n_keep) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !kept[i]) return;
    const double x = objs[(size_t)i * M];
    int rank = 0;
    for (int j = 0; j < n; ++j) {
        if (!kept[j]) continue;
        const double xj = objs[(size_t)j * M];
        rank += (xj < x || (xj == x && j < i)) ? 1 : 0;
    }
    keep_idx[rank] = i;
    atomicAdd(n_keep, 1);
}

// ------------------------------------------------------------------------------------------------
// selection state in the workspace
// ------------------------------------------------------------------------------------------------
// What the 3-objective scorer needs of the round's base front and every candidate shares (built once per round by
// base3d_build): negated coordinates in front order, the three sorted lists of preProcess and the z ranks, the slice
// areas, and the hypervolume chain after every term.
struct Base3d {
    double *nx, *ny, *nz;     // [nmax]
    double *area;             // [nmax] 2-D area of the first k+1 points of the z list
    double *vpre;             // [nmax] vpre[k] = sum of the terms 1..k of the hypervolume chain (vpre[0] = 0)
    int *xl, *yl, *zl, *zr;   // [nmax] sorted lists (positions in the front) and z rank of every point
};

struct SelState {
    double *front[2];   // virtual EP, double buffered [Emax][M]
    int *count;         // [2] sizes of front[0] / front[1]
    int *mask;          // [C] 1 = candidate still available
    int *done;          // [1] set when a round found no candidate
    Base3d b3;          // 3 objectives only
};

// ---- 2 objectives: one thread per candidate -------------------------------------------------------
// hv / sparsity of get_ep_indices(front + {p}) with front sorted by x and mutually non-dominated.
__device__ inline void score_2d(const double *__restrict__ f, int n, double px, double py, bool has_p, double &hv_out,
                                double &sp_out) {
    bool p_ok = has_p && px >= 0.0 && py >= 0.0;
    if (p_ok)
        for (int i = 0; i < n; ++i) {
            const double qx = f[2 * i], qy = f[2 * i + 1];
            if (qx >= px && qy >= py && (qx > px || qy > py)) { p_ok = false; break; }
        }
    double hv = 0.0, xprev = 0.0, sp = 0.0, lx = 0.0, ly = 0.0;
    int cnt = 0;
    bool p_done = !p_ok;
    auto emit = [&](double x, double y) {
        hv = dadd(hv, dmul(dsub(fmax(0.0, x), xprev), dsub(fmax(0.0, y), 0.0)));
        xprev = fmax(0.0, x);
        if (cnt > 0) {
            const double dx = dsub(x, lx), dy = dsub(y, ly);
            sp = dadd(sp, dadd(dmul(dx, dx), dmul(dy, dy)));
        }
        lx = x; ly = y; ++cnt;
    };
    for (int i = 0; i < n; ++i) {
        const double qx = f[2 * i], qy = f[2 * i + 1];
        if (!p_done && qx > px) { emit(px, py); p_done = true; }
        const bool dom = p_ok && px >= qx && py >= qy && (px > qx || py > qy);
        if (!dom) emit(qx, qy);
    }
    if (!p_done) emit(px, py);
    hv_out = hv;
    sp_out = cnt < 2 ? 0.0 : sp / (double)(cnt - 1);
}

__global__ void k5_score2d_kernel(SelState st, int buf, const double *__restrict__ cand, int C,
                                  double *__restrict__ hv, double *__restrict__ sp) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double h = 0.0, s = 0.0;
    if (!*st.done && st.mask[c]) score_2d(st.front[buf], st.count[buf], cand[2 * c], cand[2 * c + 1], true, h, s);
    hv[c] = h; sp[c] = s;
}

// new front = get_ep_indices(front + {p}) (population_2d.py:298-300); single thread
__device__ inline int update_front_2d(const double *__restrict__ f, int n, double px, double py, double *__restrict__ out) {
    bool p_ok = px >= 0.0 && py >= 0.0;
    if (p_ok)
        for (int i = 0; i < n; ++i) {
            const double qx = f[2 * i], qy = f[2 * i + 1];
            if (qx >= px && qy >= py && (qx > px || qy > py)) { p_ok = false; break; }
        }
    int m = 0;
    bool p_done = !p_ok;
    for (int i = 0; i < n; ++i) {
        const double qx = f[2 * i], qy = f[2 * i + 1];
        if (!p_done && qx > px) { out[2 * m] = px; out[2 * m + 1] = py; ++m; p_done = true; }
        const bool dom = p_ok && px >= qx && py >= qy && (px > qx || py > qy);
        if (!dom) { out[2 * m] = qx; out[2 * m + 1] = qy; ++m; }
    }
    if (!p_done) { out[2 * m] = px; out[2 * m + 1] = py; ++m; }
    return m;
}

// ---- 3 objectives -----------------------------------------------------------------------------
// update_ep (utils.py:42-65), single thread; returns the new size
__device__ inline int update_front_3d(const double *__restrict__ f, int n, const double *p, double *__restrict__ out) {
    if (p[0] < 0.0 || p[1] < 0.0 || p[2] < 0.0) {
        for (int i = 0; i < 3 * n; ++i) out[i] = f[i];
        return n;
    }
    bool on_ep = true;
    int m = 0;
    for (int i = 0; i < n; ++i) {
        const double *q = f + 3 * i;
        const bool dominated = p[0] >= q[0] && p[1] >= q[1] && p[2] >= q[2];
        if (q[0] >= p[0] - 1e-5 && q[1] >= p[1] - 1e-5 && q[2] >= p[2] - 1e-5 &&
            (q[0] > p[0] + 1e-5 || q[1] > p[1] + 1e-5 || q[2] > p[2] + 1e-5))
            on_ep = false;
        if (!dominated) { out[3 * m] = q[0]; out[3 * m + 1] = q[1]; out[3 * m + 2] = q[2]; ++m; }
    }
    if (on_ep) {
        int pos = m;
        for (int i = 0; i < m; ++i)
            if (p[0] < out[3 * i]) { pos = i; break; }
        for (int i = m; i > pos; --i) { out[3 * i] = out[3 * i - 3]; out[3 * i + 1] = out[3 * i - 2]; out[3 * i + 2] = out[3 * i - 1]; }
        out[3 * pos] = p[0]; out[3 * pos + 1] = p[1]; out[3 * pos + 2] = p[2];
        ++m;
    }
    return m;
}

// One CTA per candidate: L = update_ep(front, p); hv = round4(InnerHyperVolume(L)); sp = compute_sparsity(L).
// Dynamic smem: nx, ny, nz [nmax] doubles (negated coords, input order of L); area [nmax] doubles;
// xl, yl, zl [nmax] ints (sorted lists); zr [nmax] ints (z rank); keep/pos scratch [nmax] ints.
__global__ void __launch_bounds__(256) k5_score3d_kernel(SelState st, int buf, const double *__restrict__ cand, int C,
                                                         double *__restrict__ hv, double *__restrict__ sp, int nmax,
                                                         int use_cand) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const int c = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    if (use_cand) {
        if (*st.done || !st.mask[c]) {
            if (tid == 0) { hv[c] = 0.0; sp[c] = 0.0; }
            return;
        }
    }
    double *nx = reinterpret_cast<double *>(smraw), *ny = nx + nmax, *nz = ny + nmax, *area = nz + nmax;
    int *xl = reinterpret_cast<int *>(area + nmax), *yl = xl + nmax, *zl = yl + nmax, *zr = zl + nmax, *pos = zr + nmax;
    __shared__ int s_on_ep, s_n, s_ins;

    const double *f = st.front[buf];
    const int n0 = st.count[buf];
    double p[3] = {0.0, 0.0, 0.0};
    bool p_valid = false;
    if (use_cand) {
        p[0] = cand[3 * c]; p[1] = cand[3 * c + 1]; p[2] = cand[3 * c + 2];
        p_valid = p[0] >= 0.0 && p[1] >= 0.0 && p[2] >= 0.0;
    }
    if (tid == 0) { s_on_ep = 1; s_ins = 0; }
    __syncthreads();
    // ---- update_ep: keep flags (pos[i] = 1 if kept), on_ep, insertion index ----
    for (int i = tid; i < n0; i += nt) {
        const double *q = f + 3 * i;
        bool keep = true;
        if (p_valid) {
            keep = !(p[0] >= q[0] && p[1] >= q[1] && p[2] >= q[2]);
            if (q[0] >= p[0] - 1e-5 && q[1] >= p[1] - 1e-5 && q[2] >= p[2] - 1e-5 &&
                (q[0] > p[0] + 1e-5 || q[1] > p[1] + 1e-5 || q[2] > p[2] + 1e-5))
                s_on_ep = 0;                                     // benign race: every writer stores 0
        }
        pos[i] = keep ? 1 : 0;
    }
    __syncthreads();
    if (tid == 0) {       // exclusive scan of the keep flags + insertion point (n0 <= ~2k: negligible)
        const bool ins = p_valid && s_on_ep;
        int m = 0, ip = -1;
        for (int i = 0; i < n0; ++i) {
            const int k = pos[i];
            if (k) {
                if (ins && ip < 0 && p[0] < f[3 * i]) { ip = m; ++m; }   // p goes before the first kept q with p0 < q0
                pos[i] = m; ++m;
            } else pos[i] = -1;
        }
        if (ins && ip < 0) { ip = m; ++m; }
        s_n = m; s_ins = ins ? ip : -1;
    }
    __syncthreads();
    const int n = s_n, ins = s_ins;
    for (int i = tid; i < n0; i += nt)
        if (pos[i] >= 0) { nx[pos[i]] = -f[3 * i]; ny[pos[i]] = -f[3 * i + 1]; nz[pos[i]] = -f[3 * i + 2]; }
    if (tid == 0 && ins >= 0) { nx[ins] = -p[0]; ny[ins] = -p[1]; nz[ins] = -p[2]; }
    __syncthreads();
    if (n == 0) {
        if (tid == 0) { hv[c] = 0.0; sp[c] = 0.0; }
        return;
    }
    // ---- the three sorted lists of preProcess (hypervolume.py:156-164): successive stable sorts by x, y, z ----
    for (int i = tid; i < n; i += nt) {
        const double xi = nx[i], yi = ny[i], zi = nz[i];
        int rx = 0, ry = 0, rz = 0;
        for (int j = 0; j < n; ++j) {
            const double xj = nx[j], yj = ny[j], zj = nz[j];
            const bool xlt = xj < xi || (xj == xi && j < i);                    // key (x, input position)
            const bool ylt = yj < yi || (yj == yi && xlt);                       // key (y, x, input position)
            const bool zlt = zj < zi || (zj == zi && ylt);                       // key (z, y, x, input position)
            rx += xlt; ry += ylt; rz += zlt;
        }
        xl[rx] = i; yl[ry] = i; zl[rz] = i; zr[i] = rz;
    }
    __syncthreads();
    // ---- slice k: 2-D area of the first k+1 points of the z list, walked in y-list order (hypervolume.py:92-105) ----
    for (int k = tid; k < n; k += nt) {
        double h = 0.0, acc = 0.0, prevy = 0.0;
        bool first = true;
        for (int t = 0; t < n; ++t) {
            const int j = yl[t];
            if (zr[j] > k) continue;
            if (first) { h = nx[j]; prevy = ny[j]; first = false; }
            else {
                acc = dadd(acc, dmul(h, dsub(prevy, ny[j])));
                if (nx[j] < h) h = nx[j];
                prevy = ny[j];
            }
        }
        area[k] = dadd(acc, dmul(h, prevy));
    }
    __syncthreads();
    if (tid == 0) {
        double v = 0.0;
        for (int k = 1; k < n; ++k) v = dadd(v, dmul(area[k - 1], dsub(nz[zl[k]], nz[zl[k - 1]])));
        v = dsub(v, dmul(area[n - 1], nz[zl[n - 1]]));
        hv[c] = round4(v);
    } else if (tid == 32) {
        // utils.compute_sparsity: per dim ascending values (= the negated lists read backwards)
        double s = 0.0;
        if (n >= 2) {
            for (int d = 0; d < 3; ++d) {
                const int *lst = d == 0 ? xl : (d == 1 ? yl : zl);
                const double *v = d == 0 ? nx : (d == 1 ? ny : nz);
                for (int i = 1; i < n; ++i) {
                    const double g = dsub(-v[lst[n - 1 - i]], -v[lst[n - i]]);
                    s = dadd(s, dmul(g, g));
                }
            }
            s = s / (double)(n - 1);
        }
        sp[c] = s;
    }
}

// ---- 3 objectives, incremental: every candidate of a round extends the SAME base front ---------------------------
// In-place exclusive prefix sum of a[0..n) in shared memory; returns the total. Every thread of the CTA calls it.
__device__ __forceinline__ int block_excl_scan(int *a, int n, int *wtot) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    const int per = (n + nt - 1) / nt, lo = min(n, tid * per), hi = min(n, lo + per);
    int local = 0;
    for (int i = lo; i < hi; ++i) local += a[i];
    int inc = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) wtot[warp] = inc;
    __syncthreads();
    int off = 0, total = 0;
    for (int w = 0; w < nw; ++w) { const int v = wtot[w]; if (w < warp) off += v; total += v; }
    int run = off + inc - local;
    for (int i = lo; i < hi; ++i) { const int v = a[i]; a[i] = run; run += v; }
    __syncthreads();
    return total;
}

// 2-D area of the points with z rank <= k, walked in y-list order (hypervolume.py:92-105). The points come in y-list
// order already (hx[t], hy[t] = x, y of the t-th point of the y list, hz[t] = its z rank): every load is independent of
// the running sums, and all threads of a warp (one slice each) read the same t -- shared-memory broadcasts.
__device__ __forceinline__ double slice_area(const double *hx, const double *hy, const int *hz, int n, int k) {
    double h = 0.0, acc = 0.0, prevy = 0.0;
    bool first = true;
#pragma unroll 4
    for (int t = 0; t < n; ++t) {
        const double x = hx[t], y = hy[t];
        if (hz[t] > k) continue;
        if (first) { h = x; prevy = y; first = false; }
        else {
            acc = dadd(acc, dmul(h, dsub(prevy, y)));
            if (x < h) h = x;
            prevy = y;
        }
    }
    return dadd(acc, dmul(h, prevy));
}

// Base data of front f (n0 points) for the incremental scorer; all threads of ONE CTA.
// Dynamic shared memory: 5 * nmax doubles + nmax ints (coordinates; the points in y-list order).
static size_t base3d_smem(int nmax) { return (size_t)nmax * (5 * sizeof(double) + sizeof(int)); }
__device__ inline void base3d_build(const double *f, int n0, int nmax, Base3d b, unsigned char *smem) {
    const int tid = threadIdx.x, nt = blockDim.x;
    double *sx = reinterpret_cast<double *>(smem), *sy = sx + nmax, *sz = sy + nmax, *hx = sz + nmax, *hy = hx + nmax;
    int *hz = reinterpret_cast<int *>(hy + nmax);
    for (int i = tid; i < n0; i += nt) {
        const double x = -f[3 * i], y = -f[3 * i + 1], z = -f[3 * i + 2];
        sx[i] = x; sy[i] = y; sz[i] = z;
        b.nx[i] = x; b.ny[i] = y; b.nz[i] = z;
    }
    if (tid == 0) b.vpre[0] = 0.0;
    __syncthreads();
    // the three sorted lists of preProcess (hypervolume.py:156-164): successive stable sorts by x, y, z
    for (int i = tid; i < n0; i += nt) {
        const double xi = sx[i], yi = sy[i], zi = sz[i];
        int rx = 0, ry = 0, rz = 0;
#pragma unroll 4
        for (int j = 0; j < n0; ++j) {
            const double xj = sx[j], yj = sy[j], zj = sz[j];
            const bool xlt = xj < xi || (xj == xi && j < i);
            const bool ylt = yj < yi || (yj == yi && xlt);
            const bool zlt = zj < zi || (zj == zi && ylt);
            rx += xlt; ry += ylt; rz += zlt;
        }
        b.xl[rx] = i; b.yl[ry] = i; b.zl[rz] = i; b.zr[i] = rz;
        hx[ry] = xi; hy[ry] = yi; hz[ry] = rz;
    }
    __syncthreads();
    for (int k = tid; k < n0; k += nt) b.area[k] = slice_area(hx, hy, hz, n0, k);
    __syncthreads();
    for (int k = 1 + tid; k < n0; k += nt) b.vpre[k] = dmul(b.area[k - 1], dsub(sz[b.zl[k]], sz[b.zl[k - 1]]));
    __syncthreads();
    if (tid == 0) {
        double v = 0.0;
#pragma unroll 8
        for (int k = 1; k < n0; ++k) { v = dadd(v, b.vpre[k]); b.vpre[k] = v; }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(1024) k5_base3d_kernel(SelState st, int buf, int nmax) {
    extern __shared__ __align__(16) unsigned char base_smem[];
    base3d_build(st.front[buf], st.count[buf], nmax, st.b3, base_smem);
}

// One CTA per candidate p: L = update_ep(front, p); hv = round4(InnerHyperVolume(L)); sp = compute_sparsity(L) -- the same
// numbers as k5_score3d_kernel, bit for bit, without redoing what L shares with the base front:
//  * the sorted lists of L are the base lists with the points p dominates filtered out (prefix sums of the keep flags
//    along each list) and p slotted in at its rank (one comparison per point; ties broken by the position update_ep gives p);
//  * the slices below n_same = min(z rank of p, lowest z rank of a removed point) contain exactly the base points in the base
//    order, so their areas and the head of the hypervolume chain are the base's; only the slices from n_same on are walked;
//  * warps 0-7 walk slices while warp 8 forms the sparsity terms and runs that serial sum.
// Points are named by id: position in the base front, or n0 for p.
// The body scores candidate c with its arrays carved from `smraw` (score3d_inc_smem(nmax) bytes): shared memory in
// k5_score3d_inc_kernel, a per-CTA slice of global memory in k5g_score3d_inc_kernel.
constexpr int S3_WORKERS = 256, S3_THREADS = 288;
__device__ __forceinline__ void score3d_inc_body(const SelState &st, int buf, const double *__restrict__ cand, int c,
                                                 double *__restrict__ hv, double *__restrict__ sp, int nmax,
                                                 unsigned char *smraw) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
    if (*st.done || !st.mask[c]) {
        if (tid == 0) { hv[c] = 0.0; sp[c] = 0.0; }
        return;
    }
    double *cx = reinterpret_cast<double *>(smraw), *cy = cx + nmax, *cz = cy + nmax, *area = cz + nmax, *term = area + nmax;
    double *gsq = term + nmax, *hy = gsq + 3 * nmax;                       // gsq [3 * nmax]
    double *hx = term;                                                     // the slice walk is over before `term` is formed
    int *km = reinterpret_cast<int *>(hy + nmax), *tmp = km + nmax, *xl = tmp + nmax, *yl = xl + nmax, *zl = yl + nmax,
        *zr = zl + nmax;
    int *hz = tmp;                                                         // the scans are over before the slice walk
    unsigned char *rel = reinterpret_cast<unsigned char *>(zr + nmax);      // bit 0/1/2: point precedes p in the x/y/z list; bit 3: kept
    __shared__ int s_on_ep, s_ip, s_rp[3], s_zmin, wtot[S3_THREADS / 32];

    const Base3d b = st.b3;
    const int n0 = st.count[buf];
    const double p0 = cand[3 * c], p1 = cand[3 * c + 1], p2 = cand[3 * c + 2];
    const bool p_valid = p0 >= 0.0 && p1 >= 0.0 && p2 >= 0.0;
    for (int i = tid; i < n0; i += nt) { cx[i] = b.nx[i]; cy[i] = b.ny[i]; cz[i] = b.nz[i]; }
    if (tid == 0) {
        cx[n0] = -p0; cy[n0] = -p1; cz[n0] = -p2;
        s_on_ep = 1; s_ip = INT_MAX; s_rp[0] = s_rp[1] = s_rp[2] = 0; s_zmin = INT_MAX;
    }
    __syncthreads();
    // ---- update_ep (utils.py:42-65): keep flags, on_ep ----
    for (int i = tid; i < n0; i += nt) {
        const double q0 = -cx[i], q1 = -cy[i], q2 = -cz[i];
        bool keep = true;
        if (p_valid) {
            keep = !(p0 >= q0 && p1 >= q1 && p2 >= q2);
            if (q0 >= p0 - 1e-5 && q1 >= p1 - 1e-5 && q2 >= p2 - 1e-5 && (q0 > p0 + 1e-5 || q1 > p1 + 1e-5 || q2 > p2 + 1e-5))
                s_on_ep = 0;                                     // benign race: every writer stores 0
        }
        km[i] = keep ? 1 : 0;
        rel[i] = keep ? 8 : 0;
    }
    __syncthreads();
    const int kept = block_excl_scan(km, n0, wtot);              // km[i] = position of base point i among the kept ones
    const bool ins = p_valid && s_on_ep;
    if (ins)
        for (int i = tid; i < n0; i += nt)
            if ((rel[i] & 8) && p0 < -cx[i]) atomicMin(&s_ip, km[i]);      // p goes before the first kept q with p0 < q0
    __syncthreads();
    const int ip = min(s_ip, kept), n = kept + (ins ? 1 : 0);
    if (n == 0) {
        if (tid == 0) { hv[c] = 0.0; sp[c] = 0.0; }
        return;
    }
    // ---- where p ranks in the three lists; lowest base z rank among the removed points ----
    {
        const double px = cx[n0], py = cy[n0], pz = cz[n0];
        int r0 = 0, r1 = 0, r2 = 0, zmin = INT_MAX;
        for (int j = tid; j < n0; j += nt) {
            if (!(rel[j] & 8)) { zmin = min(zmin, b.zr[j]); continue; }
            if (!ins) continue;
            const bool xlt = cx[j] < px || (cx[j] == px && km[j] < ip);       // key (x, position in L)
            const bool ylt = cy[j] < py || (cy[j] == py && xlt);              // key (y, x, position)
            const bool zlt = cz[j] < pz || (cz[j] == pz && ylt);              // key (z, y, x, position)
            rel[j] |= (xlt ? 1 : 0) | (ylt ? 2 : 0) | (zlt ? 4 : 0);
            r0 += xlt; r1 += ylt; r2 += zlt;
        }
        if (r0) atomicAdd(&s_rp[0], r0);
        if (r1) atomicAdd(&s_rp[1], r1);
        if (r2) atomicAdd(&s_rp[2], r2);
        if (zmin != INT_MAX) atomicMin(&s_zmin, zmin);
    }
    __syncthreads();
    // ---- the sorted lists of L ----
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const int *bl = d == 0 ? b.xl : (d == 1 ? b.yl : b.zl);
        int *lst = d == 0 ? xl : (d == 1 ? yl : zl);
        for (int t = tid; t < n0; t += nt) tmp[t] = (rel[bl[t]] >> 3) & 1;
        __syncthreads();
        block_excl_scan(tmp, n0, wtot);
        for (int t = tid; t < n0; t += nt) {
            const int j = bl[t];
            if (!(rel[j] & 8)) continue;
            const int r = tmp[t] + ((ins && !((rel[j] >> d) & 1)) ? 1 : 0);
            lst[r] = j;
            if (d == 2) zr[j] = r;
        }
        if (tid == 0 && ins) { lst[s_rp[d]] = n0; if (d == 2) zr[n0] = s_rp[2]; }
        __syncthreads();
    }
    const int n_same = min(ins ? s_rp[2] : n, s_zmin == INT_MAX ? n : s_zmin);
    for (int t = tid; t < n; t += nt) { const int j = yl[t]; hx[t] = cx[j]; hy[t] = cy[j]; hz[t] = zr[j]; }
    __syncthreads();
    // ---- slices (warps 0-7) | sparsity (warp 8) ----
    if (warp < S3_WORKERS / 32) {
        for (int k = tid; k < n_same; k += S3_WORKERS) area[k] = b.area[k];
        for (int k = n_same + tid; k < n; k += S3_WORKERS) area[k] = slice_area(hx, hy, hz, n, k);
    } else {
        // utils.compute_sparsity: per dimension the ascending values (= the negated lists read backwards), one running sum
        const int m1 = n - 1;
        for (int idx = lane; idx < 3 * m1; idx += 32) {
            const int d = idx / m1, i = idx - d * m1 + 1;
            const int *lst = d == 0 ? xl : (d == 1 ? yl : zl);
            const double *v = d == 0 ? cx : (d == 1 ? cy : cz);
            const double g = dsub(-v[lst[n - 1 - i]], -v[lst[n - i]]);
            gsq[idx] = dmul(g, g);
        }
        __syncwarp();
        if (lane == 0) {
            double sacc = 0.0;
#pragma unroll 8
            for (int idx = 0; idx < 3 * m1; ++idx) sacc = dadd(sacc, gsq[idx]);
            sp[c] = n >= 2 ? sacc / (double)m1 : 0.0;
        }
    }
    __syncthreads();
    // ---- hypervolume: sum over the slices in order; the head of the sum is the base front's ----
    const int k0 = max(n_same, 1);
    for (int k = k0 + tid; k < n; k += nt) term[k] = dmul(area[k - 1], dsub(cz[zl[k]], cz[zl[k - 1]]));
    __syncthreads();
    if (tid == 0) {
        double v = b.vpre[k0 - 1];
#pragma unroll 8
        for (int k = k0; k < n; ++k) v = dadd(v, term[k]);
        v = dsub(v, dmul(area[n - 1], cz[zl[n - 1]]));
        hv[c] = round4(v);
    }
}

__global__ void __launch_bounds__(S3_THREADS) k5_score3d_inc_kernel(SelState st, int buf, const double *__restrict__ cand, int C,
                                                                    double *__restrict__ hv, double *__restrict__ sp, int nmax) {
    extern __shared__ __align__(16) unsigned char smraw[];
    score3d_inc_body(st, buf, cand, blockIdx.x, hv, sp, nmax, smraw);
}

// update_ep (utils.py:42-65) by all threads of one CTA: same result as update_front_3d. flags: [n] ints of shared memory.
__device__ inline void update_front_3d_block(const double *f, int n, const double *p, double *out, int *count_out, int *flags,
                                             int *wtot) {
    __shared__ int s_on, s_pos;
    const int tid = threadIdx.x, nt = blockDim.x;
    const double p0 = p[0], p1 = p[1], p2 = p[2];
    if (p0 < 0.0 || p1 < 0.0 || p2 < 0.0) {
        for (int i = tid; i < 3 * n; i += nt) out[i] = f[i];
        if (tid == 0) *count_out = n;
        __syncthreads();
        return;
    }
    if (tid == 0) { s_on = 1; s_pos = INT_MAX; }
    __syncthreads();
    for (int i = tid; i < n; i += nt) {
        const double q0 = f[3 * i], q1 = f[3 * i + 1], q2 = f[3 * i + 2];
        if (q0 >= p0 - 1e-5 && q1 >= p1 - 1e-5 && q2 >= p2 - 1e-5 && (q0 > p0 + 1e-5 || q1 > p1 + 1e-5 || q2 > p2 + 1e-5)) s_on = 0;
        flags[i] = (p0 >= q0 && p1 >= q1 && p2 >= q2) ? 0 : 1;
    }
    __syncthreads();
    const int m = block_excl_scan(flags, n, wtot);
    const bool on = s_on != 0;
    if (on)
        for (int i = tid; i < n; i += nt) {
            const double q0 = f[3 * i], q1 = f[3 * i + 1], q2 = f[3 * i + 2];
            if (!(p0 >= q0 && p1 >= q1 && p2 >= q2) && p0 < q0) atomicMin(&s_pos, flags[i]);
        }
    __syncthreads();
    const int pos = min(s_pos, m);
    for (int i = tid; i < n; i += nt) {
        const double q0 = f[3 * i], q1 = f[3 * i + 1], q2 = f[3 * i + 2];
        if (p0 >= q0 && p1 >= q1 && p2 >= q2) continue;
        const int dst = flags[i] + ((on && flags[i] >= pos) ? 1 : 0);
        out[3 * dst] = q0; out[3 * dst + 1] = q1; out[3 * dst + 2] = q2;
    }
    if (tid == 0) {
        if (on) { out[3 * pos] = p0; out[3 * pos + 1] = p1; out[3 * pos + 2] = p2; }
        *count_out = m + (on ? 1 : 0);
    }
    __syncthreads();
}

// ---- 4 objectives ---------------------------------------------------------------------------------
// update_ep (utils.py:42-65) at 4 objectives by all threads of one CTA; the same steps as update_front_3d_block.
__device__ inline void update_front_4d_block(const double *f, int n, const double *p, double *out, int *count_out, int *flags,
                                             int *wtot) {
    __shared__ int s_on, s_pos;
    const int tid = threadIdx.x, nt = blockDim.x;
    const double p0 = p[0], p1 = p[1], p2 = p[2], p3 = p[3];
    if (p0 < 0.0 || p1 < 0.0 || p2 < 0.0 || p3 < 0.0) {
        for (int i = tid; i < 4 * n; i += nt) out[i] = f[i];
        if (tid == 0) *count_out = n;
        __syncthreads();
        return;
    }
    if (tid == 0) { s_on = 1; s_pos = INT_MAX; }
    __syncthreads();
    for (int i = tid; i < n; i += nt) {
        const double *q = f + 4 * i;
        if (q[0] >= p0 - 1e-5 && q[1] >= p1 - 1e-5 && q[2] >= p2 - 1e-5 && q[3] >= p3 - 1e-5 &&
            (q[0] > p0 + 1e-5 || q[1] > p1 + 1e-5 || q[2] > p2 + 1e-5 || q[3] > p3 + 1e-5))
            s_on = 0;                                            // benign race: every writer stores 0
        flags[i] = (p0 >= q[0] && p1 >= q[1] && p2 >= q[2] && p3 >= q[3]) ? 0 : 1;
    }
    __syncthreads();
    const int m = block_excl_scan(flags, n, wtot);
    const bool on = s_on != 0;
    if (on)
        for (int i = tid; i < n; i += nt) {
            const double *q = f + 4 * i;
            if (!(p0 >= q[0] && p1 >= q[1] && p2 >= q[2] && p3 >= q[3]) && p0 < q[0]) atomicMin(&s_pos, flags[i]);
        }
    __syncthreads();
    const int pos = min(s_pos, m);
    for (int i = tid; i < n; i += nt) {
        const double *q = f + 4 * i;
        if (p0 >= q[0] && p1 >= q[1] && p2 >= q[2] && p3 >= q[3]) continue;
        const int dst = flags[i] + ((on && flags[i] >= pos) ? 1 : 0);
        out[4 * dst] = q[0]; out[4 * dst + 1] = q[1]; out[4 * dst + 2] = q[2]; out[4 * dst + 3] = q[3];
    }
    if (tid == 0) {
        if (on) { out[4 * pos] = p0; out[4 * pos + 1] = p1; out[4 * pos + 2] = p2; out[4 * pos + 3] = p3; }
        *count_out = m + (on ? 1 : 0);
    }
    __syncthreads();
}

// 2-D area (hvRecursive at dimIndex 1, hypervolume.py:92-105) of the points of the 4-D sweep that are in list 1 while
// slice (k, t) is computed: objective-3 rank <= k and objective-2 rank <= t. hx, hy, h2, h3: coordinates 0 and 1 and
// the ranks 2 and 3 of the points in list-1 order.
__device__ __forceinline__ double slice_area_4d(const double *hx, const double *hy, const int *h2, const int *h3, int n,
                                                int k, int t) {
    double h = 0.0, acc = 0.0, prevy = 0.0;
    bool first = true;
#pragma unroll 4
    for (int u = 0; u < n; ++u) {
        const double x = hx[u], y = hy[u];
        if (h3[u] > k || h2[u] > t) continue;
        if (first) { h = x; prevy = y; first = false; }
        else {
            acc = dadd(acc, dmul(h, dsub(prevy, y)));
            if (x < h) h = x;
            prevy = y;
        }
    }
    return dadd(acc, dmul(h, prevy));
}

// One CTA per candidate: L = update_ep(front, p); hv = round4(InnerHyperVolume(L)); sp = compute_sparsity(L), at 4
// objectives (use_cand = 0: L = the front itself, for pgm_front_metrics_f64).
//
// The hypervolume is hvRecursive (hypervolume.py:106-153) from dimIndex 3, restated without the linked lists but with
// the same float64 operations in the same order (tests/hv_ref.py keeps the lists; the two are compared bit for bit):
//  * The FPL lists only ever hold the points of the preProcess order that are currently inserted, in that order. At
//    level 3 the points enter in list-3 order; while point k of list 3 is processed, list 2 holds the points of
//    objective-3 rank <= k, and while the level-2 call processes the point at list-2 position t, list 1 holds those
//    of objective-2 rank <= t as well. So each level-1 call is slice_area_4d(k, t).
//  * Level 2 keeps the reference's state across calls: bounds[2] (lowered by every level-3 reinsert, set by every
//    level-2 reinsert), the stored volume[2] / area[2] of every point, and the ignore flags. A call first walks down
//    from the top of list 2 as the removal loop does, resumes its volume from the stored state of the point below the
//    first one it keeps, and takes area[2] from the predecessor for points whose flag is 2 or 3 ("ignore >= 2")
//    instead of calling level 1. Only the flags below 2 are ever reset, and none exist, so flags persist.
//  * bounds[0] and bounds[1] never rise above -1e308 and no level reads them; level 3 runs once, so its flag reset and
//    its own reuse branch never fire (a point's flag is 0 when level 3 reaches it: it was outside every earlier list).
// The level-1 calls of one level-2 call depend only on the point set, so they run in parallel (one thread per slice);
// the walk that strings them together -- volume chain, area reuse, flags -- is serial on thread 0.
//
// Dynamic shared memory (score4d_smem): 8 * nmax doubles, 7 * nmax ints, nmax flag bytes.
__global__ void __launch_bounds__(256) k5_score4d_kernel(SelState st, int buf, const double *__restrict__ cand, int C,
                                                         double *__restrict__ hv, double *__restrict__ sp, int nmax,
                                                         int use_cand) {
    extern __shared__ __align__(16) unsigned char smraw[];
    const int c = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    if (use_cand) {
        if (*st.done || !st.mask[c]) {
            if (tid == 0) { hv[c] = 0.0; sp[c] = 0.0; }
            return;
        }
    }
    double *c0 = reinterpret_cast<double *>(smraw), *c1 = c0 + nmax, *c2 = c1 + nmax, *c3 = c2 + nmax;
    double *hx = c3 + nmax, *hy = hx + nmax, *area2 = hy + nmax, *vol2 = area2 + nmax;
    int *pos = reinterpret_cast<int *>(vol2 + nmax), *r2 = pos + nmax, *r3 = r2 + nmax, *l2 = r3 + nmax, *l3 = l2 + nmax,
        *h2 = l3 + nmax, *h3 = h2 + nmax;
    unsigned char *flag = reinterpret_cast<unsigned char *>(h3 + nmax);
    double *cd[4] = {c0, c1, c2, c3};
    __shared__ int s_on_ep, s_n, s_ins, s_qt, s_qp, s_len;

    const double *f = st.front[buf];
    const int n0 = st.count[buf];
    double p[4] = {0.0, 0.0, 0.0, 0.0};
    bool p_valid = false;
    if (use_cand) {
        p[0] = cand[4 * c]; p[1] = cand[4 * c + 1]; p[2] = cand[4 * c + 2]; p[3] = cand[4 * c + 3];
        p_valid = p[0] >= 0.0 && p[1] >= 0.0 && p[2] >= 0.0 && p[3] >= 0.0;
    }
    if (tid == 0) { s_on_ep = 1; s_ins = 0; }
    __syncthreads();
    // ---- update_ep: keep flags (pos[i] = 1 if kept), on_ep, insertion index ----
    for (int i = tid; i < n0; i += nt) {
        const double *q = f + 4 * i;
        bool keep = true;
        if (p_valid) {
            keep = !(p[0] >= q[0] && p[1] >= q[1] && p[2] >= q[2] && p[3] >= q[3]);
            if (q[0] >= p[0] - 1e-5 && q[1] >= p[1] - 1e-5 && q[2] >= p[2] - 1e-5 && q[3] >= p[3] - 1e-5 &&
                (q[0] > p[0] + 1e-5 || q[1] > p[1] + 1e-5 || q[2] > p[2] + 1e-5 || q[3] > p[3] + 1e-5))
                s_on_ep = 0;                                     // benign race: every writer stores 0
        }
        pos[i] = keep ? 1 : 0;
    }
    __syncthreads();
    if (tid == 0) {
        const bool ins = p_valid && s_on_ep;
        int m = 0, ip = -1;
        for (int i = 0; i < n0; ++i) {
            if (pos[i]) {
                if (ins && ip < 0 && p[0] < f[4 * i]) { ip = m; ++m; }   // p goes before the first kept q with p0 < q0
                pos[i] = m; ++m;
            } else pos[i] = -1;
        }
        if (ins && ip < 0) { ip = m; ++m; }
        s_n = m; s_ins = ins ? ip : -1;
    }
    __syncthreads();
    const int n = s_n, ins = s_ins;
    for (int i = tid; i < n0; i += nt)
        if (pos[i] >= 0) {
#pragma unroll
            for (int d = 0; d < 4; ++d) cd[d][pos[i]] = -f[4 * i + d];
        }
    if (tid == 0 && ins >= 0) {
#pragma unroll
        for (int d = 0; d < 4; ++d) cd[d][ins] = -p[d];
    }
    __syncthreads();
    if (n == 0) {
        if (tid == 0) { hv[c] = 0.0; sp[c] = 0.0; }
        return;
    }
    // ---- utils.compute_sparsity: per dimension the ascending values (hx as scratch), one running sum on thread 0 ----
    double s = 0.0;
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        const double *v = cd[d];
        for (int i = tid; i < n; i += nt) {
            const double vi = -v[i];
            int r = 0;
            for (int j = 0; j < n; ++j) { const double vj = -v[j]; r += (vj < vi || (vj == vi && j < i)) ? 1 : 0; }
            hx[r] = vi;
        }
        __syncthreads();
        if (tid == 0)
            for (int i = 1; i < n; ++i) { const double g = dsub(hx[i], hx[i - 1]); s = dadd(s, dmul(g, g)); }
        __syncthreads();
    }
    // ---- the points that weakly dominate the reference point (hypervolume.py:55-61), compacted in order ----
    if (tid == 0) {
        sp[c] = n >= 2 ? s / (double)(n - 1) : 0.0;
        int m = 0;
        for (int i = 0; i < n; ++i)
            if (c0[i] <= 0.0 && c1[i] <= 0.0 && c2[i] <= 0.0 && c3[i] <= 0.0) {
                c0[m] = c0[i]; c1[m] = c1[i]; c2[m] = c2[i]; c3[m] = c3[i]; ++m;
            }
        s_n = m;
    }
    __syncthreads();
    const int nh = s_n;
    if (nh == 0) {
        if (tid == 0) hv[c] = 0.0;
        return;
    }
    // ---- preProcess (hypervolume.py:156-164): successive stable sorts by objectives 0, 1, 2, 3 ----
    for (int i = tid; i < nh; i += nt) {
        const double xi = c0[i], yi = c1[i], zi = c2[i], wi = c3[i];
        int ry = 0, rz = 0, rw = 0;
        for (int j = 0; j < nh; ++j) {
            const double xj = c0[j], yj = c1[j], zj = c2[j], wj = c3[j];
            const bool xlt = xj < xi || (xj == xi && j < i);                    // key (x, input position)
            const bool ylt = yj < yi || (yj == yi && xlt);                       // key (y, x, input position)
            const bool zlt = zj < zi || (zj == zi && ylt);                       // key (z, y, x, input position)
            const bool wlt = wj < wi || (wj == wi && zlt);                       // key (w, z, y, x, input position)
            ry += ylt; rz += zlt; rw += wlt;
        }
        r2[i] = rz; r3[i] = rw; l2[rz] = i; l3[rw] = i;
        hx[ry] = xi; hy[ry] = yi; h2[ry] = rz; h3[ry] = rw;
        flag[i] = 0; area2[i] = 0.0; vol2[i] = 0.0;
    }
    __syncthreads();
    // ---- the sweep; thread 0 holds bounds[2], the level-3 volume and the previous level-3 area ----
    double B = -1.0e308, hv3 = 0.0, a3prev = 0.0;
    for (int k = 0; k < nh; ++k) {
        if (tid == 0) {
            const int pk = l3[k];
            if (k > 0) {
                hv3 = dadd(hv3, dmul(a3prev, dsub(c3[pk], c3[l3[k - 1]])));
                if (B > c2[pk]) B = c2[pk];                                     // reinsert(p, 3, bounds)
            }
            // level-2 removal loop: from the top of list 2 down while q > bound or its predecessor >= bound
            int t = nh - 1;
            while (r3[l2[t]] > k) --t;
            int tp = t - 1;
            while (tp >= 0 && r3[l2[tp]] > k) --tp;
            int len = k + 1;
            while (len > 1 && (c2[l2[t]] > B || c2[l2[tp]] >= B)) {
                t = tp;
                --tp;
                while (tp >= 0 && r3[l2[tp]] > k) --tp;
                --len;
            }
            s_qt = t; s_qp = tp; s_len = len;
        }
        __syncthreads();
        // level-1 calls of this level-2 call, for the points that will not take their predecessor's area
        for (int t = s_qt + tid; t < nh; t += nt) {
            const int j = l2[t];
            if (r3[j] <= k && flag[j] < 2) area2[j] = slice_area_4d(hx, hy, h2, h3, nh, k, t);
        }
        __syncthreads();
        if (tid == 0) {
            const int qt = s_qt, qp = s_qp;
            int q = l2[qt];
            double hvol = 0.0;
            if (s_len > 1) {
                const int pq = l2[qp];
                hvol = dadd(vol2[pq], dmul(area2[pq], dsub(c2[q], c2[pq])));
            }
            vol2[q] = hvol;
            double aprev = qp >= 0 ? area2[l2[qp]] : 0.0;                      // the sentinel's area is 0
            if (flag[q] >= 2) area2[q] = aprev;
            else if (area2[q] <= aprev) flag[q] = 2;
            for (int t = qt + 1; t < nh; ++t) {
                const int pt = l2[t];
                if (r3[pt] > k) continue;
                hvol = dadd(hvol, dmul(area2[q], dsub(c2[pt], c2[q])));
                B = c2[pt];                                                      // bounds[dimIndex] = pCargoDimIndex
                aprev = area2[q];
                q = pt;
                vol2[q] = hvol;
                if (flag[q] >= 2) area2[q] = aprev;
                else if (area2[q] <= aprev) flag[q] = 2;
            }
            hvol = dsub(hvol, dmul(area2[q], c2[q]));
            // level 3: area[3] of point k; ignore = 3 when it did not grow (read by the later level-2 calls)
            if (hvol <= a3prev) flag[l3[k]] = 3;
            a3prev = hvol;
        }
    }
    if (tid == 0) {
        hv3 = dsub(hv3, dmul(a3prev, c3[l3[nh - 1]]));
        hv[c] = round4(hv3);
    }
}

// ---- arg-max + virtual EP update: single CTA ---------------------------------------------------------
// 3 objectives: dynamic shared memory of base3d_smem(nmax) bytes (first used as nmax ints by the front update); the new
// front's base data for the next round's scorer is built here. 4 objectives: nmax ints for the front update.
// GLOBAL (3 objectives only, k5g_pick3d_kernel): the front update's flags are pick_smem in global memory, and the base
// data is left to the k5g_base3d_* kernels.
template <int M, bool GLOBAL>
__device__ __forceinline__ void pick_body(const SelState &st, int buf, const double *__restrict__ cand, int C,
                                          const double *__restrict__ hv, const double *__restrict__ sp, double alpha,
                                          int32_t *__restrict__ best_out, int nmax, unsigned char *pick_smem) {
    __shared__ double sv[32];
    __shared__ int si[32];
    __shared__ int wtot[32];
    const int tid = threadIdx.x;
    __shared__ int s_copy, s_bi;
    if (tid == 0) { s_copy = *st.done; s_bi = -1; }
    __syncthreads();
    if (!s_copy) {
        double bv = -INFINITY;
        int bi = -1;
        for (int c = tid; c < C; c += blockDim.x)
            if (st.mask[c]) {
                const double m = dsub(hv[c], dmul(alpha, sp[c]));
                if (m > bv) { bv = m; bi = c; }      // ascending c per thread: strict '>' keeps the first index
            }
        // max value, ties -> smallest index (the reference's strict '>' scan in index order)
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
        }
        if ((tid & 31) == 0) { sv[tid >> 5] = bv; si[tid >> 5] = bi; }
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < (int)((blockDim.x + 31) >> 5); ++w) {
                const double ov = sv[w]; const int oi = si[w];
                if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
            }
            *best_out = bi;
            s_bi = bi;
            if (bi < 0) { *st.done = 1; s_copy = 1; }      // "Too few candidates": stop, keep the front
            else {
                st.mask[bi] = 0;
                if (M == 2) st.count[buf ^ 1] = update_front_2d(st.front[buf], st.count[buf], cand[2 * bi], cand[2 * bi + 1], st.front[buf ^ 1]);
            }
        }
        __syncthreads();
        if (M == 3 && s_bi >= 0) {
            update_front_3d_block(st.front[buf], st.count[buf], cand + 3 * s_bi, st.front[buf ^ 1], &st.count[buf ^ 1],
                                  reinterpret_cast<int *>(pick_smem), wtot);
            if (!GLOBAL) base3d_build(st.front[buf ^ 1], st.count[buf ^ 1], nmax, st.b3, pick_smem);
        }
        if (M == 4 && s_bi >= 0)
            update_front_4d_block(st.front[buf], st.count[buf], cand + 4 * s_bi, st.front[buf ^ 1], &st.count[buf ^ 1],
                                  reinterpret_cast<int *>(pick_smem), wtot);
    } else if (tid == 0) *best_out = -1;
    if (s_copy) {      // no pick this round: carry the front over so the buffers keep alternating
        const int n = st.count[buf];
        for (int i = tid; i < n * M; i += blockDim.x) st.front[buf ^ 1][i] = st.front[buf][i];
        if (tid == 0) st.count[buf ^ 1] = n;
    }
}

template <int M>
__global__ void __launch_bounds__(1024) k5_pick_kernel(SelState st, int buf, const double *__restrict__ cand, int C,
                                                       const double *__restrict__ hv, const double *__restrict__ sp,
                                                       double alpha, int32_t *__restrict__ best_out, int nmax) {
    extern __shared__ __align__(16) unsigned char pick_smem[];
    pick_body<M, false>(st, buf, cand, C, hv, sp, alpha, best_out, nmax, pick_smem);
}

// ---- 3 objectives on fronts past the shared-memory layouts: global-memory scratch ------------------------------------
// The same float64 operations in the same order as k5_base3d_kernel / k5_score3d_inc_kernel / k5_pick_kernel<3> /
// k5_score3d_kernel, so every result is bit-identical to theirs wherever both run; the per-point arrays live in the
// workspace instead of shared memory, so a front has no size limit besides the workspace.
struct Glob3d {
    double *hx, *hy;            // [nmax] x, y of the base front's points in y-list order
    int *hz;                    // [nmax] their z ranks
    int *flags;                 // [nmax] scratch of the front update
    unsigned char *scratch;     // [S3G_CTAS][stride] one score3d_inc_smem(nmax) layout per CTA of the scorer
    size_t stride;
};
// CTAs of the global scorer, each looping over candidates with one scratch: the workspace does not grow with C.
// 296 = two per SM of a B200.
constexpr int S3G_CTAS = 296;

// The base data of base3d_build, in three launches over the whole grid. Ranks: one thread per point, the front streamed
// through shared-memory tiles, the comparisons of base3d_build (integers, so any schedule gives the same lists).
__global__ void __launch_bounds__(256) k5g_base3d_rank_kernel(SelState st, int buf, Glob3d g) {
    __shared__ double tx[256], ty[256], tz[256];
    const Base3d b = st.b3;
    const double *f = st.front[buf];
    const int n0 = st.count[buf], i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < n0;
    double xi = 0.0, yi = 0.0, zi = 0.0;
    if (valid) {
        xi = -f[3 * i]; yi = -f[3 * i + 1]; zi = -f[3 * i + 2];
        b.nx[i] = xi; b.ny[i] = yi; b.nz[i] = zi;
    }
    if (i == 0) b.vpre[0] = 0.0;
    int rx = 0, ry = 0, rz = 0;
    for (int j0 = 0; j0 < n0; j0 += 256) {
        const int nj = min(256, n0 - j0);
        __syncthreads();
        for (int t = threadIdx.x; t < nj; t += blockDim.x) {
            tx[t] = -f[3 * (j0 + t)]; ty[t] = -f[3 * (j0 + t) + 1]; tz[t] = -f[3 * (j0 + t) + 2];
        }
        __syncthreads();
        if (valid)
#pragma unroll 4
            for (int t = 0; t < nj; ++t) {
                const int j = j0 + t;
                const double xj = tx[t], yj = ty[t], zj = tz[t];
                const bool xlt = xj < xi || (xj == xi && j < i);
                const bool ylt = yj < yi || (yj == yi && xlt);
                const bool zlt = zj < zi || (zj == zi && ylt);
                rx += xlt; ry += ylt; rz += zlt;
            }
    }
    if (valid) {
        b.xl[rx] = i; b.yl[ry] = i; b.zl[rz] = i; b.zr[i] = rz;
        g.hx[ry] = xi; g.hy[ry] = yi; g.hz[ry] = rz;
    }
}

// slice areas: one thread per slice
__global__ void __launch_bounds__(256) k5g_base3d_area_kernel(SelState st, int buf, Glob3d g) {
    const int n0 = st.count[buf], k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n0) st.b3.area[k] = slice_area(g.hx, g.hy, g.hz, n0, k);
}

// the hypervolume chain: terms in parallel, the running sum on thread 0 (one CTA)
__global__ void __launch_bounds__(1024) k5g_base3d_chain_kernel(SelState st, int buf) {
    const Base3d b = st.b3;
    const int n0 = st.count[buf], tid = threadIdx.x;
    for (int k = 1 + tid; k < n0; k += blockDim.x) b.vpre[k] = dmul(b.area[k - 1], dsub(b.nz[b.zl[k]], b.nz[b.zl[k - 1]]));
    __syncthreads();
    if (tid == 0) {
        double v = 0.0;
#pragma unroll 8
        for (int k = 1; k < n0; ++k) { v = dadd(v, b.vpre[k]); b.vpre[k] = v; }
    }
}

// The incremental scorer on per-CTA global scratch: a grid of resident CTAs loops over the candidates.
__global__ void __launch_bounds__(S3_THREADS) k5g_score3d_inc_kernel(SelState st, int buf, const double *__restrict__ cand, int C,
                                                                     double *__restrict__ hv, double *__restrict__ sp, int nmax,
                                                                     Glob3d g) {
    unsigned char *scratch = g.scratch + (size_t)blockIdx.x * g.stride;
    for (int c = blockIdx.x; c < C; c += gridDim.x) {
        score3d_inc_body(st, buf, cand, c, hv, sp, nmax, scratch);
        __syncthreads();                                   // the next candidate reuses the scratch and the shared words
    }
}

__global__ void __launch_bounds__(1024) k5g_pick3d_kernel(SelState st, int buf, const double *__restrict__ cand, int C,
                                                          const double *__restrict__ hv, const double *__restrict__ sp,
                                                          double alpha, int32_t *__restrict__ best_out, Glob3d g) {
    pick_body<3, true>(st, buf, cand, C, hv, sp, alpha, best_out, 0, reinterpret_cast<unsigned char *>(g.flags));
}

// Metrics of front[0] from its base data (pgm_front_metrics_f64): k5_score3d_kernel's hypervolume and sparsity, whose
// sums are the base chain and the base lists read backwards. front[0] holds n >= 1 points.
__global__ void k5g_metrics3d_kernel(SelState st, double *__restrict__ out) {
    const Base3d b = st.b3;
    const int n = st.count[0];
    if (threadIdx.x == 0) {
        const double v = dsub(b.vpre[n - 1], dmul(b.area[n - 1], b.nz[b.zl[n - 1]]));
        out[0] = round4(v);
    } else if (threadIdx.x == 32) {
        double s = 0.0;
        if (n >= 2) {
            for (int d = 0; d < 3; ++d) {
                const int *lst = d == 0 ? b.xl : (d == 1 ? b.yl : b.zl);
                const double *v = d == 0 ? b.nx : (d == 1 ? b.ny : b.nz);
                for (int i = 1; i < n; ++i) {
                    const double gap = dsub(-v[lst[n - 1 - i]], -v[lst[n - i]]);
                    s = dadd(s, dmul(gap, gap));
                }
            }
            s = s / (double)(n - 1);
        }
        out[1] = s;
    }
}

__global__ void k5_init_kernel(SelState st, const double *__restrict__ ep, int E, int M, int C) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < E * M) st.front[0][i] = ep[i];
    if (i < C) st.mask[i] = 1;
    if (i == 0) { st.count[0] = E; st.count[1] = 0; *st.done = 0; }
}

__global__ void k5_finish_kernel(SelState st, int buf, int M, double *front_out, int32_t *n_front) {
    const int n = st.count[buf];
    if (n_front && blockIdx.x == 0 && threadIdx.x == 0) *n_front = n;
    if (front_out)
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n * M; i += gridDim.x * blockDim.x) front_out[i] = st.front[buf][i];
}

// 2-D metrics of an arbitrary point set: Pareto filter (kept/keep_idx from the kernels above), then closed forms
__global__ void k5_metrics2d_kernel(const double *__restrict__ pts, const int32_t *__restrict__ keep_idx,
                                    const int32_t *__restrict__ n_keep, double *__restrict__ out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int n = *n_keep;
    double hv = 0.0, xprev = 0.0, sp = 0.0;
    for (int i = 0; i < n; ++i) {
        const double x = pts[2 * keep_idx[i]], y = pts[2 * keep_idx[i] + 1];
        hv = dadd(hv, dmul(dsub(fmax(0.0, x), xprev), dsub(fmax(0.0, y), 0.0)));
        xprev = fmax(0.0, x);
        if (i > 0) {
            const double dx = dsub(x, pts[2 * keep_idx[i - 1]]), dy = dsub(y, pts[2 * keep_idx[i - 1] + 1]);
            sp = dadd(sp, dadd(dmul(dx, dx), dmul(dy, dy)));
        }
    }
    out[0] = hv;
    out[1] = n < 2 ? 0.0 : sp / (double)(n - 1);
}

static size_t score3d_smem(int nmax) { return (size_t)nmax * (4 * sizeof(double) + 5 * sizeof(int)); }
static size_t score3d_inc_smem(int nmax) { return (size_t)nmax * (9 * sizeof(double) + 6 * sizeof(int) + 1) + 16; }
// Largest shared-memory layout of the 3-D kernels: fronts up to 2 111 points for the incremental scorer
// (archive + num_tasks + 1) and 3 936 for the one-front scorer.
constexpr size_t SCORE3D_SMEM_MAX = 200 * 1024;

// global3: carve the global-memory 3-D path's arrays (Glob3d) as well, for up to C candidates.
static size_t sel_carve(SelState &st, Glob3d &g, char *ws, int E, int C, int M, int num_tasks, bool global3) {
    size_t off = 0;
    auto seg = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t fb = (size_t)(E + num_tasks + 1) * M * sizeof(double);
    const size_t o0 = seg(fb), o1 = seg(fb), oc = seg(2 * sizeof(int)), om = seg((size_t)(C > 0 ? C : 1) * sizeof(int)), od = seg(sizeof(int));
    if (ws) {
        st.front[0] = (double *)(ws + o0); st.front[1] = (double *)(ws + o1);
        st.count = (int *)(ws + oc); st.mask = (int *)(ws + om); st.done = (int *)(ws + od);
    }
    if (M == 3) {
        const size_t nmax = (size_t)(E + num_tasks + 1);
        const size_t od5 = seg(5 * nmax * sizeof(double)), oi4 = seg(4 * nmax * sizeof(int));
        if (ws) {
            double *d = (double *)(ws + od5);
            int *i = (int *)(ws + oi4);
            st.b3.nx = d; st.b3.ny = d + nmax; st.b3.nz = d + 2 * nmax; st.b3.area = d + 3 * nmax; st.b3.vpre = d + 4 * nmax;
            st.b3.xl = i; st.b3.yl = i + nmax; st.b3.zl = i + 2 * nmax; st.b3.zr = i + 3 * nmax;
        }
        if (global3) {
            const size_t stride = (score3d_inc_smem((int)nmax) + 255) / 256 * 256;
            const int ctas = C < 1 ? 1 : (C < S3G_CTAS ? C : S3G_CTAS);
            const size_t ohx = seg(nmax * sizeof(double)), ohy = seg(nmax * sizeof(double)), ohz = seg(nmax * sizeof(int)),
                         ofl = seg(nmax * sizeof(int)), osc = seg(ctas * stride);
            if (ws) {
                g.hx = (double *)(ws + ohx); g.hy = (double *)(ws + ohy); g.hz = (int *)(ws + ohz); g.flags = (int *)(ws + ofl);
                g.scratch = (unsigned char *)(ws + osc); g.stride = stride;
            }
        }
    }
    return off;
}

// Which 3-D path pgm_select_greedy_x_f64 takes (the workspace query sizes for it; pgm_front_metrics_x_f64's own choice,
// at 3 936 points, is never global where this one is not).
static bool select_global3(int M, int nmax, int flags) {
    return M == 3 && ((flags & PGM_SEL_GLOBAL) || score3d_inc_smem(nmax) > SCORE3D_SMEM_MAX);
}

// base data of front[buf] for the global path
static void base3d_global(const SelState &st, int buf, const Glob3d &g, int nmax, cudaStream_t s) {
    const int blocks = (nmax + 255) / 256;
    k5g_base3d_rank_kernel<<<blocks, 256, 0, s>>>(st, buf, g);
    k5g_base3d_area_kernel<<<blocks, 256, 0, s>>>(st, buf, g);
    k5g_base3d_chain_kernel<<<1, 1024, 0, s>>>(st, buf);
}

static size_t score4d_smem(int nmax) { return (size_t)nmax * (8 * sizeof(double) + 7 * sizeof(int) + 1); }
// Largest front (points of L = update_ep(front, p)) the 4-D scorer's shared-memory layout holds: 2 202 points.
constexpr size_t SCORE4D_SMEM_MAX = 200 * 1024;

}  // namespace pgm

using namespace pgm;

extern "C" int pgm_ep_filter_f64(const double *objs, int n, int M, int32_t *keep_idx, int32_t *n_keep, void *stream) {
    PGM_REQUIRE(keep_idx && n_keep && (objs || n == 0), "pgm_ep_filter_f64: null pointer");
    PGM_REQUIRE(n >= 0 && M >= 1 && M <= 4, "pgm_ep_filter_f64: need 1 <= M <= 4 (got %d)", M);
    cudaStream_t st = (cudaStream_t)stream;
    PGM_CUDA(cudaMemsetAsync(n_keep, 0, sizeof(int32_t), st));
    if (n == 0) return PGM_OK;
    // keep flags live in keep_idx's tail? no: n flags + n indices cannot overlap -> small side allocation is
    // avoided by packing the flags into the upper half of a temporary borrowed from the caller: require 2n ints
    int *kept = reinterpret_cast<int *>(keep_idx) + n;      // caller provides keep_idx with room for 2n int32
    const int blocks = (n + 255) / 256;
#define PGM_K5F(MM) case MM: k5_dominance_kernel<MM><<<blocks, 256, 0, st>>>(objs, n, kept); \
                             k5_rank_kernel<MM><<<blocks, 256, 0, st>>>(objs, n, kept, keep_idx, n_keep); break;
    switch (M) { PGM_K5F(1) PGM_K5F(2) PGM_K5F(3) PGM_K5F(4) }
#undef PGM_K5F
    PGM_CUDA(cudaGetLastError());
    return PGM_OK;
}

extern "C" size_t pgm_select_workspace_bytes_x(int E, int C, int M, int num_tasks, int flags) {
    SelState st;
    Glob3d g;
    // + room for the ep_filter scratch used by pgm_front_metrics_f64 (2 * n int32 + count)
    return sel_carve(st, g, nullptr, E, C, M, num_tasks, select_global3(M, E + num_tasks + 1, flags)) +
           ((size_t)(2 * E + 2) * sizeof(int32_t) + 255) / 256 * 256;
}

extern "C" size_t pgm_select_workspace_bytes(int E, int C, int M, int num_tasks) {
    return pgm_select_workspace_bytes_x(E, C, M, num_tasks, 0);
}

extern "C" int pgm_select_greedy_x_f64(const double *ep, int E, const double *cand, int C, int M, double alpha,
                                       int num_tasks, int flags, int32_t *best_ids, double *hv, double *sparsity,
                                       double *front_out, int32_t *n_front, void *workspace, size_t workspace_bytes,
                                       void *stream) {
    PGM_REQUIRE((ep || E == 0) && (cand || C == 0) && best_ids && hv && sparsity && workspace, "pgm_select_greedy_f64: null pointer");
    PGM_REQUIRE(M >= 2 && M <= 4, "pgm_select_greedy_f64: exact hypervolume is implemented for 2 to 4 objectives (got %d)", M);
    PGM_REQUIRE(E >= 0 && C >= 0 && num_tasks >= 1, "pgm_select_greedy_f64: bad sizes E=%d C=%d num_tasks=%d", E, C, num_tasks);
    PGM_REQUIRE((flags & ~PGM_SEL_GLOBAL) == 0, "pgm_select_greedy_f64: unknown flags 0x%x", flags);
    PGM_REQUIRE(!(flags & PGM_SEL_GLOBAL) || M == 3, "pgm_select_greedy_f64: PGM_SEL_GLOBAL is a 3-objective path (got M=%d)", M);
    PGM_REQUIRE(((uintptr_t)workspace & 255) == 0, "pgm_select_greedy_f64: workspace must be 256-byte aligned");
    const int nmax = E + num_tasks + 1;
    const bool global3 = select_global3(M, nmax, flags);
    SelState st;
    Glob3d g;
    const size_t need = sel_carve(st, g, (char *)workspace, E, C, M, num_tasks, global3);
    if (need > workspace_bytes) { set_error("pgm_select_greedy_f64: workspace too small: need %zu, got %zu", need, workspace_bytes); return PGM_ERR_WORKSPACE; }
    cudaStream_t s = (cudaStream_t)stream;
    const size_t smem3 = score3d_inc_smem(nmax), smemb = base3d_smem(nmax);
    if (M == 3 && !global3) {
        PGM_CUDA(cudaFuncSetAttribute(k5_score3d_inc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3));
        PGM_CUDA(cudaFuncSetAttribute(k5_base3d_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemb));
        PGM_CUDA(cudaFuncSetAttribute(k5_pick_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemb));
    }
    const size_t smem4 = score4d_smem(nmax), smemp4 = (size_t)nmax * sizeof(int);
    if (M == 4) {
        PGM_REQUIRE(smem4 <= SCORE4D_SMEM_MAX, "pgm_select_greedy_f64: front of %d points exceeds the 4-D scorer's shared memory "
                    "(at most %d points: archive + num_tasks + 1)", nmax, (int)(SCORE4D_SMEM_MAX / score4d_smem(1)));
        PGM_CUDA(cudaFuncSetAttribute(k5_score4d_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4));
    }
    {
        const int nthr = (E * M > C ? E * M : C) + 1;
        k5_init_kernel<<<(nthr + 255) / 256, 256, 0, s>>>(st, ep, E, M, C);
        if (M == 3 && C > 0) {
            if (global3) base3d_global(st, 0, g, nmax, s);
            else k5_base3d_kernel<<<1, 1024, smemb, s>>>(st, 0, nmax);
        }
    }
    for (int r = 0; r < num_tasks; ++r) {
        const int buf = r & 1;
        double *hv_r = hv + (size_t)r * C, *sp_r = sparsity + (size_t)r * C;
        if (global3) {
            if (C > 0) k5g_score3d_inc_kernel<<<C < S3G_CTAS ? C : S3G_CTAS, S3_THREADS, 0, s>>>(st, buf, cand, C, hv_r, sp_r, nmax, g);
            k5g_pick3d_kernel<<<1, 1024, 0, s>>>(st, buf, cand, C, hv_r, sp_r, alpha, best_ids + r, g);
            if (C > 0 && r + 1 < num_tasks) base3d_global(st, buf ^ 1, g, nmax, s);
            continue;
        }
        if (C > 0) {
            if (M == 2) k5_score2d_kernel<<<(C + 127) / 128, 128, 0, s>>>(st, buf, cand, C, hv_r, sp_r);
            else if (M == 3) k5_score3d_inc_kernel<<<C, S3_THREADS, smem3, s>>>(st, buf, cand, C, hv_r, sp_r, nmax);
            else k5_score4d_kernel<<<C, 256, smem4, s>>>(st, buf, cand, C, hv_r, sp_r, nmax, 1);
        }
        if (M == 2) k5_pick_kernel<2><<<1, 1024, 0, s>>>(st, buf, cand, C, hv_r, sp_r, alpha, best_ids + r, nmax);
        else if (M == 3) k5_pick_kernel<3><<<1, 1024, smemb, s>>>(st, buf, cand, C, hv_r, sp_r, alpha, best_ids + r, nmax);
        else k5_pick_kernel<4><<<1, 1024, smemp4, s>>>(st, buf, cand, C, hv_r, sp_r, alpha, best_ids + r, nmax);
    }
    k5_finish_kernel<<<8, 256, 0, s>>>(st, num_tasks & 1, M, front_out, n_front);
    PGM_CUDA(cudaGetLastError());
    return PGM_OK;
}

extern "C" int pgm_select_greedy_f64(const double *ep, int E, const double *cand, int C, int M, double alpha,
                                     int num_tasks, int32_t *best_ids, double *hv, double *sparsity, double *front_out,
                                     int32_t *n_front, void *workspace, size_t workspace_bytes, void *stream) {
    return pgm_select_greedy_x_f64(ep, E, cand, C, M, alpha, num_tasks, 0, best_ids, hv, sparsity, front_out, n_front,
                                   workspace, workspace_bytes, stream);
}

extern "C" int pgm_front_metrics_x_f64(const double *pts, int n, int M, int flags, double *out, void *workspace,
                                       size_t workspace_bytes, void *stream) {
    PGM_REQUIRE(out && workspace && (pts || n == 0), "pgm_front_metrics_f64: null pointer");
    PGM_REQUIRE(M >= 2 && M <= 4, "pgm_front_metrics_f64: implemented for 2 to 4 objectives (got %d)", M);
    PGM_REQUIRE(n >= 0, "pgm_front_metrics_f64: bad size n=%d", n);
    PGM_REQUIRE((flags & ~PGM_SEL_GLOBAL) == 0, "pgm_front_metrics_f64: unknown flags 0x%x", flags);
    PGM_REQUIRE(!(flags & PGM_SEL_GLOBAL) || M == 3, "pgm_front_metrics_f64: PGM_SEL_GLOBAL is a 3-objective path (got M=%d)", M);
    PGM_REQUIRE(((uintptr_t)workspace & 255) == 0, "pgm_front_metrics_f64: workspace must be 256-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    const int nmax3 = n + 2;
    const bool global3 = M == 3 && ((flags & PGM_SEL_GLOBAL) || score3d_smem(nmax3) > SCORE3D_SMEM_MAX);
    SelState st;
    Glob3d g;
    const size_t base = sel_carve(st, g, (char *)workspace, n, 1, M, 1, global3);
    const size_t need = base + ((size_t)(2 * n + 2) * sizeof(int32_t) + 255) / 256 * 256;
    if (need > workspace_bytes) { set_error("pgm_front_metrics_f64: workspace too small: need %zu, got %zu", need, workspace_bytes); return PGM_ERR_WORKSPACE; }
    if (n == 0) { PGM_CUDA(cudaMemsetAsync(out, 0, 2 * sizeof(double), s)); return PGM_OK; }
    if (M == 2) {
        int32_t *keep_idx = (int32_t *)((char *)workspace + base);
        int32_t *n_keep = keep_idx + 2 * n;
        PGM_CUDA(cudaMemsetAsync(n_keep, 0, sizeof(int32_t), s));
        const int blocks = (n + 255) / 256;
        k5_dominance_kernel<2><<<blocks, 256, 0, s>>>(pts, n, (int *)(keep_idx + n));
        k5_rank_kernel<2><<<blocks, 256, 0, s>>>(pts, n, (int *)(keep_idx + n), keep_idx, n_keep);
        k5_metrics2d_kernel<<<1, 32, 0, s>>>(pts, keep_idx, n_keep, out);
    } else if (M == 4) {
        const size_t smem4 = score4d_smem(n);
        PGM_REQUIRE(smem4 <= SCORE4D_SMEM_MAX, "pgm_front_metrics_f64: %d points exceed the 4-D scorer's shared memory (at most %d)",
                    n, (int)(SCORE4D_SMEM_MAX / score4d_smem(1)));
        PGM_CUDA(cudaFuncSetAttribute(k5_score4d_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4));
        k5_init_kernel<<<(n * M + 256) / 256, 256, 0, s>>>(st, pts, n, M, 0);
        k5_score4d_kernel<<<1, 256, smem4, s>>>(st, 0, nullptr, 1, out, out + 1, n, 0);
    } else if (global3) {
        k5_init_kernel<<<(n * M + 256) / 256, 256, 0, s>>>(st, pts, n, M, 0);
        base3d_global(st, 0, g, nmax3, s);
        k5g_metrics3d_kernel<<<1, 64, 0, s>>>(st, out);
    } else {
        const size_t smem3 = score3d_smem(nmax3);
        PGM_CUDA(cudaFuncSetAttribute(k5_score3d_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3));
        k5_init_kernel<<<(n * M + 256) / 256, 256, 0, s>>>(st, pts, n, M, 0);
        k5_score3d_kernel<<<1, 256, smem3, s>>>(st, 0, nullptr, 1, out, out + 1, nmax3, 0);
    }
    PGM_CUDA(cudaGetLastError());
    return PGM_OK;
}

extern "C" int pgm_front_metrics_f64(const double *pts, int n, int M, double *out, void *workspace,
                                     size_t workspace_bytes, void *stream) {
    return pgm_front_metrics_x_f64(pts, n, M, 0, out, workspace, workspace_bytes, stream);
}
