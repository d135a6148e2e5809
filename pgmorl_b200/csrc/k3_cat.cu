// K3 for Categorical heads: the generic cluster kernel (k3_body.cuh) with CAT = true, at hidden widths 32, 64 and 128,
// 2..16 CTAs per task, the three chunk / gather variants and both value losses. A translation unit of its own so that it
// compiles beside k3_ppo.cu.
#include "k3_body.cuh"

namespace pgm {

template <int HW, int C, int TM, int KG1, int NA, bool DB, bool VU>
__global__ void __launch_bounds__(NTHREADS, 1) k3_ppo_cat_kernel(const K3Args a) {
    k3_ppo_body<C, TM, KG1, NA, DB, VU, HW, true>(a);
}

template <typename Kern>
static int k3_cat_go(Kern kern, int C, const K3Args &a, size_t smem, int P, cudaStream_t st) {
    PGM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (C > 8) PGM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(P * C); cfg.blockDim = dim3(NTHREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    PGM_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
    return PGM_OK;
}

// the variants k3_plan picks: wide (KG1 and NA of the width, as for Gaussian heads), or narrow with TM = 2 / 4
template <int HW, int C, bool VU>
static int k3_cat_c(const K3Args &a, int TM, bool wide, size_t smem, int P, cudaStream_t st) {
    constexpr int KGB = HW == 64 ? 6 : (HW == 128 ? 2 : 3), NAB = HW == 32 ? 1 : 2;
    if (wide) return k3_cat_go(k3_ppo_cat_kernel<HW, C, 2, KGB, NAB, false, VU>, C, a, smem, P, st);
    return TM == 2 ? k3_cat_go(k3_ppo_cat_kernel<HW, C, 2, 1, 1, true, VU>, C, a, smem, P, st)
                   : k3_cat_go(k3_ppo_cat_kernel<HW, C, 4, 1, 1, true, VU>, C, a, smem, P, st);
}

template <int HW, bool VU>
static int k3_cat_h(const K3Args &a, int C, int TM, bool wide, size_t smem, int P, cudaStream_t st) {
    switch (C) {
        case 2: return k3_cat_c<HW, 2, VU>(a, TM, wide, smem, P, st);
        case 4: return k3_cat_c<HW, 4, VU>(a, TM, wide, smem, P, st);
        case 8: return k3_cat_c<HW, 8, VU>(a, TM, wide, smem, P, st);
        case 16: return k3_cat_c<HW, 16, VU>(a, TM, wide, smem, P, st);
    }
    set_error("ppo: bad cluster %d for a categorical head", C);
    return PGM_ERR_ARG;
}

template <bool VU>
static int k3_cat_v(const K3Args &a, int hidden, int C, int TM, bool wide, size_t smem, int P, cudaStream_t st) {
    if (hidden == 32) return k3_cat_h<32, VU>(a, C, TM, wide, smem, P, st);
    if (hidden == 128) return k3_cat_h<128, VU>(a, C, TM, wide, smem, P, st);
    return k3_cat_h<64, VU>(a, C, TM, wide, smem, P, st);
}

int k3_launch_cat(const K3Args &a, int hidden, int C, int TM, bool wide, bool vu, size_t smem, int P, cudaStream_t st) {
    return vu ? k3_cat_v<true>(a, hidden, C, TM, wide, smem, P, st) : k3_cat_v<false>(a, hidden, C, TM, wide, smem, P, st);
}

}  // namespace pgm
