/*
 * Instantiations of the fused 4-state kernels (fused4.cuh): their own translation unit, because the ~90
 * template instances dominate the build time and change rarely.  The __constant__ matrices of the CM kernels
 * live here too, so the copy into them does as well.
 */
#include <cuda_runtime.h>
#include "fused4.cuh"

/* mode 3: the configurations of mode 2 less the four in which ptxas (CUDA 12.9) spills at the register cap
 * (-Xptxas -v); the tuning in run_fused picks among the others */
template <int C, int BD, int STAGED, bool PACK>
static f4_kernel_t f4_gm_kernel()
{
    constexpr bool spills = (C == 4 && BD == 384 && STAGED <= 1 && PACK == (STAGED == 0)) || (C == 2 && BD <= 256 && STAGED == 0);
    if constexpr (spills) return nullptr;
    else return fused4_kernel<C, 3, BD, STAGED, PACK, false>;
}

/* the outside-pass modes without edge-form tables: 2 (marginals) and 3 (per-edge outer-product matrices) */
template <int BD, int STAGED, bool PACK>
static f4_kernel_t f4_select_marg(int C, int mode)
{
    switch (C * 2 + (mode == 3 ? 1 : 0)) {
    case 2: return fused4_kernel<1, 2, BD, STAGED, PACK, false>;
    case 3: return f4_gm_kernel<1, BD, STAGED, PACK>();
    case 4: return fused4_kernel<2, 2, BD, STAGED, PACK, false>;
    case 5: return f4_gm_kernel<2, BD, STAGED, PACK>();
    case 6: return fused4_kernel<3, 2, BD, STAGED, PACK, false>;
    case 7: return f4_gm_kernel<3, BD, STAGED, PACK>();
    case 8: return fused4_kernel<4, 2, BD, STAGED, PACK, false>;
    case 9: return f4_gm_kernel<4, BD, STAGED, PACK>();
    }
    return nullptr;
}

template <int BD, int STAGED, bool PACK, bool CM = false>
static f4_kernel_t f4_select_c(int C, bool edge)
{
    switch (C * 2 + (edge ? 1 : 0)) {
    case 2: return fused4_kernel<1, 0, BD, STAGED, PACK, CM>;
    case 3: return fused4_kernel<1, 1, BD, STAGED, PACK, CM>;
    case 4: return fused4_kernel<2, 0, BD, STAGED, PACK, CM>;
    case 5: return fused4_kernel<2, 1, BD, STAGED, PACK, CM>;
    case 6: return fused4_kernel<3, 0, BD, STAGED, PACK, CM>;
    case 7: return fused4_kernel<3, 1, BD, STAGED, PACK, CM>;
    case 8: return fused4_kernel<4, 0, BD, STAGED, PACK, CM>;
    case 9: return fused4_kernel<4, 1, BD, STAGED, PACK, CM>;
    }
    return nullptr;
}

#define F4_KEY(bd, staged, pack, cm) ((bd) * 100 + (staged) * 10 + ((pack) ? 2 : 0) + ((cm) ? 1 : 0))

f4_kernel_t f4_get_kernel(int bd, int staged, bool pack, bool cm, int C, int mode)
{
    const int key = F4_KEY(bd, staged, pack, cm);
    if (mode == 2 || mode == 3) {
        switch (key) {
        case F4_KEY(384, 1, true, false): return f4_select_marg<384, 1, true>(C, mode);
        case F4_KEY(384, 1, false, false): return f4_select_marg<384, 1, false>(C, mode);
        case F4_KEY(256, 1, false, false): return f4_select_marg<256, 1, false>(C, mode);
        case F4_KEY(384, 0, true, false): return f4_select_marg<384, 0, true>(C, mode);
        case F4_KEY(384, 0, false, false): return f4_select_marg<384, 0, false>(C, mode);
        case F4_KEY(256, 0, false, false): return f4_select_marg<256, 0, false>(C, mode);
        case F4_KEY(128, 0, false, false): return f4_select_marg<128, 0, false>(C, mode);
        }
        return nullptr;
    }
    const bool edge = mode == 1;
    switch (key) {
    case F4_KEY(512, 2, true, true): return f4_select_c<512, 2, true, true>(C, edge);
    case F4_KEY(512, 2, false, true): return f4_select_c<512, 2, false, true>(C, edge);
    case F4_KEY(384, 2, false, true): return f4_select_c<384, 2, false, true>(C, edge);
    case F4_KEY(512, 2, true, false): return edge ? nullptr : f4_select_c<512, 2, true, false>(C, false);
    case F4_KEY(384, 2, true, false): return f4_select_c<384, 2, true>(C, edge);
    case F4_KEY(384, 1, false, false): return f4_select_c<384, 1, false>(C, edge);
    case F4_KEY(512, 1, false, false): return edge ? f4_select_c<512, 1, false>(C, true) : nullptr;
    case F4_KEY(256, 2, false, false): return f4_select_c<256, 2, false>(C, edge);
    case F4_KEY(512, 0, true, false): return f4_select_c<512, 0, true>(C, edge);
    case F4_KEY(384, 0, true, false): return f4_select_c<384, 0, true>(C, edge);
    case F4_KEY(384, 0, false, false): return f4_select_c<384, 0, false>(C, edge);
    case F4_KEY(256, 0, false, false): return f4_select_c<256, 0, false>(C, edge);
    case F4_KEY(128, 0, false, false): return f4_select_c<128, 0, false>(C, edge);
    }
    return nullptr;
}

cudaError_t f4_upload_const(const double *Pint, const double *Fint, size_t bytes, cudaStream_t st)
{
    cudaError_t r = cudaMemcpyToSymbolAsync(f4_cP, Pint, bytes, 0, cudaMemcpyDeviceToDevice, st);
    if (r != cudaSuccess || !Fint) return r;
    return cudaMemcpyToSymbolAsync(f4_cF, Fint, bytes, 0, cudaMemcpyDeviceToDevice, st);
}
