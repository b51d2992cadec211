// mali_perturb.cuh -- mali_perturb_columns (include/mali_b200.h): a batch of columns that each differ from one set-up
// source column at a single depth, formed without re-forming their other depths.  This is the shape of a response
// function's columns (response_fn.py: T[k] +- 25 K for every k): the background, nStar, C, the profiles and the
// continua's fields are local in depth, so a column is the source's colconst block with one depth re-formed, plus the
// heights (convert_scales' column-mass recurrence is not local) and, for a temperature change in the last two depths,
// the boundary Planck pair.
//
// Every depth re-formation runs the per-point body of the kernel the full set-up runs (mali_kernels.cuh: eos_point,
// background_point, setup_levels_point, setup_gij_point, cont_group_body, MALI_COMPUTE_PHI_BODY) on the column's own
// inputs, so the result carries the bits mali_upload_columns_thermo + mali_background + mali_setup_columns +
// mali_compute_phi produce from those inputs.
#pragma once

#include "mali_kernels.cuh"

namespace mali {

struct PerturbParams {
    int N, Nspect, Lw, sumNlevel, Natom, col0, src;
    int64_t colStride, popStride, JStride, off_bbc, off_tab;
    const int32_t *depth;                   // [ncol] the re-formed depth of each column
    const double *T, *ne, *nHTot, *vturb;   // [ncol][N] the columns' own inputs
    const double *bbc;                      // [ncol][Nspect][2] or null
    const double *pops0, *srcWork, *srcNStar, *srcVBroad;
    double *work, *nStar, *vBroad;          // [ncol][N][kEosWork] (+ [ncol][N] convert_scales tau), [ncol][sumNlevel][N], [ncol][Natom][N]
    double *colconst, *pops, *J;
};

// grid (x, ncol): the source's colconst block, its EOS work rows, nStar and vBroad copied to every column of the range;
// J zeroed (the source was never iterated: the J-dagger fields of its records are zero too); the populations set to pops0
__global__ void perturb_clone_kernel(const PerturbParams p)
{
    const int c = blockIdx.y, col = p.col0 + c;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    // colconst blocks are whole multiples of 16 doubles (mali_model_create), so they copy as double2
    const double2 *s = reinterpret_cast<const double2 *>(p.colconst + (size_t)p.src * p.colStride);
    double2 *d = reinterpret_cast<double2 *>(p.colconst + (size_t)col * p.colStride);
    for (int64_t q = tid; q < p.colStride / 2; q += nth) d[q] = s[q];
    double *Jc = p.J + (size_t)col * p.JStride;
    for (int64_t q = tid; q < p.JStride; q += nth) Jc[q] = 0.0;
    double *n = p.pops + (size_t)col * p.popStride;
    for (int64_t q = tid; q < p.popStride; q += nth) n[q] = p.pops0[q];
    const int64_t nw = (int64_t)p.N * kEosWork, ns = (int64_t)p.sumNlevel * p.N, nv = (int64_t)p.Natom * p.N;
    for (int64_t q = tid; q < nw; q += nth) p.work[(size_t)c * nw + q] = p.srcWork[q];
    for (int64_t q = tid; q < ns; q += nth) p.nStar[(size_t)c * ns + q] = p.srcNStar[q];
    for (int64_t q = tid; q < nv; q += nth) p.vBroad[(size_t)c * nv + q] = p.srcVBroad[q];
}

// one thread per column: the EOS point of its depth (eos_kernel)
__global__ void perturb_eos_kernel(const EosParams P, const PerturbParams p, int ncol)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncol) return;
    eos_point(P, p.T, p.nHTot, p.work, c * p.N + p.depth[c]);
}

// grid (x, ncol), one thread per wavelength: the background fields of the column's depth (background_kernel) and, where
// the caller gives one, the column's boundary Planck pair
__global__ void perturb_background_kernel(const EosParams P, const TileDesc *tiles, const double *wavelength,
                                          const double *ne, const PerturbParams p)
{
    const int c = blockIdx.y;
    const int la = blockIdx.x * blockDim.x + threadIdx.x;
    if (la >= p.Nspect) return;
    background_point(P, tiles, wavelength, p.N, p.Nspect, p.Lw, p.T, ne, p.work, p.colconst, p.colStride, p.off_tab,
                     p.col0, c, la, p.depth[c]);
    if (p.bbc) {
        double *dst = p.colconst + (size_t)(p.col0 + c) * p.colStride + p.off_bbc + 2 * la;
        const double *src = p.bbc + ((size_t)c * p.Nspect + la) * 2;
        dst[0] = src[0];
        dst[1] = src[1];
    }
}

// one thread per (column, atom): LTE populations, C and vBroad of the column's depth (setup_levels_kernel)
template <int NLMAX>
__global__ void perturb_levels_kernel(const AtomLevels A, const PerturbParams p, int64_t off_C, int64_t off_nTotal, int ncol)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= ncol * p.Natom) return;
    const int c = idx / p.Natom, a = idx - c * p.Natom;
    setup_levels_point<NLMAX>(A, p.N, p.T, p.ne, p.vturb, p.colconst, p.colStride, off_C, off_nTotal, p.nStar, p.vBroad,
                              nullptr, p.popStride, p.sumNlevel, p.col0, a, c, p.depth[c]);
}

// grid (continuum, column), threads over the continuum's wavelengths: its g_ij fields at the column's depth
// (setup_gij_kernel)
__global__ void perturb_gij_kernel(const GijCont *conts, const GijTile *gt, const double *wavelength, const double *alpha,
                                   const PerturbParams p)
{
    const GijCont ct = conts[blockIdx.x];
    const int c = blockIdx.y;
    const double hc_k = kHC / (kKBoltzmann * kNmToM);
    double *tab = p.colconst + (size_t)(p.col0 + c) * p.colStride + p.off_tab;
    const double *ns = p.nStar + (size_t)c * p.sumNlevel * p.N;
    const int k = p.depth[c];
    for (int lt = threadIdx.x; lt < ct.Nlam; lt += blockDim.x)
        setup_gij_point(ct, gt, wavelength, alpha, p.N, p.Lw, p.T, ns, tab, hc_k, c, lt, k);
}

// grid (tile with continuum groups, column), one thread per wavelength of the tile: the groups' fields at the column's
// depth (cont_group_kernel), from the g_ij fields perturb_gij_kernel has just written
struct GroupDepthIdx {
    int k;
    __device__ __forceinline__ unsigned tile() const { return blockIdx.x; }
    __device__ __forceinline__ unsigned col() const { return blockIdx.y; }
    __device__ __forceinline__ int first() const { return k * (int)blockDim.x + threadIdx.x; }   // (blockDim.x == Lw)
    __device__ __forceinline__ int end(int, int Lw) const { return (k + 1) * Lw; }
    __device__ __forceinline__ int step() const { return blockDim.x; }
};
__global__ void perturb_group_kernel(const TileDesc *tiles, const SlotDesc *slots, const int32_t *groupTiles,
                                     const double *twohc, const PerturbParams p)
{
    cont_group_body(tiles, slots, groupTiles, twohc, p.N, p.Nspect, p.Lw, p.colconst, p.colStride, p.off_tab, p.col0,
                    GroupDepthIdx{p.depth[blockIdx.y]});
}

// one warp per (line, column): the profile rows and weight fields of the column's depth (compute_phi_kernel)
__global__ void perturb_phi_kernel(const PhiLine *lines, const PhiTile *ptile, const double *wavelength, const double *wlambda,
                                   const double *muz, const double *wmu, int Nrays, int Ntrans, const double *aDamp,
                                   const double *vlos, const PerturbParams p)
{
    // the names MALI_COMPUTE_PHI_BODY reads
    const int N = p.N, Nspect = p.Nspect, Lw = p.Lw, Natom = p.Natom, col0 = p.col0;
    const int64_t colStride = p.colStride, offTab = p.off_tab;
    const double *vBroad = p.vBroad;
    double *colconst = p.colconst;
    const int lane = threadIdx.x & 31;
    const PhiLine ln = lines[blockIdx.x];
    const int c = blockIdx.y;
    const int k = p.depth[c];
    MALI_COMPUTE_PHI_BODY();
}

}  // namespace mali
