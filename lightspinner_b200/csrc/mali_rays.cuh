// mali_rays.cuh -- emergent intensity at user angles from the current state (mali_compute_rays; Lightweaver's
// Context.compute_rays, no reference counterpart).  Included by mali_api.cu only.
//
// I_out[c][la][m] is what the NEXT formal solution would return as I[la][mu] if mu[m] were one of its quadrature angles:
// the opacity and emissivity of the column's current populations, the scattering term of the current J (the J-dagger
// the next formal solution reads), the lines' Voigt profiles evaluated at mu[m] for the up-going direction with
// compute_phi_kernel's expressions (rh_method.py:223-231), and the up sweep of the generic kernel (thermalised lower
// boundary, the last-point quirk of formal_solver.py:137-139).  Always the exact arithmetic form (Arith<false>).
// Nothing but I_out and the optional fault word is written.
#pragma once
#include "mali_device.cuh"

namespace mali {

constexpr int kRaysMaxMu = 64;   // MALI_RAYS_MAX_MU

struct RaysParams {
    int32_t N, Nrays, Nspect, Natom, Ntrans, Lw, ntile, nchunk, nmu, col0, ncol;
    int64_t colStride, popStride, JStride;
    int64_t off_z, off_bbc, off_tab;
    const TileDesc *tiles;
    const SlotDesc *slots;
    const double *alpha, *twohc, *wavelength, *lambda0;   // lambda0 [Ntrans] (nm; lines)
    const double *colconst, *pops, *J;
    const double *aDamp, *vBroad, *vlos;   // [ncol][Ntrans][N], [ncol][Natom][N], [ncol][N]: relative to col0
    double *I;                             // [ncol][Nspect][nmu]
    int32_t *bad;                          // [ncol] or null: bit 1 as in mali_buffers.status
    double mu[kRaysMaxMu], zmu[kRaysMaxMu];   // the angles and 1/mu (host: 1.0 / mu, as mali_model_create forms zmu)
};

// One warp per (column, wavelength tile, mu-chunk), the lane mapping of the formal-solution kernels: ls = lane / Nrays,
// angle = chunk * Nrays + lane % Nrays.  Per lane the up sweep of one ray, in registers: no Gamma, no J, no shared memory
// and no warp-collective operation, so lanes without a ray leave at once.
__global__ void __launch_bounds__(128) rays_kernel(const RaysParams p)
{
    const int lane = threadIdx.x & 31;
    const int64_t w = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int perCol = p.ntile * p.nchunk;
    if (w >= (int64_t)perCol * p.ncol) return;
    const int c = (int)(w / perCol), r = (int)(w - (int64_t)c * perCol);
    const int ti = r / p.nchunk, chunk = r - ti * p.nchunk;
    const TileDesc td = p.tiles[ti];
    const int N = p.N, Nrays = p.Nrays, Nspect = p.Nspect, Lw = p.Lw;
    const int ls = lane / Nrays, m = chunk * Nrays + (lane - ls * Nrays);
    const int la = td.la0 + ls;
    if (ls >= Lw || la >= Nspect || m >= p.nmu) return;

    const int col = p.col0 + c;
    const double *cc = p.colconst + (size_t)col * p.colStride;
    const double *zz = cc + p.off_z;
    const double *tab = cc + p.off_tab + td.recOff;   // this tile's record of depth row 0
    const double *npop = p.pops + (size_t)col * p.popStride;
    const double *Jcol = p.J + (size_t)col * p.JStride;
    const double *aD = p.aDamp + (size_t)c * p.Ntrans * N;
    const double *vB = p.vBroad + (size_t)c * p.Natom * N;
    const double *vL = p.vlos + (size_t)c * N;
    const SlotDesc *slots = p.slots + td.slot0;
    const int nslot = td.nslot;

    const double mu = p.mu[m], zmu = p.zmu[m];
    const double wav = __ldg(p.wavelength + la);
    const double bbc0 = cc[p.off_bbc + 2 * la], bbc1 = cc[p.off_bbc + 2 * la + 1];
    const double sqrtPi = sqrt(kPi);

    Sweep sw;
    double chiProbe = 0.0;
    // s = -1: chi at N-2 first, needed by the thermalised lower boundary (as fs_gamma_kernel's up sweep)
    for (int s = -1; s < N; ++s) {
        const bool probe = s < 0;
        const int k = probe ? N - 2 : N - 1 - s;
        const double *rec = tab + (size_t)k * td.stride;

        // ---- opacity and emissivity at depth k (rh_method.py:601-632), the slots in slot order
        double chiTot = 0.0, etaTot = 0.0;
        for (int tt = 0; tt < nslot; ++tt) {
            const SlotDesc &sd = slots[tt];
            const int lt = la - sd.Nblue;
            const bool act = lt >= 0 && lt < sd.Nlam;
            const int ltC = act ? lt : 0;
            double Vij, Vji, Uji;
            if (sd.isLine) {
                double phi = 0.0;
                if (act) {   // compute_phi_kernel's direction-1 expressions (rh_method.py:223-231) at this angle
                    const double vb = vB[(size_t)sd.atom * N + k];
                    const double l0 = __ldg(p.lambda0 + sd.t);
                    const double rnorm = 1.0 / (sqrtPi * vb);
                    const VoigtPre vp = voigt_pre(aD[(size_t)sd.t * N + k]);
                    const double vd = mu * vL[k] / vb;
                    const double v = (wav - l0) * kCLight / (vb * l0);
                    phi = voigt_H_pre(vp, v + vd) * rnorm;
                }
                Vij = sd.c0 * phi;   // hc/4pi*Bij*phi (rh_method.py:279), as the table holds it
                Vji = sd.c2 * Vij;
                Uji = sd.c1 * Vji;
            } else {
                Vij = act ? __ldg(p.alpha + sd.toff + ltC) : 0.0;
                Vji = act ? __ldg(rec + sd.fOff + ls) : 0.0;         // the record holds g_ij * alpha (rh_method.py:285)
                Uji = __ldg(p.twohc + sd.toff + ltC) * Vji;
            }
            const double ni = npop[(size_t)sd.rowI * N + k], nj = npop[(size_t)sd.rowJ * N + k];
            chiTot += ni * Vij - nj * Vji;
            etaTot += nj * Uji;
        }
        const double *bg = rec + td.bgOff + ls;
        chiTot += __ldg(bg);
        if (probe) {
            chiProbe = chiTot;
            continue;
        }
        const double Jdag = Jcol[(size_t)k * Nspect + la];
        const double rchi = rcp_full(chiTot);
        const double S = div_by(etaTot + __ldg(bg + Lw) + __ldg(bg + 2 * Lw) * Jdag, chiTot, rchi);

        // ---- short characteristic, up-going: formal_solver.py
        double Ik, Psi;
        if (s == 0)
            sw.first(true, zmu, chiTot, S, zz[k], chiProbe, zz[N - 2], bbc0, bbc1, Ik, Psi);
        else
            sw.step(s == N - 1, zmu, chiTot, rchi, S, zz[k], Ik, Psi);
    }
    p.I[((size_t)c * Nspect + la) * p.nmu + m] = sw.Iupw;   // the emergent intensity (rh_method.py:638)
    if (p.bad != nullptr && sw.bad()) atomicOr(p.bad + c, 2);
}

}  // namespace mali
