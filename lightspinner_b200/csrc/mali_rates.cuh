// mali_rates.cuh -- radiative rates R_ij / R_ji of every transition from the current state (mali_compute_rates;
// Lightweaver's trans.Rij / trans.Rji).  Included by mali_api.cu only.
//
// The rates are the Gamma integrands of fs_gamma_kernel with PsiStar = 0 (rh_method.py:643-681 without the
// approximate-operator terms), integrated over every (wavelength, angle, direction) of the quadrature with the
// intensity the NEXT formal solution would compute: the opacity and emissivity of the current populations, the
// scattering term of the current J, the line profiles already in the records, and the generic kernel's Sweep
// (thermalised lower boundary, the last-point quirk).  Always the exact arithmetic form.
//
// rates_kernel stores per-(tile, slot, depth) partials at the rows of the formal-solution scratch the Gamma partials
// use; rates_finish_kernel sums them per transition in ascending tile order, as gamma_finish_kernel does.  That scratch
// holds nothing between calls (every formal solution rewrites it before reading it), so the call reuses it.
#pragma once
#include "mali_device.cuh"

namespace mali {

struct RatesParams {
    int32_t N, Nrays, Nspect, Lw, ntile, Ntrans, col0, ncol;
    int64_t colStride, popStride, JStride, scratchStride;
    int64_t off_z, off_bbc, off_tab, off_part, upOff;
    const TileDesc *tiles;
    const SlotDesc *slots;
    const double *alpha, *twohc, *wlacont;   // concatenated per-wavelength tables
    const double *zmu, *hw;                  // [Nrays]: 1/muz, 0.5*wmu
    const double *colconst, *pops, *J;
    double *scratch;
    const int32_t *trPartOff, *trPartRows;   // as FinishParams
    double *Rij, *Rji;                       // [ncol][Ntrans][N], relative to col0
    int32_t *bad;                            // [ncol] or null: bit 1 as in mali_buffers.status
};

// One warp per (column, tile, sweep direction), the lane mapping of the formal-solution kernels: ls = lane / Nrays,
// mu = lane % Nrays.  Lanes without a ray stay for the warp reduction and contribute zeros.
__global__ void __launch_bounds__(128) rates_kernel(const RatesParams p)
{
    const int lane = threadIdx.x & 31;
    const int64_t w = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int perCol = 2 * p.ntile;
    if (w >= (int64_t)perCol * p.ncol) return;   // warp-uniform
    const int c = (int)(w / perCol), r = (int)(w - (int64_t)c * perCol);
    const int ti = r >> 1, d = r & 1;
    const TileDesc td = p.tiles[ti];
    const int N = p.N, Nrays = p.Nrays, Nspect = p.Nspect;
    const int ls = lane / Nrays, mu = lane - ls * Nrays;
    const int la = td.la0 + ls;
    const bool valid = (ls < p.Lw) && (la < Nspect);
    const int laC = valid ? la : td.la0;
    const int lsC = valid ? ls : 0;
    const int laneV = valid ? lane : 0;
    const int muC = valid ? mu : 0;

    const int col = p.col0 + c;
    const double *cc = p.colconst + (size_t)col * p.colStride;
    const double *zz = cc + p.off_z;
    const double *tab = cc + p.off_tab + td.recOff;   // this tile's record of depth row 0
    const double *npop = p.pops + (size_t)col * p.popStride;
    const double *Jcol = p.J + (size_t)col * p.JStride;
    double *part = p.scratch + (size_t)col * p.scratchStride + p.off_part + (d ? p.upOff : 0);
    const SlotDesc *slots = p.slots + td.slot0;
    const int nslot = td.nslot;

    const double zmu = p.zmu[muC], hw = p.hw[muC];
    const double bbc0 = cc[p.off_bbc + 2 * laC], bbc1 = cc[p.off_bbc + 2 * laC + 1];
    const double fourPi = 4.0 * kPi;
    const int dk = d ? -1 : 1;
    const int kS = d ? N - 1 : 0;

    Sweep sw;
    double chiProbe = 0.0;
    // s = -1 (up sweep only): chi at kS+dk first, needed by the thermalised lower boundary
    for (int s = (d ? -1 : 0); s < N; ++s) {
        const bool probe = s < 0;
        const int k = probe ? (kS + dk) : (kS + s * dk);
        const double *rec = tab + (size_t)k * td.stride;

        // ---- opacity and emissivity at depth k (rh_method.py:601-632), the slots in slot order
        double chiTot = 0.0, etaTot = 0.0;
        for (int tt = 0; tt < nslot; ++tt) {
            const SlotDesc &sd = slots[tt];
            const int lt = laC - sd.Nblue;
            const bool act = valid && lt >= 0 && lt < sd.Nlam;
            const int ltC = act ? lt : 0;
            double Vij, Vji, Uji;
            if (sd.isLine) {
                Vij = act ? __ldg(rec + sd.vOff + d * td.vDir + laneV) : 0.0;   // hc/4pi*Bij*phi (rh_method.py:279)
                Vji = sd.c2 * Vij;
                Uji = sd.c1 * Vji;
            } else {
                Vij = act ? __ldg(p.alpha + sd.toff + ltC) : 0.0;
                Vji = act ? __ldg(rec + sd.fOff + lsC) : 0.0;                     // g_ij * alpha (rh_method.py:285)
                Uji = __ldg(p.twohc + sd.toff + ltC) * Vji;
            }
            const double ni = npop[(size_t)sd.rowI * N + k], nj = npop[(size_t)sd.rowJ * N + k];
            chiTot += ni * Vij - nj * Vji;
            etaTot += nj * Uji;
        }
        const double *bg = rec + td.bgOff + lsC;
        chiTot += __ldg(bg);
        if (probe) {
            chiProbe = chiTot;
            continue;
        }
        const double Jdag = Jcol[(size_t)k * Nspect + laC];
        const double rchi = rcp_full(chiTot);
        const double S = div_by(etaTot + __ldg(bg + p.Lw) + __ldg(bg + 2 * p.Lw) * Jdag, chiTot, rchi);

        // ---- short characteristic: formal_solver.py
        double Ik, Psi;
        if (s == 0)
            sw.first(d != 0, zmu, chiTot, S, zz[k], chiProbe, zz[kS + dk], bbc0, bbc1, Ik, Psi);
        else
            sw.step(s == N - 1, zmu, chiTot, rchi, S, zz[k], Ik, Psi);

        // ---- the Gamma integrands with PsiStar = 0: row 2 tt is R_ji (Gamma[i][j]), row 2 tt + 1 is R_ij
        for (int c0 = 0; c0 < nslot; c0 += 4) {
            double v[8];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int tt = c0 + q;
                v[2 * q] = 0.0;
                v[2 * q + 1] = 0.0;
                if (tt < nslot) {
                    const SlotDesc &sd = slots[tt];
                    const int lt = laC - sd.Nblue;
                    const bool act = valid && lt >= 0 && lt < sd.Nlam;
                    const int ltC = act ? lt : 0;
                    double Vij, Vji, Uji, wla;
                    if (sd.isLine) {
                        Vij = act ? __ldg(rec + sd.vOff + d * td.vDir + laneV) : 0.0;
                        Vji = sd.c2 * Vij;
                        Uji = sd.c1 * Vji;
                        wla = act ? __ldg(rec + sd.fOff + lsC) : 0.0;              // wlambda*wphi/HC
                    } else {
                        Vij = act ? __ldg(p.alpha + sd.toff + ltC) : 0.0;
                        Vji = act ? __ldg(rec + sd.fOff + lsC) : 0.0;
                        Uji = __ldg(p.twohc + sd.toff + ltC) * Vji;
                        wla = act ? __ldg(p.wlacont + sd.toff + ltC) : 0.0;        // wlambda/lambda/h
                    }
                    const double wlamu = (wla * hw) * fourPi;
                    v[2 * q] = act ? (Uji + Vji * Ik) * wlamu : 0.0;
                    v[2 * q + 1] = act ? (Vij * Ik) * wlamu : 0.0;
                }
            }
            const double tot = reduce_scatter8(v, lane);
            const int e = lane >> 2;   // value index owned by this lane group
            const int tt = c0 + (e >> 1);
            if ((lane & 3) == 0 && tt < nslot) __stcg(part + (size_t)(td.partRow0 + 2 * tt + (e & 1)) * N + k, tot);
        }
    }
    if (valid && sw.bad() && p.bad != nullptr) atomicOr(p.bad + c, 2);
}

// R_ij / R_ji = the partials of a transition summed in ascending tile order, down copy plus up copy, as
// gamma_finish_kernel sums them: deterministic, independent of the batch and the column range.  One thread per
// (column, transition, depth), coalesced over depth.
__global__ void rates_finish_kernel(const RatesParams p)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int t = blockIdx.y;
    const int c = blockIdx.z;
    const int N = p.N;
    if (k >= N) return;
    const double *part = p.scratch + (size_t)(p.col0 + c) * p.scratchStride + p.off_part;
    double sji = 0.0, sij = 0.0;
    for (int q = p.trPartOff[t]; q < p.trPartOff[t + 1]; ++q) {
        const int row = p.trPartRows[q];
        sji += part[(size_t)row * N + k] + part[(size_t)row * N + k + p.upOff];
        sij += part[(size_t)(row + 1) * N + k] + part[(size_t)(row + 1) * N + k + p.upOff];
    }
    const size_t o = ((size_t)c * p.Ntrans + t) * N + k;
    p.Rij[o] = sij;
    p.Rji[o] = sji;
}

}  // namespace mali
