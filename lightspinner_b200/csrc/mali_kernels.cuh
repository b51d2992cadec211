// mali_kernels.cuh -- the generic formal-solution kernel (any number of transitions per tile; runtime loops), the
// finish / statistical-equilibrium / upload kernels and the test hooks.  Included by mali_api.cu only (the
// structure-specialised formal-solution kernels live in mali_fs_spec.cuh / mali_fs_class.cu).
#pragma once
#include "mali_device.cuh"
#include "mali_eos.h"

namespace mali {

// fp64 CUDA-core peak probe for the roofline: 8 independent unfused mul/add chains per thread.
__global__ void fp64_peak_kernel(int iters, double seed, double *out)
{
    double a[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) a[q] = seed + q + threadIdx.x * 1e-9;
    const double m = 1.0000001, c = 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int q = 0; q < 8; ++q) a[q] = __dadd_rn(__dmul_rn(a[q], m), c);
    }
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < 8; ++q) s += a[q];
    if (s == 123.456) out[0] = s;  // keeps the work alive
}

__global__ void exp_hook_kernel(int n, const double *x, double *y)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = exp_m(x[i]);
}

__global__ void div_hook_kernel(int n, const double *a, const double *b, double *q, int *bad)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double r = rcp_full(b[i]);
    q[i] = div_by(a[i], b[i], r);
    bad[i] = div_domain_ok(a[i], b[i], q[i]) ? 0 : 1;
}

// --------------------------------------------------------------------------------------------------------
// Context.formal_sol_gamma_matrices, rh_method.py:595-692, for one (column, tile) per warp.
//
// lane -> (ls = lane / Nrays, mu = lane % Nrays): wavelength la = tile.la0 + ls, angle mu.  Each lane runs the
// downward then the upward recurrence of its ray, one depth point per step; at every point it (1) builds the
// total opacity / source function from the active transitions (uv, rh_method.py:245-288), (2) advances the short
// characteristic, (3) adds its share of J (segmented sum over the Nrays lanes of a wavelength), (4) forms the
// Gamma integrands and reduces them over the 32 lanes.  Per-warp partial sums go to a per-column scratch
// (down sweep: store, up sweep: add) and are combined in fixed order by gamma_finish_kernel -> deterministic.
__global__ void __launch_bounds__(128) fs_gamma_kernel(const FsParams p)
{
    extern __shared__ double smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tslot = (blockIdx.x % p.blocksPerCol) * p.warpsPerBlock + warp;
    const int col = p.col0 + blockIdx.x / p.blocksPerCol;
    if (tslot >= p.nClassTiles) return;
    if (p.done != nullptr && p.done[col] != 0) return;

    const TileDesc td = p.tiles[p.classTiles[tslot]];
    const int N = p.N, Nrays = p.Nrays, Nspect = p.Nspect;
    const int ls = lane / Nrays, mu = lane - ls * Nrays;
    const int la = td.la0 + ls;
    const bool valid = (ls < p.Lw) && (la < Nspect);
    const int laC = valid ? la : td.la0;
    const int muC = valid ? mu : 0;
    const bool leader = valid && (mu == 0);

    // per-lane level accumulators (the reference's atom.chi / atom.U / atom.eta scratch, rh_method.py:464-466)
    double *lvl = smem + (size_t)warp * p.smemPerWarp;
#define CHI_L(d) lvl[((d) * 2 + 0) * 32 + lane]
#define U_L(d) lvl[((d) * 2 + 1) * 32 + lane]
#define ETA_A(a) lvl[(2 * p.Dmax + (a)) * 32 + lane]

    const double *cc = p.colconst + (size_t)col * p.colStride;
    const double *zz = cc + p.off_z;
    const double *tab = cc + p.off_tab + td.recOff;   // this tile's record of depth row 0
    const int lsC = valid ? ls : 0;
    const int laneV = valid ? lane : 0;
    const double *npop = p.pops + (size_t)col * p.popStride;
    double *Jcol = p.J + (size_t)col * p.JStride;
    double *scr = p.scratch + (size_t)col * p.scratchStride;
    double *Jpart = scr + p.off_jpart;
    double *part = scr + p.off_part;
    const SlotDesc *slots = p.slots + td.slot0;
    const int nslot = td.nslot;

    const double zmu = p.zmu[muC], hw = p.hw[muC];
    const double bbc0 = cc[p.off_bbc + 2 * laC], bbc1 = cc[p.off_bbc + 2 * laC + 1];
    const double fourPi = 4.0 * kPi;  // (x*4)*pi == x*(4*pi) exactly: scaling by 4 commutes with rounding

    for (int d = 0; d < 2; ++d) {
        const int dk = d ? -1 : 1;
        const int kS = d ? N - 1 : 0;
        Sweep sw;
        double chiProbe = 0.0;
        // s = -1 (upgoing only): evaluate chi at kS+dk first, needed by the thermalised lower boundary
        for (int s = (d ? -1 : 0); s < N; ++s) {
            const bool probe = s < 0;
            const int k = probe ? (kS + dk) : (kS + s * dk);

            // ---- (1) opacity and emissivity at depth k: rh_method.py:601-632
            double chiTot = 0.0, etaTot = 0.0;
            if (!probe) {
                for (int q = 0; q < td.nlevslot; ++q) {
                    CHI_L(q) = 0.0;
                    U_L(q) = 0.0;
                }
                for (int a = 0; a < p.Natom; ++a) ETA_A(a) = 0.0;
            }
            for (int tt = 0; tt < nslot; ++tt) {
                const SlotDesc &sd = slots[tt];
                const int lt = laC - sd.Nblue;
                const bool act = valid && lt >= 0 && lt < sd.Nlam;
                const int ltC = act ? lt : 0;
                const double *rec = tab + (size_t)k * td.stride;
                double Vij, Vji, Uji;
                if (sd.isLine) {
                    const double phi = act ? __ldg(rec + sd.vOff + d * td.vDir + laneV) : 0.0;
                    Vij = phi;  // the table holds hc/4pi*Bij*phi (rh_method.py:279), folded in at upload
                    Vji = sd.c2 * Vij;
                    Uji = sd.c1 * Vji;
                } else {
                    const double a = act ? __ldg(p.alpha + sd.toff + ltC) : 0.0;
                    Vij = a;
                    Vji = act ? __ldg(rec + sd.fOff + lsC) : 0.0;      // the record holds g_ij * alpha (rh_method.py:285)
                    Uji = __ldg(p.twohc + sd.toff + ltC) * Vji;
                }
                const double ni = npop[(size_t)sd.rowI * N + k], nj = npop[(size_t)sd.rowJ * N + k];
                const double chi_t = ni * Vij - nj * Vji;
                const double eta_t = nj * Uji;
                if (!probe) {
                    CHI_L(sd.lsI) += chi_t;
                    CHI_L(sd.lsJ) -= chi_t;
                    U_L(sd.lsJ) += Uji;
                    ETA_A(sd.atom) += eta_t;
                }
                chiTot += chi_t;
                etaTot += eta_t;
            }
            const size_t kl = (size_t)k * Nspect + laC;
            const double *bg = tab + (size_t)k * td.stride + td.bgOff + lsC;
            chiTot += __ldg(bg);
            if (probe) {
                chiProbe = chiTot;
                continue;
            }
            const double Jdag = Jcol[kl];
            const double rchi = rcp_full(chiTot);
            const double S = div_by(etaTot + __ldg(bg + p.Lw) + __ldg(bg + 2 * p.Lw) * Jdag, chiTot, rchi);

            // ---- (2) short characteristic: formal_solver.py
            const double zk = zz[k];
            double Ik, Psi;
            if (s == 0)
                sw.first(d != 0, zmu, chiTot, S, zk, chiProbe, zz[kS + dk], bbc0, bbc1, Ik, Psi);
            else
                sw.step(s == N - 1, zmu, chiTot, rchi, S, zk, Ik, Psi);

            // ---- (3) J: rh_method.py:640.  Sum over the Nrays lanes of this wavelength in mu order.
            {
                const double x = valid ? hw * Ik : 0.0;
                double sum = x;
                for (int m = 1; m < Nrays; ++m) sum += __shfl_down_sync(0xffffffffu, x, m);
                // down: store the partial; up: complete it.  j_finish_kernel then forms dJ and moves Jpart -> J
                if (leader) __stcg(Jpart + kl + (d ? p.upOff : 0), sum);
            }

            // ---- (4) Gamma integrands: rh_method.py:643-681
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
                        const double *rec = tab + (size_t)k * td.stride;
                        double Vij, Vji, Uji, wla;
                        if (sd.isLine) {
                            const double phi = act ? __ldg(rec + sd.vOff + d * td.vDir + laneV) : 0.0;
                            Vij = phi;
                            Vji = sd.c2 * Vij;
                            Uji = sd.c1 * Vji;
                            wla = act ? __ldg(rec + sd.fOff + lsC) : 0.0;
                        } else {
                            const double a = act ? __ldg(p.alpha + sd.toff + ltC) : 0.0;
                            Vij = a;
                            Vji = act ? __ldg(rec + sd.fOff + lsC) : 0.0;
                            Uji = __ldg(p.twohc + sd.toff + ltC) * Vji;
                            wla = act ? __ldg(p.wlacont + sd.toff + ltC) : 0.0;
                        }
                        const double Ieff = Ik - Psi * ETA_A(sd.atom);
                        const double wlamu = (wla * hw) * fourPi;
                        const double g1 = (Uji + Vji * Ieff) - ((CHI_L(sd.lsI) * Psi) * U_L(sd.lsJ));
                        const double g2 = (Vij * Ieff) - ((CHI_L(sd.lsJ) * Psi) * U_L(sd.lsI));
                        v[2 * q] = act ? g1 * wlamu : 0.0;
                        v[2 * q + 1] = act ? g2 * wlamu : 0.0;
                    }
                }
                const double tot = reduce_scatter8(v, lane);
                const int e = lane >> 2;  // value index owned by this lane group
                const int tt = c0 + (e >> 1);
                if ((lane & 3) == 0 && tt < nslot) {
                    double *dst = part + (size_t)(td.partRow0 + 2 * tt + (e & 1)) * N + k;
                    __stcg(dst + (d ? p.upOff : 0), tot);  // down and up partials are summed by gamma_finish_kernel
                }
            }
        }
        // emergent intensity: rh_method.py:638 (the upgoing value survives)
        if (d == 1 && valid) p.I[(size_t)col * p.IStride + (size_t)la * Nrays + mu] = sw.Iupw;
        if (valid && sw.bad() && p.status != nullptr) atomicOr(p.status + col, 2);
    }

#undef CHI_L
#undef U_L
#undef ETA_A
}

// --------------------------------------------------------------------------------------------------------
// dJ = max |1 - JDag/J| (rh_method.py:705-706) and J <- the new mean intensity the sweeps accumulated in Jpart.
// Elementwise over one column's [Nspace][Nspect] plane; block max -> one atomicMax per block.
struct TileJ {
    int32_t off, stride;   // J-dagger field of the tile's depth-0 record; record stride
};
// (memory-latency bound: 32 registers per thread keep all 64 warps of an SM resident)
__global__ void __launch_bounds__(256, 8)
j_finish_kernel(double *__restrict__ J, int64_t JStride, const double *__restrict__ scratch, int64_t scratchStride,
                                int64_t offJpart, int64_t upOff, double *__restrict__ colconst, int64_t colStride, int64_t offTab,
                                const TileJ *__restrict__ tileJ, int Nspect, int Lw,
                                unsigned long long *dJbits, const int32_t *done, int col0)
{
    const int col = col0 + blockIdx.y;
    if (done != nullptr && done[col] != 0) return;
    double *Jc = J + (size_t)col * JStride;
    double *tab = colconst + (size_t)col * colStride + offTab;
    const double *Jn = scratch + (size_t)col * scratchStride + offJpart;
    unsigned long long b = 0ull;
    const int N = (int)(JStride / Nspect);
    const int jw = (Lw + 3) & ~3;                              // width of the J-dagger field of a record
    const int ntile = (Nspect + Lw - 1) / Lw;
    for (int k = blockIdx.x; k < N; k += gridDim.x) {          // one depth row at a time: no 64-bit divisions
        const int64_t q0 = (int64_t)k * Nspect;
        for (int idx = threadIdx.x; idx < ntile * jw; idx += blockDim.x) {
            const int ti = idx / jw, ls = idx - ti * jw;
            const int la = ti * Lw + ls;
            double jn = 0.0;
            if (ls < Lw && la < Nspect) {
                jn = Jn[q0 + la] + Jn[q0 + la + upOff];  // down-sweep + up-sweep sums, rh_method.py:640
                const unsigned long long v = absbits(1.0 - Jc[q0 + la] / jn);
                b = v > b ? v : b;
                Jc[q0 + la] = jn;
            }
            // the copy the next formal solution reads (J-dagger): a field of the tile-major records, so that it
            // arrives with the record's TMA and the depth loop holds no global loads; whole sectors are written
            const TileJ tj = tileJ[ti];
            tab[tj.off + (size_t)k * tj.stride + ls] = jn;
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, b, off);
        b = o > b ? o : b;
    }
    __shared__ unsigned long long wmax[8];
    if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = b;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) b = wmax[w] > b ? wmax[w] : b;
        atomicMax(dJbits + col, b);
    }
}

// --------------------------------------------------------------------------------------------------------
// Gamma = C + sum of the per-tile partials in ascending tile order, then the diagonal (rh_method.py:587-590,
// 698-703).  One thread per (column, atom, depth); coalesced over depth.
__global__ void gamma_finish_kernel(const FinishParams p)
{
    // block = 32 depth points x 8 "pair lanes": the transitions of an atom are dealt to the pair lanes by their
    // (i, j) entry, so every Gamma entry has one owner (deterministic order) and the sums of different transitions
    // run in parallel; the diagonal is formed after a block barrier
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = threadIdx.y, ny = blockDim.y;
    const int a = blockIdx.y;
    const int col = p.col0 + blockIdx.z;
    if (p.done != nullptr && p.done[col] != 0) return;
    const bool on = k < p.N;
    const int N = p.N;
    const int NL = p.Nlevel[a];
    const double *C = p.colconst + (size_t)col * p.colStride + p.off_C + (size_t)p.g2Off[a] * N;
    double *G = p.Gamma + (size_t)col * p.gammaStride + (size_t)p.g2Off[a] * N;
    const double *part = p.scratch + (size_t)col * p.scratchStride + p.off_part;

    if (on)
        for (int e = y; e < NL * NL; e += ny) G[(size_t)e * N + k] = 0.0 + C[(size_t)e * N + k];
    __syncthreads();
    if (on)
        for (int t = 0; t < p.Ntrans; ++t) {
            const int32_t *tr = p.trans + 6 * t;
            if (tr[0] != a) continue;
            const int i = tr[1], j = tr[2];
            if ((i * NL + j) % ny != y) continue;
            double sij = 0.0, sji = 0.0;
            for (int r = p.trPartOff[t]; r < p.trPartOff[t + 1]; ++r) {
                const int row = p.trPartRows[r];
                sij += part[(size_t)row * N + k] + part[(size_t)row * N + k + p.upOff];
                sji += part[(size_t)(row + 1) * N + k] + part[(size_t)(row + 1) * N + k + p.upOff];
            }
            G[((size_t)i * NL + j) * N + k] += sij;
            G[((size_t)j * NL + i) * N + k] += sji;
        }
    __syncthreads();
    if (on)
        for (int i = y; i < NL; i += ny) {   // rh_method.py:698-703: zero the diagonal, then minus the column sum
            double GamDiag = 0.0;
            for (int l = 0; l < NL; ++l) GamDiag += (l == i) ? 0.0 : G[((size_t)l * NL + i) * N + k];
            G[((size_t)i * NL + i) * N + k] = -GamDiag;
        }
}

// --------------------------------------------------------------------------------------------------------
// Context.stat_equil (rh_method.py:710-745): one thread per (column, atom, depth) solves the Nlevel x Nlevel
// system Gamma' n = nTotal e_iEliminate by LU with partial pivoting, then two rounds of iterative refinement
// with the residual accumulated in double-double (the systems have cond ~ 1e6..1e9, SURVEY.md 7.3-1: the aim is
// to sit closer to the exact solution than LAPACK does, not to clone its rounding).
template <int NLMAX>
__global__ void stat_equil_kernel(const FinishParams p)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int a = blockIdx.y;
    const int col = p.col0 + blockIdx.z;
    if (k >= p.N) return;
    if (p.done != nullptr && p.done[col] != 0) return;
    if (p.iter != nullptr && p.iter[col] < p.iterMin) return;
    const int N = p.N;
    const int NL = p.Nlevel[a];
    const double *G = p.Gamma + (size_t)col * p.gammaStride + (size_t)p.g2Off[a] * N + k;
    double *n = p.pops + (size_t)col * p.popStride + (size_t)p.lvlOff[a] * N;
    const double nTot = p.colconst[(size_t)col * p.colStride + p.off_nTotal + (size_t)a * N + k];

    // iEliminate = argmax(n[:, k]) (first maximum, rh_method.py:727)
    int iEl = 0;
    double nmax = n[k];
    for (int l = 1; l < NL; ++l) {
        const double v = n[(size_t)l * N + k];
        if (v > nmax) {
            nmax = v;
            iEl = l;
        }
    }
    double *ngH = nullptr;   // Ng acceleration: this column's history block, shifted to this atom's first level
    if (p.ngHist != nullptr) {
        ngH = p.ngHist + (size_t)col * p.ngStride + (size_t)p.lvlOff[a] * N + k;
        double *snap = ngH + (size_t)p.ngRing * p.popStride;   // n as the solve found it (dPops of an extrapolation)
        for (int l = 0; l < NL; ++l) snap[(size_t)l * N] = n[(size_t)l * N + k];
    }
    double x[NLMAX];
    if (!solve_stat_equil_any<NLMAX>(G, N, NL, iEl, nTot, x)) {
        atomicOr(p.status + col, 1);  // the reference would raise LinAlgError here
        return;
    }
    unsigned long long db = 0ull;
    for (int l = 0; l < NL; ++l) {
        const double nOld = n[(size_t)l * N + k];
        const unsigned long long b = absbits(1.0 - nOld / x[l]);
        db = b > db ? b : db;
        n[(size_t)l * N + k] = x[l];
    }
    if (ngH != nullptr) {    // push the solution into the ring (the newest slot; ngNse already counts this solve)
        double *slot = ngH + (size_t)((p.ngNse[col] - 1) % p.ngRing) * p.popStride;
        for (int l = 0; l < NL; ++l) slot[(size_t)l * N] = x[l];
    }
    atomicMax(p.dPopsBits + col, db);
}

// --------------------------------------------------------------------------------------------------------
// Ng acceleration of the population iteration (Auer 1987), per column and active atom.  The vector is the atom's
// populations x = n[level][k] flattened over (level, depth); x0 is the newest solved vector, x1, x2, ... the older
// ones.  With d_i = x_i - x_{i+1} (i = 0..order) and w = 1 / x0^2 elementwise, solve the order x order system
//     A c = b,   A_ij = sum w (d0 - d_{i+1})(d0 - d_{j+1}),   b_i = sum w d0 (d0 - d_{i+1}),
// and form x* = (1 - sum c) x0 + sum_i c_i x_{i+1}.  x* is accepted only if A is non-singular and every entry of x* is
// finite and > 0.  The sums are block-wide: a fixed element-to-thread assignment, a warp shuffle tree, then the
// warps' sums added in warp order -- no atomics, so the result does not depend on the batch or the column range.
// ng_solve_block is shared by ng_kernel and the test hook (mali_ng_hook).
constexpr int kNgThreads = 256;

__host__ __device__ __forceinline__ bool ng_due(int nse, int order, int delay, int period)
{
    return nse > delay && nse >= order + 2 && (nse - delay) % period == 0;
}

template <int ORDER>
__device__ __forceinline__ double ng_value(const double *const *x, const double *c, double keep, int64_t idx)
{
    double v = keep * x[0][idx];
#pragma unroll
    for (int i = 0; i < ORDER; ++i) v = v + c[i] * x[i + 1][idx];
    return v;
}

// Block-wide (kNgThreads threads, every one of them must call it): the coefficients c[ORDER] and 1 - sum c of the
// extrapolation of the vectors x[0..ORDER+1] (length n), and whether x* is accepted.  The result is block-uniform.
template <int ORDER>
__device__ bool ng_solve_block(const double *const *x, int64_t n, double *c, double *keep)
{
    constexpr int kA = ORDER * (ORDER + 1) / 2, kS = kA + ORDER;   // upper triangle of A, then b
    __shared__ double wsum[kNgThreads / 32][kS];
    double s[kS];
#pragma unroll
    for (int q = 0; q < kS; ++q) s[q] = 0.0;
    for (int64_t idx = threadIdx.x; idx < n; idx += kNgThreads) {
        double d[ORDER + 1], e[ORDER];
#pragma unroll
        for (int i = 0; i <= ORDER; ++i) d[i] = x[i][idx] - x[i + 1][idx];
        const double x0 = x[0][idx];
        const double w = 1.0 / (x0 * x0);
#pragma unroll
        for (int i = 0; i < ORDER; ++i) e[i] = d[0] - d[i + 1];
        int q = 0;
#pragma unroll
        for (int i = 0; i < ORDER; ++i) {
            const double we = w * e[i];
#pragma unroll
            for (int j = i; j < ORDER; ++j) s[q++] += we * e[j];
        }
        const double wd = w * d[0];
#pragma unroll
        for (int i = 0; i < ORDER; ++i) s[kA + i] += wd * e[i];
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < kS; ++q) {
        double v = s[q];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
        if (lane == 0) wsum[warp][q] = v;
    }
    __syncthreads();
    // every thread adds the warps' sums in the same order and solves the same small system: no broadcast needed
    double M[ORDER][ORDER + 1];
    {
        double t[kS];
#pragma unroll
        for (int q = 0; q < kS; ++q) {
            t[q] = wsum[0][q];
            for (int w = 1; w < kNgThreads / 32; ++w) t[q] += wsum[w][q];
        }
        int q = 0;
#pragma unroll
        for (int i = 0; i < ORDER; ++i)
#pragma unroll
            for (int j = i; j < ORDER; ++j) {
                M[i][j] = t[q];
                M[j][i] = t[q];
                ++q;
            }
#pragma unroll
        for (int i = 0; i < ORDER; ++i) M[i][ORDER] = t[kA + i];
    }
    // Gaussian elimination with partial pivoting; an exactly zero (or non-finite) pivot is a singular system
    bool ok = true;
#pragma unroll
    for (int col = 0; col < ORDER; ++col) {
        int piv = col;
#pragma unroll
        for (int r = col + 1; r < ORDER; ++r)
            if (fabs(M[r][col]) > fabs(M[piv][col])) piv = r;
        if (piv != col)
#pragma unroll
            for (int j = 0; j <= ORDER; ++j) {
                const double tmp = M[col][j];
                M[col][j] = M[piv][j];
                M[piv][j] = tmp;
            }
        const double pv = M[col][col];
        if (!(fabs(pv) > 0.0) || !isfinite(pv)) ok = false;
#pragma unroll
        for (int r = col + 1; r < ORDER; ++r) {
            const double f = M[r][col] / pv;
#pragma unroll
            for (int j = col; j <= ORDER; ++j) M[r][j] = M[r][j] - f * M[col][j];
        }
    }
    double csum = 0.0;
#pragma unroll
    for (int i = ORDER - 1; i >= 0; --i) {
        double v = M[i][ORDER];
#pragma unroll
        for (int j = i + 1; j < ORDER; ++j) v = v - M[i][j] * c[j];
        c[i] = v / M[i][i];
    }
#pragma unroll
    for (int i = 0; i < ORDER; ++i) {
        csum = csum + c[i];
        if (!isfinite(c[i])) ok = false;
    }
    *keep = 1.0 - csum;
    // positivity / finiteness vote over every entry of x*
    bool good = ok;
    if (ok)
        for (int64_t idx = threadIdx.x; idx < n; idx += kNgThreads) {
            const double v = ng_value<ORDER>(x, c, *keep, idx);
            good = good && v > 0.0 && isfinite(v);
        }
    return __syncthreads_and(good) != 0;
}

struct NgParams {
    int32_t N, Natom, col0, order, delay, period, ring, iterMin;
    int64_t popStride, histStride;
    const int32_t *Nlevel, *lvlOff;
    double *pops, *hist;           // hist: per column ring slots, the snapshot, then one dPops bit pattern per atom
    int32_t *nse, *accepted;       // [ncol], [ncol][Natom]
    double *dPops;
    const int32_t *status, *done, *iter;   // done / iter may be null (per-call entry point)
};

__device__ __forceinline__ bool ng_column_active(const NgParams &p, int col)
{
    if (p.done != nullptr && p.done[col] != 0) return false;        // as stat_equil_kernel: not solved this iteration
    if (p.iter != nullptr && p.iter[col] < p.iterMin) return false;
    if (p.status[col] != 0) return false;                           // a singular system: the column is failing
    return ng_due(p.nse[col], p.order, p.delay, p.period);
}

// One block per (atom, column): the extrapolation, the write-back into n and the newest ring slot, and the atom's
// max |1 - n_start / n_final| (bit pattern, combined over the atoms by ng_dpops_kernel).
template <int ORDER>
__global__ void __launch_bounds__(kNgThreads) ng_kernel(const NgParams p)
{
    const int a = blockIdx.x, col = p.col0 + blockIdx.y;
    if (!ng_column_active(p, col)) return;
    const int R = ORDER + 2, s = p.nse[col];
    const int64_t off = (int64_t)p.lvlOff[a] * p.N, len = (int64_t)p.Nlevel[a] * p.N;
    double *H = p.hist + (size_t)col * p.histStride;
    const double *x[ORDER + 2];
#pragma unroll
    for (int i = 0; i < R; ++i) x[i] = H + (size_t)((s - 1 - i) % R) * p.popStride + off;
    double c[ORDER], keep;
    const bool acc = ng_solve_block<ORDER>(x, len, c, &keep);
    double *n = p.pops + (size_t)col * p.popStride + off;
    double *newest = H + (size_t)((s - 1) % R) * p.popStride + off;
    const double *snap = H + (size_t)R * p.popStride + off;
    unsigned long long db = 0ull;
    for (int64_t idx = threadIdx.x; idx < len; idx += kNgThreads) {
        double v = n[idx];
        if (acc) {
            v = ng_value<ORDER>(x, c, keep, idx);   // reads x0 = newest[idx] before this thread overwrites it
            n[idx] = v;
            newest[idx] = v;
        }
        const unsigned long long b = absbits(1.0 - snap[idx] / v);
        db = b > db ? b : db;
    }
#pragma unroll
    for (int off2 = 16; off2 > 0; off2 >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, db, off2);
        db = o > db ? o : db;
    }
    __shared__ unsigned long long wmax[kNgThreads / 32];
    if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = db;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kNgThreads / 32; ++w) db = wmax[w] > db ? wmax[w] : db;
        H[(size_t)(R + 1) * p.popStride + a] = __longlong_as_double((long long)db);
        if (acc) p.accepted[(size_t)col * p.Natom + a] += 1;
    }
}

// dPops of the iteration for the columns that were extrapolated: the max over the atoms, in atom order.
__global__ void ng_dpops_kernel(const NgParams p, int ncol)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncol) return;
    const int col = p.col0 + c;
    if (!ng_column_active(p, col)) return;
    const double *part = p.hist + (size_t)col * p.histStride + (size_t)(p.ring + 1) * p.popStride;
    unsigned long long db = 0ull;
    for (int a = 0; a < p.Natom; ++a) {
        const unsigned long long b = (unsigned long long)__double_as_longlong(part[a]);
        db = b > db ? b : db;
    }
    p.dPops[col] = __longlong_as_double((long long)db);
}

// Test hook: one extrapolation of hist [ORDER+2][n] (newest first) -> out (x* if accepted, else x0).
template <int ORDER>
__global__ void __launch_bounds__(kNgThreads) ng_hook_kernel(int64_t n, const double *hist, double *out, int32_t *accepted)
{
    const double *x[ORDER + 2];
#pragma unroll
    for (int i = 0; i < ORDER + 2; ++i) x[i] = hist + (size_t)i * n;
    double c[ORDER], keep;
    const bool acc = ng_solve_block<ORDER>(x, n, c, &keep);
    for (int64_t idx = threadIdx.x; idx < n; idx += kNgThreads) out[idx] = acc ? ng_value<ORDER>(x, c, keep, idx) : x[0][idx];
    if (threadIdx.x == 0) *accepted = acc ? 1 : 0;
}

// --------------------------------------------------------------------------------------------------------
// Test hook: piecewise_linear_1d for independent rays, one thread per ray, same Sweep code as the fused kernel.
__global__ void sweep_hook_kernel(int N, int nray, const double *z, const double *muz, const int32_t *toFrom,
                                  const double *bbc0, const double *bbc1, const double *chi, const double *S,
                                  double *I, double *Psi)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nray) return;
    const bool up = toFrom[r] != 0;
    const double zmu = 1.0 / muz[r];
    const int dk = up ? -1 : 1, kS = up ? N - 1 : 0;
    const double *c = chi + (size_t)r * N, *s = S + (size_t)r * N;
    Sweep sw;
    double Ik, Pk;
    sw.first(up, zmu, c[kS], s[kS], z[kS], c[kS + dk], z[kS + dk], bbc0[r], bbc1[r], Ik, Pk);
    I[(size_t)r * N + kS] = Ik;
    Psi[(size_t)r * N + kS] = Pk;
    for (int q = 1; q < N; ++q) {
        const int k = kS + q * dk;
        sw.step(q == N - 1, zmu, c[k], rcp_full(c[k]), s[k], z[k], Ik, Pk);
        I[(size_t)r * N + k] = Ik;
        Psi[(size_t)r * N + k] = Pk;
    }
}

// Test hook: ComputationalTransition.uv from the packed device tables of one column.
__global__ void uv_hook_kernel(const FsParams p, int col, SlotDesc sd, int recOff, int stride, int vDir, int la, int ls,
                               int mu, int d, double *Uji, double *Vij, double *Vji)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= p.N) return;
    const double *rec = p.colconst + (size_t)col * p.colStride + p.off_tab + (size_t)k * stride + recOff;
    const int lt = la - sd.Nblue;
    double vij, vji, uji;
    if (sd.isLine) {
        vij = rec[sd.vOff + d * vDir + ls * p.Nrays + mu];  // hc/4pi*Bij*phi
        vji = sd.c2 * vij;
        uji = sd.c1 * vji;
    } else {
        vij = p.alpha[sd.toff + lt];
        vji = rec[sd.fOff + ls];            // g_ij * alpha, one IEEE multiply folded in at upload
        uji = p.twohc[sd.toff + lt] * vji;
    }
    Uji[k] = uji;
    Vij[k] = vij;
    Vji[k] = vji;
}

// --------------------------------------------------------------------------------------------------------
// Upload path: the host pack is a plain concatenation of the reference's depth-contiguous arrays; pack_tiles_kernel
// gathers it into the tile-major records (see mali_types.cuh).  32 x 32 tiles through shared memory: reads are
// coalesced along depth (the source's contiguous axis), writes along the record (the destination's).
struct PackSlot {
    int32_t isLine, Nblue, Nlam, lineIdx, toff, pad;
    int64_t srcOff;   // host pack: lines phi[Nlam][Nrays][2][N]; continua g_ij[Nlam][N]
    int64_t wphiOff;  // host pack: wphi[N] of the line
    double c0;        // hc/4pi*Bij
};
struct PackTile {
    int32_t recOff, recSize, la0, nslot, slot0, vb, jw, sf;  // vb: one direction's Vij rows; jw: J-dagger field; sf: all fields
};
struct PackChunk {
    int32_t tile, e0;  // 32 consecutive record elements of one tile
};

__global__ void pack_tiles_kernel(const PackChunk *chunks, const PackTile *tiles, const PackSlot *slots,
                                  const double *wlambda, const double *alpha, int N, int Nrays, int Nspect, int Lw, const double *staging,
                                  int64_t hpStride, int64_t hpBgChi, int64_t hpBgEta, int64_t hpBgSca, double *colconst,
                                  int64_t colStride, int64_t offTab, int col0, int skipPhi)
{
    __shared__ double tile[32][33];
    const PackChunk ch = chunks[blockIdx.x];
    const PackTile pt = tiles[ch.tile];
    // a chunk of Vij rows only: compute_phi_kernel writes those rows whole
    if (skipPhi && (ch.e0 + 32 <= pt.vb || (ch.e0 >= pt.vb + pt.sf))) return;
    const double *src = staging + (size_t)blockIdx.z * hpStride;
    double *dst = colconst + (size_t)(col0 + blockIdx.z) * colStride + offTab + pt.recOff;
    const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
    const int k = blockIdx.y * 32 + tx;
    for (int q = ty; q < 32; q += 8) {
        const int e = ch.e0 + q;
        double v = 0.0;
        if (e < pt.recSize && k < N) {
            const bool inV0 = e < pt.vb, inV1 = e >= pt.vb + pt.sf;
            if (inV0 || inV1) {  // Vij rows: direction 0 before the fields, direction 1 after them
                const int d = inV1 ? 1 : 0;
                const int ev = inV1 ? e - pt.vb - pt.sf : e;
                const int j = ev / kVRow, idx = ev % kVRow;
                const int ls = idx / Nrays, mu = idx - ls * Nrays;
                int sq = -1;
                for (int u = 0; u < pt.nslot; ++u)
                    if (slots[pt.slot0 + u].isLine && slots[pt.slot0 + u].lineIdx == j) sq = u;
                if (sq >= 0 && ls < Lw && !skipPhi) {   // skipPhi: compute_phi_kernel fills the line entries
                    const PackSlot ps = slots[pt.slot0 + sq];
                    const int la = pt.la0 + ls, lt = la - ps.Nblue;
                    if (la < Nspect && lt >= 0 && lt < ps.Nlam)
                        v = ps.c0 * src[ps.srcOff + ((size_t)(lt * Nrays + mu) * 2 + d) * N + k];
                }
            } else if (e >= pt.vb + pt.jw) {  // (the J-dagger field at the head of the fields starts as zeros)
                const int ef = e - pt.vb - pt.jw;
                const int f = ef / Lw, ls = ef - f * Lw;
                const int la = pt.la0 + ls;
                const int laClamp = la < Nspect ? la : Nspect - 1;
                if (f < 3) {
                    if (skipPhi < 3)        // (3: background_kernel forms chi / eta / sca on the device)
                        v = src[(f == 0 ? hpBgChi : (f == 1 ? hpBgEta : hpBgSca)) + (size_t)laClamp * N + k];
                } else if (f - 3 < pt.nslot) {
                    const PackSlot ps = slots[pt.slot0 + f - 3];
                    const int lt = la - ps.Nblue;
                    if (la < Nspect && lt >= 0 && lt < ps.Nlam) {
                        if (ps.isLine) {  // wla = wlambda(lt) * wphi[k] / HC   (rh_method.py:451)
                            if (!skipPhi) v = wlambda[ps.toff + lt] * src[ps.wphiOff + k] / kHC;
                        } else if (skipPhi < 2)     // (2: setup_gij_kernel forms the continua's fields on the device)
                            v = src[ps.srcOff + (size_t)lt * N + k] * alpha[ps.toff + lt];   // Vji = g_ij * alpha, rh_method.py:285
                    }
                }
            }
        }
        tile[q][tx] = v;
    }
    __syncthreads();
    for (int q = ty; q < 32; q += 8) {
        const int kk = blockIdx.y * 32 + q, e = ch.e0 + tx;
        if (kk < N && e < pt.recSize) dst[(size_t)kk * pt.recSize + e] = tile[tx][q];
    }
}

// --------------------------------------------------------------------------------------------------------
// ComputationalTransition.compute_phi (rh_method.py:198-243) on the device.  One warp per (column, line, depth);
// the lanes are the (wavelength, angle) pairs of one tile in the record's own lane order, so each tile's two Vij
// rows (down / up direction) are written as whole 256-byte rows.  The warp walks the tiles the line spans,
// evaluates the Voigt profile (mali_voigt.h) for both directions, accumulates the normalisation wPhi (:233; a fixed
// shuffle tree instead of the reference's sequential sum) and finally writes the wavelength-weight fields
// wlambda*wphi/HC (:451) of its depth row.
struct PhiLine {
    int32_t t, atom, Nblue, Nlam, toff, tile0, tab0, ntile;  // tab0: first entry of the per-tile tables below
    double lambda0, c0;                                      // line centre (nm); hc/4pi*Bij
};
struct PhiTile {
    int32_t v0, vDir, f, stride;   // depth-0 offsets of the line's direction-0 Vij row and of its weight field; distance
};                                 // to the direction-1 row; record stride of the tile
// The body of compute_phi_kernel from the line, depth and column on (`ln`, `k`, `c`, `lane` and the kernel's parameters
// in scope), shared with the depth re-formation of mali_perturb_columns (mali_perturb.cuh).  A macro rather than an
// inlined function: every function form of it changed the instruction order of the kernel (the loop over the weight
// fields), whose SASS is kept byte for byte.
#define MALI_COMPUTE_PHI_BODY()                                                                                       \
    do {                                                                                                              \
    const double ad = aDamp[((size_t)c * Ntrans + ln.t) * N + k];                                                     \
    const double vb = vBroad[((size_t)c * Natom + ln.atom) * N + k];                                                  \
    const double vl = vlos[(size_t)c * N + k];                                                                        \
    double *tab = colconst + (size_t)(col0 + c) * colStride + offTab;                                                 \
    const int ls = lane / Nrays, mu = lane - ls * Nrays;                                                              \
    const bool lane_on = ls < Lw;                                                                                     \
    const double sqrtPi = sqrt(kPi);                                                                                  \
    const double rnorm = 1.0 / (sqrtPi * vb);                                                                         \
    const VoigtPre vp = voigt_pre(ad);   /* the damping-only part of the Voigt evaluation, once per (line, depth) */  \
    const double vd = lane_on ? muz[mu] * vl / vb : 0.0;   /* :223 */                                                 \
    const double wm = lane_on ? wmu[mu] : 0.0;                                                                        \
    double wPhi = 0.0;                                                                                                \
    for (int j = 0; j < ln.ntile; ++j) {                                                                              \
        const int la = (ln.tile0 + j) * Lw + ls, lt = la - ln.Nblue;                                                  \
        const bool on = lane_on && lt >= 0 && lt < ln.Nlam && la < Nspect;                                            \
        double p0 = 0.0, p1 = 0.0;                                                                                    \
        if (on) {                                                                                                     \
            const double v = (wavelength[la] - ln.lambda0) * kCLight / (vb * ln.lambda0);   /* :225 */                \
            p0 = voigt_H_pre(vp, v - vd) * rnorm;   /* :229-231 */                                                    \
            p1 = voigt_H_pre(vp, v + vd) * rnorm;                                                                     \
            wPhi += (p0 + p1) * ((wlambda[ln.toff + lt] * 0.5) * wm);   /* :227, :233 */                              \
        }                                                                                                             \
        const PhiTile pt = ptile[ln.tab0 + j];                                                                        \
        double *v0 = tab + pt.v0 + (size_t)k * pt.stride;                                                             \
        v0[lane] = ln.c0 * p0;   /* whole rows, zero where the line is not active */                                  \
        v0[pt.vDir + lane] = ln.c0 * p1;                                                                              \
    }                                                                                                                 \
    _Pragma("unroll")                                                                                                 \
    for (int off = 16; off > 0; off >>= 1) wPhi += __shfl_xor_sync(0xffffffffu, wPhi, off);                           \
    const double wphi = 1.0 / wPhi;   /* :235 */                                                                      \
    for (int j = 0; j < ln.ntile; ++j) {                                                                              \
        if (lane < Lw) {                                                                                              \
            const int la = (ln.tile0 + j) * Lw + lane, lt = la - ln.Nblue;                                            \
            const bool on = lt >= 0 && lt < ln.Nlam && la < Nspect;                                                   \
            const PhiTile pt = ptile[ln.tab0 + j];                                                                    \
            tab[pt.f + (size_t)k * pt.stride + lane] = on ? wlambda[ln.toff + lt] * wphi / kHC : 0.0;   /* :451 */    \
        }                                                                                                             \
    }                                                                                                                 \
    } while (0)
__global__ void compute_phi_kernel(const PhiLine *lines, const PhiTile *ptile, const double *wavelength, const double *wlambda,
                                   const double *muz, const double *wmu, int N, int Nrays, int Nspect, int Lw, int Ntrans,
                                   int Natom, const double *aDamp, const double *vBroad, const double *vlos,
                                   double *colconst, int64_t colStride, int64_t offTab, int col0)
{
    const int lane = threadIdx.x & 31;
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= N) return;
    const PhiLine ln = lines[blockIdx.y];
    const int c = blockIdx.z;                      // column inside the call's inputs
    MALI_COMPUTE_PHI_BODY();
}

// --------------------------------------------------------------------------------------------------------
// Per-column set-up on the device (SURVEY.md 8f rank 3): LTE populations (lte_pops, atomic_set.py:105-145), collisional
// rates (compute_collisions, rh_method.py:474-487 over collisional_rates.py:36-96), Doppler widths (v_broad,
// atomic_model.py:241-245) and the continua's g_ij (rh_method.py:453-454) from T, ne, nTotal, vturb of each column.
struct AtomLevels {     // model-level data, device arrays concatenated over the atoms' levels
    const int32_t *Nlevel, *lvlOff, *g2Off;   // [Natom], [Natom+1], [Natom+1]
    const double *dE, *gi0, *nDebye, *g;      // E_SI[l]-E_SI[0]; g[l]/g[0]; Debye shift count; g[l]
    const int32_t *dZ;                        // stage[l]-stage[0]
    const double *vTherm;                     // [Natom]
    const int32_t *coll;                      // [Ncoll][8]: atom, kind, i, j, table points, knot offset, coefficient offset, cubic
    const double *knots, *coef, *fill, *par;
    double c1, c2;                            // atomic_set.py:107, :111 (evaluated on the host with the reference's expressions)
    int32_t Ncoll, Natom;
};

// the table interpolant of collisional_rates.py:15-19 -- scipy interp1d: constant fill values outside the table; inside,
// a cubic not-a-knot B-spline (make_interp_spline) evaluated with de Boor's recurrence exactly as scipy's
// _bspl.evaluate_spline does (same operations, same order), or the linear form for a 2-point table
__device__ __forceinline__ double coll_table(const AtomLevels &A, int c, double x)
{
    const int32_t *cd = A.coll + 8 * c;
    const int n = cd[4];
    const double *t = A.knots + cd[5], *cf = A.coef + cd[6];
    if (!cd[7]) {     // linear: interp1d._call_linear
        if (x < t[0]) return A.fill[2 * c];
        if (x > t[n - 1]) return A.fill[2 * c + 1];
        int hi = 1;
        while (hi < n - 1 && t[hi] < x) ++hi;            // searchsorted(x, x_new) clipped to [1, n-1]
        const double slope = (cf[hi] - cf[hi - 1]) / (t[hi] - t[hi - 1]);
        return slope * (x - t[hi - 1]) + cf[hi - 1];
    }
    // knots t[0 .. n+3]; table range [t[3], t[n]]
    if (x < t[3]) return A.fill[2 * c];
    if (x > t[n]) return A.fill[2 * c + 1];
    int ell = 3;
    while (ell < n - 1 && x >= t[ell + 1]) ++ell;        // t[ell] <= x < t[ell+1]; the right end belongs to the last interval
    double h[4], hh[4];
    h[0] = 1.0;
    for (int j = 1; j <= 3; ++j) {
        for (int q = 0; q < j; ++q) hh[q] = h[q];
        h[0] = 0.0;
        for (int q = 1; q <= j; ++q) {
            const double xb = t[ell + q], xa = t[ell + q - j];
            if (xb == xa) {
                h[q] = 0.0;
                continue;
            }
            const double w = hh[q - 1] / (xb - xa);
            h[q - 1] += w * (xb - x);
            h[q] = w * (x - xa);
        }
    }
    double out = 0.0;
    for (int a = 0; a <= 3; ++a) out += cf[ell + a - 3] * h[a];
    return out;
}

// atom a at depth k of column c of the call's inputs (column col0 + c of colconst / pops); shared with
// mali_perturb_columns (mali_perturb.cuh)
template <int NLMAX>
__device__ __forceinline__ void setup_levels_point(const AtomLevels &A, int N, const double *T, const double *ne,
                                                   const double *vturb, double *colconst, int64_t colStride, int64_t off_C,
                                                   int64_t off_nTotal, double *nStar, double *vBroad, double *pops,
                                                   int64_t popStride, int sumNlevel, int col0, int a, int c, int k)
{
    const double t = T[(size_t)c * N + k], xne = ne[(size_t)c * N + k], vt = vturb[(size_t)c * N + k];
    double *cc = colconst + (size_t)(col0 + c) * colStride;
    const double nTot = cc[off_nTotal + (size_t)a * N + k];
    const int NL = A.Nlevel[a], l0 = A.lvlOff[a];
    // ---- lte_pops, atomic_set.py:105-145
    const double dEion = A.c2 * sqrt(xne / t);
    const double cNe_T = 0.5 * xne * pow(A.c1 / t, 1.5);
    double ns[NLMAX];
    double total = 1.0;
    for (int i = 1; i < NL; ++i) {
        const double dE_kT = (A.dE[l0 + i] - A.nDebye[l0 + i] * dEion) / (kKBoltzmann * t);
        double v = A.gi0[l0 + i] * exp(-dE_kT);
        const int dZ = A.dZ[l0 + i];
        const double den = dZ == 0 ? 1.0 : (dZ == 1 ? cNe_T : (dZ == 2 ? cNe_T * cNe_T : pow(cNe_T, (double)dZ)));
        v /= den;
        ns[i] = v;
        total += v;
    }
    ns[0] = nTot / total;
    for (int i = 1; i < NL; ++i) ns[i] *= ns[0];
    for (int i = 0; i < NL; ++i) {
        nStar[((size_t)c * sumNlevel + l0 + i) * N + k] = ns[i];
        if (pops) pops[(size_t)(col0 + c) * popStride + (size_t)(l0 + i) * N + k] = ns[i];   // start from LTE (rh_method.py:415)
    }
    // ---- compute_collisions, rh_method.py:474-487: C[i][j] = rate from j to i, terms added in the model's order
    double Cm[NLMAX * NLMAX];
    for (int e = 0; e < NL * NL; ++e) Cm[e] = 0.0;
    const double sqT = sqrt(t);
    for (int q = 0; q < A.Ncoll; ++q) {
        const int32_t *cd = A.coll + 8 * q;
        if (cd[0] != a) continue;
        const int kind = cd[1], i = cd[2], j = cd[3];
        const double Cv = coll_table(A, q, t);
        if (kind == 0) {          // Omega, collisional_rates.py:43-46
            const double Cdown = A.par[q] * xne * Cv / (A.g[l0 + j] * sqT);
            Cm[i * NL + j] += Cdown;
            Cm[j * NL + i] += Cdown * ns[j] / ns[i];
        } else if (kind == 1) {   // CI, :70-72
            const double Cup = Cv * xne * exp(-A.par[q] / (kKBoltzmann * t)) * sqT;
            Cm[j * NL + i] += Cup;
            Cm[i * NL + j] += Cup * ns[i] / ns[j];
        } else {                  // CE, :94-96
            const double Cdown = Cv * xne * A.par[q] * sqT;
            Cm[i * NL + j] += Cdown;
            Cm[j * NL + i] += Cdown * ns[j] / ns[i];
        }
    }
    double *Cdst = cc + off_C + (size_t)A.g2Off[a] * N + k;
    for (int e = 0; e < NL * NL; ++e) Cdst[(size_t)e * N] = Cm[e] < 0.0 ? 0.0 : Cm[e];
    // ---- v_broad, atomic_model.py:241-245
    vBroad[((size_t)c * A.Natom + a) * N + k] = sqrt(A.vTherm[a] * t + vt * vt);
}
template <int NLMAX>
__global__ void setup_levels_kernel(const AtomLevels A, int N, const double *T, const double *ne, const double *vturb,
                                    double *colconst, int64_t colStride, int64_t off_C, int64_t off_nTotal, double *nStar,
                                    double *vBroad, double *pops, int64_t popStride, int sumNlevel, int col0)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    setup_levels_point<NLMAX>(A, N, T, ne, vturb, colconst, colStride, off_C, off_nTotal, nStar, vBroad, pops, popStride,
                              sumNlevel, col0, blockIdx.y, blockIdx.z, k);
}

// g_ij of the continua (rh_method.py:453-454): nStar_i / nStar_j * exp(-(hc/k) / lambda / T), written -- times the
// cross-section alpha, i.e. as Vji of rh_method.py:285 -- into the slot fields of the tile records.  One block row per (continuum, column); threads run over (wavelength, depth).
struct GijCont {
    int32_t rowI, rowJ, Nblue, Nlam, tile0, tab0;   // level rows in nStar; wavelength range; first tile; first GijTile
    int32_t toff, pad;                               // the continuum's entries of the per-wavelength tables (alpha)
};
struct GijTile {
    int32_t f, stride;    // depth-0 offset of the continuum's field in that tile's records; record stride
};
// wavelength lt of continuum ct at depth k of column c of the call's inputs (tab: that column's table); shared with
// mali_perturb_columns (mali_perturb.cuh)
__device__ __forceinline__ void setup_gij_point(const GijCont &ct, const GijTile *gt, const double *wavelength,
                                                const double *alpha, int N, int Lw, const double *T, const double *ns,
                                                double *tab, double hc_k, int c, int lt, int k)
{
    const int la = ct.Nblue + lt;
    const int ti = la / Lw, ls = la - ti * Lw;
    const GijTile g = gt[ct.tab0 + ti - ct.tile0];
    const double v = ns[(size_t)ct.rowI * N + k] / ns[(size_t)ct.rowJ * N + k] *
                     exp(-hc_k / wavelength[la] / T[(size_t)c * N + k]);
    tab[g.f + (size_t)k * g.stride + ls] = v * alpha[ct.toff + lt];     // the field holds Vji = g_ij * alpha (:285)
}
__global__ void setup_gij_kernel(const GijCont *conts, const GijTile *gt, const double *wavelength, const double *alpha, int N, int Lw,
                                 int sumNlevel, const double *T, const double *nStar, double *colconst, int64_t colStride,
                                 int64_t offTab, int col0)
{
    const GijCont ct = conts[blockIdx.y];
    const int c = blockIdx.z;
    const double hc_k = kHC / (kKBoltzmann * kNmToM);
    double *tab = colconst + (size_t)(col0 + c) * colStride + offTab;
    const double *ns = nStar + (size_t)c * sumNlevel * N;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < ct.Nlam * N; idx += gridDim.x * blockDim.x) {
        const int lt = idx / N, k = idx - lt * N;
        setup_gij_point(ct, gt, wavelength, alpha, N, Lw, T, ns, tab, hc_k, c, lt, k);
    }
}

// --------------------------------------------------------------------------------------------------------
// The continuum groups' fields (mali_fs_spec.cuh, spec_group_*): for every group of bound-free transitions of a tile
// that share their upper level, sum_t Uji_t(lambda, k) with Uji = 2hc/lambda^3 * Vji exactly as uv forms it
// (rh_method.py:284-286; the slots' fields hold Vji = g_ij * alpha), summed in slot order -- the population-independent part of that level's U and of the group's
// emissivity.  Runs whenever the g_ij fields of a column are (re)written; one thread per (depth, wavelength of the tile).
// The whole body, shared with mali_perturb_columns (mali_perturb.cuh), which runs one depth of a column: the index
// policy gives the group tile, the column of the call and the threads' loop over idx = k * Lw + ls, and is read where
// the kernel read blockIdx / threadIdx when it was a single body, which keeps cont_group_kernel's instructions as they were.
struct GroupGridIdx {
    __device__ __forceinline__ unsigned tile() const { return blockIdx.y; }
    __device__ __forceinline__ unsigned col() const { return blockIdx.z; }
    __device__ __forceinline__ int first() const { return blockIdx.x * blockDim.x + threadIdx.x; }
    __device__ __forceinline__ int end(int N, int Lw) const { return N * Lw; }
    __device__ __forceinline__ int step() const { return gridDim.x * blockDim.x; }
};
template <class Ix>
__device__ __forceinline__ void cont_group_body(const TileDesc *tiles, const SlotDesc *slots, const int32_t *groupTiles,
                                                const double *twohc, int N, int Nspect, int Lw, double *colconst,
                                                int64_t colStride, int64_t offTab, int col0, Ix ix)
{
    const TileDesc td = tiles[groupTiles[ix.tile()]];
    double *tab = colconst + (size_t)(col0 + ix.col()) * colStride + offTab + td.recOff;
    const SlotDesc *sl = slots + td.slot0;
    for (int idx = ix.first(); idx < ix.end(N, Lw); idx += ix.step()) {
        const int k = idx / Lw, ls = idx - k * Lw;
        const int la = td.la0 + ls;
        double *rec = tab + (size_t)k * td.stride;
        int g = 0;
        for (int q = 0; q < td.nslot; ++q) {
            if (sl[q].isLine) continue;
            bool first = true;
            for (int u = 0; u < q; ++u)
                if (!sl[u].isLine && sl[u].lsJ == sl[q].lsJ) first = false;
            if (!first) continue;
            double sum = 0.0;
            for (int u = q; u < td.nslot; ++u) {
                if (sl[u].isLine || sl[u].lsJ != sl[q].lsJ) continue;
                const int lt = la - sl[u].Nblue;
                if (la < Nspect && lt >= 0 && lt < sl[u].Nlam) {
                    sum = sum + twohc[sl[u].toff + lt] * rec[sl[u].fOff + ls];
                }
            }
            rec[td.bgOff + (3 + td.nslot + g) * Lw + ls] = sum;
            ++g;
        }
    }
}
__global__ void cont_group_kernel(const TileDesc *tiles, const SlotDesc *slots, const int32_t *groupTiles,
                                  const double *twohc, int N, int Nspect, int Lw, double *colconst, int64_t colStride,
                                  int64_t offTab, int col0)
{
    cont_group_body(tiles, slots, groupTiles, twohc, N, Nspect, Lw, colconst, colStride, offTab, col0, GroupGridIdx{});
}

// --------------------------------------------------------------------------------------------------------
// Background / EOS on the device (SURVEY.md 8f rank 1): Background.compute_background_eos (background.py:21-53) and the
// column-mass branch of AtmosphereConstructor.convert_scales (atmosphere.py:70-112) for a batch of columns.
struct EosParams {
    eos::Tables E;
    double amu_wph;        // Amu * weightPerH                                  (background.py:33, atmosphere.py:81-82)
    double cm3, g_to_kg;   // CM_TO_M**3, G_TO_KG
    double cm_to_m;        // CM_TO_M
    double thomson;        // the Thomson cross-section of background.py:11
};
// per (column, depth) thermodynamic state: work[(c * N + k) * kEosWork + ...]
constexpr int kEosWork = 20;   // pgas, pe, chi_c (per m at 5000 A), then the 17 background partials

// one thread per (column, depth): gas and electron pressure from (T, rho), the background partial densities, and the
// 5000 A opacity the scale conversion needs
// point idx = c * N + k of the call's inputs; shared with mali_perturb_columns (mali_perturb.cuh)
__device__ __forceinline__ void eos_point(const EosParams &P, const double *T, const double *nHTot, double *work, int idx)
{
    const double t = T[idx];
    const double rho = P.amu_wph * nHTot[idx] * P.cm3 / P.g_to_kg;                       // background.py:33
    double *w = work + (size_t)idx * kEosWork;
    eos::PointCache C;                      // the temperature-only factors of the EOS iterations, formed once
    eos::point_cache(P.E, t, C);
    const double pgas = eos::pg_from_rho(P.E, C, t, rho);
    const double pe = eos::pe_from_rho(P.E, C, t, rho);
    w[0] = pgas;
    w[1] = pe;
    eos::background_partials(P.E, C, t, pgas, pe, w + 3);
    const double TK = t * eos::BK, TKEV = TK / eos::EV, HTK = eos::HH / TK, TLOG = log(t), xne = pe / TK;
    double op, sc;
    eos::cop_one(t, TKEV, HTK, TLOG, xne, 5000.0, w + 3, op, sc);
    w[2] = op / P.cm_to_m;                                                                // atmosphere.py:92
}
__global__ void eos_kernel(const EosParams P, int N, int ncol, const double *T, const double *nHTot, double *work)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= N * ncol) return;
    eos_point(P, T, nHTot, work, idx);
}

// one thread per (column, wavelength, depth): chi = cop / CM_TO_M, eta = planck(T, lambda) * chi (utils.py:17-22 as numpy
// evaluates it for an array of wavelengths), sca = ne * sigma_T  -- written into the bg fields of the tile records.
// One thread's work; shared with mali_perturb_columns (mali_perturb.cuh).
__device__ __forceinline__ void background_point(const EosParams &P, const TileDesc *tiles, const double *wavelength, int N,
                                                 int Nspect, int Lw, const double *T, const double *ne, const double *work,
                                                 double *colconst, int64_t colStride, int64_t offTab, int col0, int c,
                                                 int la, int k)
{
    const size_t idx = (size_t)c * N + k;
    const double t = T[idx];
    const double *w = work + idx * kEosWork;
    const double TK = t * eos::BK, TKEV = TK / eos::EV, HTK = eos::HH / TK, TLOG = log(t), xne = w[1] / TK;
    const double wav = wavelength[la];
    double op, sc;
    eos::cop_one(t, TKEV, HTK, TLOG, xne, wav * 10, w + 3, op, sc);
    const double chi = op / P.cm_to_m;
    // utils.planck with an array argument: numpy power / exp
    const double hc_Tkla = kHC / (kKBoltzmann * kNmToM * wav) / t;
    const double twohnu3_c2 = (2.0 * kHC) / pow(kNmToM * wav, 3.0);
    const double eta = twohnu3_c2 / (exp(hc_Tkla) - 1.0) * chi;
    const int ti = la / Lw, ls = la - ti * Lw;
    const TileDesc td = tiles[ti];
    double *f = colconst + (size_t)(col0 + c) * colStride + offTab + td.recOff + (size_t)k * td.stride + td.bgOff + ls;
    f[0] = chi;
    f[Lw] = eta;
    f[2 * Lw] = ne[idx] * P.thomson;
    // lanes of the last tile past the end of the spectrum carry the last wavelength's values (as the host pack does)
    if (la == Nspect - 1)
        for (int q = ls + 1; q < Lw; ++q) {
            f[q - ls] = chi;
            f[Lw + q - ls] = eta;
            f[2 * Lw + q - ls] = ne[idx] * P.thomson;
        }
}
__global__ void background_kernel(const EosParams P, const TileDesc *tiles, const double *wavelength, int N, int Nspect,
                                  int Lw, const double *T, const double *ne, const double *work, double *colconst,
                                  int64_t colStride, int64_t offTab, int col0)
{
    const int c = blockIdx.z;
    const int la = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    background_point(P, tiles, wavelength, N, Nspect, Lw, T, ne, work, colconst, colStride, offTab, col0, c, la, k);
}

// one thread per column: the column-mass branch of convert_scales (atmosphere.py:94-111): heights from the column
// mass and density, the 5000 A optical depth, and the shift that puts tau_500 = 1 at height 0 (numpy.interp)
__global__ void convert_scales_kernel(const EosParams P, int N, int ncol, const double *cmass, const double *nHTot,
                                      const double *work, double *colconst, int64_t colStride, int64_t off_z, int col0,
                                      double *tau_out)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncol) return;
    const double *cm = cmass + (size_t)c * N, *nh = nHTot + (size_t)c * N;
    const double *w = work + (size_t)c * N * kEosWork;
    double *z = colconst + (size_t)(col0 + c) * colStride + off_z;
    double *tau = tau_out + (size_t)c * N;
    double hPrev = 0.0, rhoPrev = P.amu_wph * nh[0], chiPrev = w[2];
    double tauPrev = chiPrev / rhoPrev * cm[0];
    z[0] = 0.0;
    tau[0] = tauPrev;
    for (int k = 1; k < N; ++k) {
        const double rho = P.amu_wph * nh[k], chi = w[(size_t)k * kEosWork + 2];
        const double h = hPrev - 2.0 * (cm[k] - cm[k - 1]) / (rhoPrev + rho);
        const double ta = tauPrev + 0.5 * (chiPrev + chi) * (hPrev - h);
        z[k] = h;
        tau[k] = ta;
        hPrev = h;
        rhoPrev = rho;
        chiPrev = chi;
        tauPrev = ta;
    }
    // numpy.interp(1.0, tau, height): tau increases with depth
    double h1;
    if (1.0 <= tau[0])
        h1 = z[0];
    else if (1.0 >= tau[N - 1])
        h1 = z[N - 1];
    else {
        int j = 0;
        while (!(tau[j + 1] > 1.0)) ++j;        // tau[j] <= 1 < tau[j+1]
        const double slope = (z[j + 1] - z[j]) / (tau[j + 1] - tau[j]);
        h1 = slope * (1.0 - tau[j]) + z[j];
    }
    for (int k = 0; k < N; ++k) z[k] -= h1;
}

struct CopyJob {
    int64_t srcOff, dstOff, len;
    int32_t toPops;  // destination is the pops buffer instead of colconst
    int32_t pad;     // non-zero: a block the device-side set-up produces itself (C, n)
};
__global__ void pack_misc_kernel(const CopyJob *copies, int ncopies, const double *staging, int64_t hpStride,
                                 double *colconst, int64_t colStride, double *pops, int64_t popStride, double *J,
                                 int64_t JStride, int col0, int skipDerived)
{
    const int col = col0 + blockIdx.y;
    const double *src = staging + (size_t)blockIdx.y * hpStride;
    double *cc = colconst + (size_t)col * colStride;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (int c = 0; c < ncopies; ++c) {
        const CopyJob cj = copies[c];
        if (skipDerived && cj.pad) continue;      // C and the starting populations come from setup_levels_kernel
        double *dst = cj.toPops ? pops + (size_t)col * popStride + cj.dstOff : cc + cj.dstOff;
        for (int64_t q = tid; q < cj.len; q += nth) dst[q] = src[cj.srcOff + q];
    }
    double *Jc = J + (size_t)col * JStride;
    for (int64_t q = tid; q < JStride; q += nth) Jc[q] = 0.0;
}

}  // namespace mali
