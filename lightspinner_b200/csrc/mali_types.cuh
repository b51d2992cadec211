// mali_types.cuh -- device-side descriptors of the B200 MALI hot path.
//
// Layout vocabulary (SURVEY.md appendix B): a *column* is one 1D atmosphere; a *ray* is one
// (wavelength la, angle mu) pair of a column, swept down (toFrom=0) then up (toFrom=1) over the
// Nspace depth points; a *tile* is the group of Lw = 32 / Nrays consecutive wavelengths (all angles)
// one warp owns; a *slot* is one radiative transition overlapping a tile's wavelength range.
//
// The per-column tables are stored TILE-MAJOR, DEPTH-CONTIGUOUS: tile after tile, and inside a tile one *record* per
// depth point k (record stride = the tile's record size), holding everything the tile's warp reads at that depth:
//     [ Vij rows of direction 0 (down sweep): one per line slot, each kVRow = 32 doubles = (wavelength, angle) in lane order ]
//     [ fields: J-dagger[Lw rounded up to 4]: the mean intensity of the previous iteration, rewritten by
//               j_finish_kernel (the only part of a record that changes between iterations; zero after upload)
//               bg chi[Lw] | bg eta[Lw] | bg sca[Lw]
//               per slot: wla[Lw] (lines, rh_method.py:451) or Vji = g_ij * alpha [Lw] (continua, :453-454, :285)
//               per continuum group (the tile's bound-free transitions with one upper level): sum_t Uji_t [Lw], formed
//               from the g_ij fields by cont_group_kernel whenever those are (re)written       (padded to 4 doubles) ]
//     [ Vij rows of direction 1 (up sweep) ]
// The fields sit BETWEEN the two directions' rows, so what one sweep direction needs at a depth -- [rows 0 | fields]
// or [fields | rows 1] -- is one contiguous piece: one TMA bulk copy per depth step, and a sweep walks its tile's
// records as a single sequential stream.  Entries for wavelengths on which a transition is not active are zero, so
// the kernels need no activity masks for their loads; records are 32-byte aligned.
//
// Level populations reach the formal-solution kernels through a second per-column table, depth-major:
//     popsT[k] = [ z[k] | n[0][k] ... n[sumNlevel-1][k] | pad ]           (row width PW = 1 + sumNlevel rounded up to 4)
// (heights first, then every level of every active atom), rebuilt from n[level][k] at the start of every formal
// solution, so that the populations and heights of a depth step also arrive by TMA with that step's record and the
// shared memory a warp needs does not depend on the number of depth points.
#pragma once
#include <cstdint>

namespace mali {

// constants.py:1-4,17 -- digit for digit
constexpr double kCLight = 2.99792458E+08;
constexpr double kHPlanck = 6.6260755E-34;
constexpr double kHC = kHPlanck * kCLight;
constexpr double kKBoltzmann = 1.380658E-23;
constexpr double kNmToM = 1.0E-09;
constexpr double kPi = 3.141592653589793;  // == numpy.pi

struct SlotDesc {
    int32_t t;        // transition index (reference order)
    int32_t isLine;
    int32_t Nblue, Nlam;
    int32_t rowI, rowJ;  // rows of the lower / upper level in n[sumNlevel][Nspace]
    int32_t atom;
    int32_t lsI, lsJ;    // level-slot of the lower / upper level inside the tile
    int32_t toff;        // offset of this transition in the per-wavelength tables (alpha, twohc, wlacont)
    int32_t flags;       // bit 0 / 1: this slot is the first of its tile to touch level-slot lsI / lsJ
    int32_t fOff;        // record offset of the slot's per-wavelength field: wla[Lw] (lines) or g_ij * alpha [Lw] (continua)
    int32_t vOff;        // lines: record offset of the direction-0 Vij row (direction 1: + TileDesc::vDir); else -1
    int32_t pad;
    double c0, c1, c2;   // lines: hc/4pi*Bij (folded into the Vij table at upload), Aji/Bji, Bji/Bij  (rh_method.py:279-281,450)
};

struct TileDesc {
    int32_t la0;       // first wavelength of the tile
    int32_t nslot;     // transitions overlapping [la0, la0+Lw)
    int32_t slot0;     // first SlotDesc of the tile
    int32_t nlevslot;  // distinct (atom, level) pairs touched by the tile's slots
    int32_t partRow0;  // first row of the tile's Gamma partials (2 rows per slot: [i,j] then [j,i])
    int32_t recOff;    // offset of the tile's first record (depth 0) inside the column's table
    int32_t bgOff;     // record offset of bg chi[Lw] (eta, sca follow at +Lw, +2Lw)
    int32_t vDir;      // distance between the direction-0 and direction-1 Vij rows (line rows + fields)
    int32_t stride;    // record size = distance between the tile's records of consecutive depth points
    int32_t ngroup;    // continuum groups of the tile: their fields sum_t Uji_t [Lw] follow the slots' fields
    int32_t pad1, pad2;
};

constexpr int kVRow = 32;  // doubles per Vij row of a record (Lw * Nrays <= 32 lanes, zero padded)

// Kernel parameters (passed by value -> constant bank).
struct FsParams {
    // sizes
    int32_t N, Nrays, Nspect, Natom, Ntrans, Lw, ntile, Dmax;
    int32_t col0, ncol, blocksPerCol, warpsPerBlock;
    int32_t smemPerWarp;  // doubles
    // strides (doubles per column)
    int64_t colStride, popStride, JStride, IStride, scratchStride;
    // offsets inside one column's colconst block
    int64_t off_z, off_bbc, off_tab;
    // offsets inside one column's scratch block
    int64_t off_jpart, off_part;
    int64_t upOff;  // the up sweep writes its partial sums this many doubles further on (no read-modify-write)
    // model tables (device)
    const TileDesc *tiles;
    const SlotDesc *slots;
    const int32_t *classTiles;  // tile indices handled by this launch (tiles are grouped by slot count)
    int32_t nClassTiles;
    const double *alpha, *twohc, *wlacont;  // concatenated per-wavelength tables
    const double *zmu, *hw;                 // [Nrays]: 1/muz, 0.5*wmu
    // batch buffers (device)
    const double *colconst;
    const double *pops;
    double *J, *I, *scratch;
    unsigned long long *dJbits;
    int32_t *status;      // may be null; bit 1: a divisor left the fast-division domain
    const int32_t *done;  // may be null
};

struct FinishParams {
    int32_t N, Natom, Ntrans, col0, ncol;
    int32_t sumNlevel, sumNlevel2;
    int64_t colStride, popStride, gammaStride, scratchStride;
    int64_t off_C, off_nTotal, off_part, upOff;
    const int32_t *Nlevel;     // [Natom]
    const int32_t *lvlOff;     // [Natom+1]
    const int32_t *g2Off;      // [Natom+1]
    const int32_t *trans;      // [Ntrans][6]
    const int32_t *trPartOff;  // [Ntrans+1] CSR into trPartRows
    const int32_t *trPartRows; // partial row of the [i,j] entry (the [j,i] entry is row+1), ascending tile order
    const double *colconst;
    double *pops, *Gamma;
    const double *scratch;
    unsigned long long *dPopsBits;
    int32_t *status;
    const int32_t *done;
    const int32_t *iter;  // may be null; with iter: only columns with iter[col] >= iterMin are solved
    int32_t iterMin;
    // Ng acceleration (mali_stat_equil_ng / mali_iterate_ng; null otherwise): per column ngStride doubles holding
    // ngRing ring slots of [sumNlevel][N] solved populations, then the snapshot of n taken before the solve.
    // stat_equil_kernel writes the snapshot and pushes the solution into slot (ngNse[col] - 1) % ngRing.
    double *ngHist;
    const int32_t *ngNse;
    int64_t ngStride;
    int32_t ngRing;
};

}  // namespace mali
