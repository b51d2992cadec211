// mali_api.cu -- host side of libmali_b200.so: model flattening (tiles / slots / record layout) and the C ABI
// declared in include/mali_b200.h.  No torch types, no exceptions across the boundary.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/mali_b200.h"
#include "mali_kernels.cuh"
#include "mali_rays.cuh"
#include "mali_rates.cuh"
#include "mali_perturb.cuh"
#include "mali_fs_launch.h"

using namespace mali;

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) return fail((int)e_, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

template <class T>
cudaError_t to_device(const std::vector<T> &h, T **d)
{
    *d = nullptr;
    const size_t bytes = std::max<size_t>(h.size(), 1) * sizeof(T);
    cudaError_t e = cudaMalloc((void **)d, bytes);
    if (e != cudaSuccess) return e;
    if (!h.empty()) e = cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
    return e;
}

// First kernel of every statistical-equilibrium stage: inside mali_iterate it counts the iteration (test.py:24;
// the formal solution of this iteration is done), then resets dPops of the columns that are about to be solved.
// With Ng acceleration (nse != null) it also counts the solve in the column's nse.
__global__ void se_prepare_kernel(unsigned long long *bits, const int32_t *done, int32_t *iter, int iterMin, int count,
                                  int col0, int ncol, int32_t *nse)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncol) return;
    const int col = col0 + c;
    if (done != nullptr && done[col] != 0) return;
    if (iter != nullptr) {
        if (count) iter[col] += 1;
        if (iter[col] < iterMin) return;
    }
    bits[col] = 0ull;
    if (nse != nullptr) nse[col] += 1;
}

// First kernel of every formal solution, one block per column: resets dJ and rebuilds the depth-major popsT table
// (mali_types.cuh) from the heights and the CURRENT populations n[level][k] -- the caller may have edited them since
// the last call, as the reference's users do through the eqPops alias.
// Inside mali_iterate (ctl.on) it also closes the previous iteration of the loop of test.py:20-29 for its column:
// the convergence test on that iteration's (dJ, dPops), and a stop on a fault.
struct IterCtl {
    int32_t on;
    double tolJ, tolPops;
    int32_t *iter, *doneW;
    const int32_t *status;
    const double *dPops;
};
__device__ __forceinline__ void iterate_check(const IterCtl &c, int col, double dJ)
{
    if (c.iter[col] == 0) return;        // nothing to judge before the first iteration
    const double a = dJ, b = c.dPops[col];
    if (c.tolJ >= 0.0 && !(a > c.tolJ || b > c.tolPops)) c.doneW[col] = 1;  // the negation of `while dJ > 2e-3 or dPops > 1e-3`
    // a singular system / a formal-solver domain fault (status) or a NaN: stop touching the column and flag it
    // (the reference raises at this point; the host wrapper turns done == 2 into the same exceptions)
    if (a != a || b != b || c.status[col] != 0) c.doneW[col] = 2;
}
__global__ void fs_prepare_kernel(unsigned long long *dJbits, const int32_t *done, int col0, double *colconst,
                                  int64_t colStride, int64_t off_z, int64_t off_popsT, int PW, int N, int sumNlevel,
                                  const double *pops, int64_t popStride, const IterCtl ctl)
{
    const int col = col0 + blockIdx.x;
    if (done != nullptr && done[col] != 0) return;
    if (ctl.on) {    // block-uniform outcome: every thread evaluates the same test on the same values
        iterate_check(ctl, col, __longlong_as_double((long long)dJbits[col]));
        __syncthreads();
        if (ctl.doneW[col] != 0) return;
    }
    __syncthreads();
    if (threadIdx.x == 0) dJbits[col] = 0ull;
    double *cc = colconst + (size_t)col * colStride;
    const double *z = cc + off_z, *n = pops + (size_t)col * popStride;
    double *pt = cc + off_popsT;
    for (int idx = threadIdx.x; idx < N * PW; idx += blockDim.x) {
        const int k = idx / PW, c = idx - k * PW;
        pt[idx] = c == 0 ? z[k] : (c - 1 < sumNlevel ? n[(size_t)(c - 1) * N + k] : 0.0);
    }
}

// Closes the LAST iteration of a mali_iterate call (the earlier ones are closed by the next iteration's
// fs_prepare_kernel): convergence test / fault stop per column.
__global__ void iterate_close_kernel(const double *dJ, const IterCtl ctl, int col0, int ncol)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncol) return;
    const int col = col0 + c;
    if (ctl.doneW[col] != 0) return;
    iterate_check(ctl, col, dJ[col]);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------
// The structure-specialised kernels and their instance registry live in mali_fs_class.cu (one translation unit per
// register class); tiles are routed to them by structure key.
static const SpecEntry *find_spec(const std::string &key)
{
    static std::map<std::string, const SpecEntry *> index;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const SpecEntry *e = mali_fs_registry(); e->key; ++e) index[e->key] = e;
    });
    auto it = index.find(key);
    return it == index.end() ? nullptr : it->second;
}

// ---------------------------------------------------------------------------------------------------------
struct IterGraphKey {
    mali_buffers b;
    int32_t col0, ncol;
    double tolJ, tolPops;
    int32_t arith;
    mali_ng_buffers ng;      // all zero for mali_iterate: a plain graph is never replayed for an Ng call, or the reverse
    mali_ng_params ngp;
};
struct IterGraph {
    IterGraphKey key;
    cudaGraphExec_t exec;
    long long kernels;   // kernel nodes of one iteration
};

struct mali_model {
    int device = 0;
    mutable std::vector<IterGraph> iterGraphs;   // captured iterations of mali_iterate
    int arith = MALI_ARITH_EXACT;   // arithmetic mode of the specialised formal-solution kernels (mali_model_set_arith)
    int N = 0, Nrays = 0, Nspect = 0, Natom = 0, Ntrans = 0, Lw = 0, ntile = 0, Dmax = 0, Tmax = 0;
    int sumNlevel = 0, sumNlevel2 = 0, maxNlevel = 0, nPartRows = 0;
    std::vector<int32_t> Nlevel, lvlOff, g2Off, trans, toff;
    std::vector<SlotDesc> slots;
    std::vector<TileDesc> tiles;
    std::vector<SlotDesc> transSlot;     // one descriptor per transition (uv hook)
    std::vector<int32_t> genericTiles;   // tiles without a specialised instance -> generic kernel
    std::vector<TileR<2>> spec0;         // tiles served by the structure-specialised kernels, per register class,
    std::vector<TileR<4>> spec1;         // heaviest first
    std::vector<TileR<8>> spec2;
    int specTiles = 0;
    mali_layout lay{};
    int64_t off_z = 0, off_bbc = 0, off_C = 0, off_nTotal = 0, off_tab = 0, off_popsT = 0, rowStride = 0;
    int popsW = 0;
    int64_t off_jpart = 0, off_part = 0, upOff = 0;
    int smemClass[3] = {0, 0, 0};   // shared-memory bytes per warp of the three specialised kernels
    std::vector<CopyJob> cjobs;
    int packChunks = 0, packChunksFields = 0;   // all re-layout chunks; the leading ones that touch record fields
    // device copies
    TileDesc *d_tiles = nullptr;
    SlotDesc *d_slots = nullptr;
    double *d_alpha = nullptr, *d_twohc = nullptr, *d_wlacont = nullptr, *d_wlambda = nullptr, *d_zmu = nullptr,
           *d_hw = nullptr;
    int32_t *d_Nlevel = nullptr, *d_lvlOff = nullptr, *d_g2Off = nullptr, *d_trans = nullptr, *d_trPartOff = nullptr,
            *d_trPartRows = nullptr, *d_genericTiles = nullptr;
    TileJ *d_tileJ = nullptr;
    PhiTile *d_phiTiles = nullptr;
    PhiLine *d_phiLines = nullptr;
    double *d_wavelength = nullptr, *d_muz = nullptr, *d_wmu = nullptr;
    double *d_lambda0 = nullptr;        // [Ntrans] line centres (zeros without mali_model_desc.lambda0): mali_compute_rays
    int nPhiLines = 0;
    AtomLevels atoms{};                 // model-level atom data of the device-side set-up (mali_model_set_atoms)
    std::vector<void *> atomDev;
    bool haveAtoms = false;
    EosParams eos{};                    // EOS / background tables (mali_model_set_eos)
    std::vector<void *> eosDev;
    bool haveEos = false;
    GijCont *d_gijCont = nullptr;
    GijTile *d_gijTiles = nullptr;
    int nGijCont = 0;
    int32_t *d_groupTiles = nullptr;    // tiles with continuum groups (cont_group_kernel)
    int nGroupTiles = 0;
    std::vector<std::vector<PhiTile>> phiTilesHost;   // per transition: where its profile entries live (mali_line_layout)
    std::vector<int32_t> phiTile0Host;
    bool haveLambda0 = false;
    CopyJob *d_cjobs = nullptr;
    PackChunk *d_pchunks = nullptr;
    PackTile *d_ptiles = nullptr;
    PackSlot *d_pslots = nullptr;
    // optional per-launch timing of the formal-solution stage (mali_profile_begin / mali_profile_end)
    mutable std::vector<cudaEvent_t> profEvents;
    // the three register-class kernels of one formal solution are independent: they run on the caller's stream
    // and two side streams (fork / join by events), so that one kernel's tail overlaps the others
    cudaStream_t sideStream[2] = {nullptr, nullptr};
    cudaStream_t iterStream = nullptr;      // mali_iterate's own stream when the caller is on the legacy default stream
    cudaEvent_t iterFork = nullptr, iterJoin = nullptr;
    mutable long long graphLaunches = 0;    // iterations replayed from a captured graph (mali_model_info-style diagnostics)
    cudaEvent_t forkEvent = nullptr, joinEvent[2] = {nullptr, nullptr};
    mutable int profUsed = 0;
    mutable bool profOn = false;
    mutable long long launches = 0;  // kernels launched through this model since creation
    mutable int32_t *d_depth = nullptr;  // mali_perturb_columns' depth list on the device
    mutable int depthCap = 0;
};

extern "C" {

const char *mali_last_error(void) { return g_err.c_str(); }

int mali_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int mali_planck_bc(const double *wavelength, int32_t Nspect, double Tm2, double Tm1, double *out)
{
    if (!wavelength || !out || Nspect < 0) return fail(MALI_EINVAL, "mali_planck_bc: bad argument");
    // utils.py:17-22 as numba compiles it: cube by repeated multiplication, libm exp (SURVEY.md A.7)
    for (int la = 0; la < Nspect; ++la) {
        const double wav = wavelength[la];
        const double y = kNmToM * wav;
        const double twohnu3_c2 = (2.0 * kHC) / (y * y * y);
        const double T[2] = {Tm2, Tm1};
        for (int q = 0; q < 2; ++q) {
            const double hc_Tkla = kHC / (kKBoltzmann * kNmToM * wav) / T[q];
            out[2 * la + q] = twohnu3_c2 / (std::exp(hc_Tkla) - 1.0);
        }
    }
    return MALI_OK;
}

int mali_model_create(const mali_model_desc *d, int device, mali_model **out)
{
    if (!d || !out) return fail(MALI_EINVAL, "mali_model_create: null argument");
    *out = nullptr;
    if (d->Nspace < 3) return fail(MALI_ELIMIT, "Nspace=%d: the short-characteristic sweep needs >= 3 depth points", d->Nspace);
    if (d->Nrays < 1 || d->Nrays > 32) return fail(MALI_ELIMIT, "Nrays=%d not in [1, 32]", d->Nrays);
    if (d->Nspect < 1 || d->Natom < 1 || d->Ntrans < 0) return fail(MALI_EINVAL, "bad model sizes");
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(MALI_EINVAL, "device %d out of range (%d devices)", device, ndev);
    CU(cudaSetDevice(device));
    // the opt-in to more than 48 KB of dynamic shared memory is a per-device function attribute: set it for the
    // device this model lives on (deep columns need it), every time a model is created there
    CU(mali_fs_set_attr_0());
    CU(mali_fs_set_attr_1());
    CU(mali_fs_set_attr_2());
    CU(mali_fs_set_attr_0_fast());
    CU(mali_fs_set_attr_1_fast());
    CU(mali_fs_set_attr_2_fast());
    CU(cudaFuncSetAttribute(fs_gamma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));

    auto *m = new mali_model();
    m->device = device;
    if (const char *a = getenv("MALI_ARITH")) m->arith = (strcmp(a, "exact") == 0) ? MALI_ARITH_EXACT : MALI_ARITH_CONTRACTED;
    else m->arith = MALI_ARITH_DEFAULT;
    m->N = d->Nspace;
    m->Nrays = d->Nrays;
    m->Nspect = d->Nspect;
    m->Natom = d->Natom;
    m->Ntrans = d->Ntrans;
    m->Lw = 32 / d->Nrays;
    m->ntile = (d->Nspect + m->Lw - 1) / m->Lw;
    const int N = m->N, Lw = m->Lw;

    m->Nlevel.assign(d->Nlevel, d->Nlevel + d->Natom);
    m->lvlOff.assign(d->Natom + 1, 0);
    m->g2Off.assign(d->Natom + 1, 0);
    for (int a = 0; a < d->Natom; ++a) {
        if (m->Nlevel[a] < 1 || m->Nlevel[a] > 16) {
            delete m;
            return fail(MALI_ELIMIT, "atom %d: Nlevel=%d not in [1, 16]", a, d->Nlevel[a]);
        }
        m->lvlOff[a + 1] = m->lvlOff[a] + m->Nlevel[a];
        m->g2Off[a + 1] = m->g2Off[a] + m->Nlevel[a] * m->Nlevel[a];
        m->maxNlevel = std::max(m->maxNlevel, m->Nlevel[a]);
    }
    m->sumNlevel = m->lvlOff[d->Natom];
    m->sumNlevel2 = m->g2Off[d->Natom];
    m->trans.assign(d->trans, d->trans + (size_t)d->Ntrans * MALI_TRANS_STRIDE);
    m->toff.assign(d->Ntrans + 1, 0);
    for (int t = 0; t < d->Ntrans; ++t) {
        const int32_t *tr = &m->trans[(size_t)t * 6];
        const bool bad = tr[0] < 0 || tr[0] >= d->Natom || tr[1] < 0 || tr[2] < 0 || tr[1] >= m->Nlevel[tr[0]] ||
                         tr[2] >= m->Nlevel[tr[0]] || tr[1] == tr[2] || tr[4] < 0 || tr[5] < 1 ||
                         tr[4] + tr[5] > d->Nspect;
        if (bad) {
            delete m;
            return fail(MALI_EINVAL, "transition %d: inconsistent descriptor (atom %d, levels %d -> %d of %d, wavelengths [%d, %d) of %d)",
                        t, tr[0], tr[1], tr[2], (tr[0] >= 0 && tr[0] < d->Natom) ? m->Nlevel[tr[0]] : -1, tr[4], tr[4] + tr[5], d->Nspect);
        }
        m->toff[t + 1] = m->toff[t] + tr[5];
    }
    const int ntab = m->toff[d->Ntrans];

    // ---- host pack: reference layouts, plain concatenation
    mali_layout &L = m->lay;
    int64_t h = 0;
    auto htake = [&](int64_t n) { int64_t r = h; h += n; return r; };
    L.hp_height = htake(N);
    L.hp_bbc = htake(2 * (int64_t)d->Nspect);
    L.hp_nTotal = htake((int64_t)d->Natom * N);
    L.hp_bg_chi = htake((int64_t)d->Nspect * N);  // from here on: blocks mali_background can form on the device
    L.hp_bg_eta = htake((int64_t)d->Nspect * N);
    L.hp_bg_sca = htake((int64_t)d->Nspect * N);
    L.hp_C = htake((int64_t)m->sumNlevel2 * N);   // from here on: blocks mali_setup_columns can form on the device
    std::vector<int64_t> hpPhi(d->Ntrans, 0), hpGij(d->Ntrans, 0);
    L.hp_gijcont = h;
    for (int t = 0; t < d->Ntrans; ++t)
        if (!m->trans[(size_t)t * 6 + 3]) hpGij[t] = htake((int64_t)m->trans[(size_t)t * 6 + 5] * N);
    L.hp_n = htake((int64_t)m->sumNlevel * N);
    L.hp_phi = h;     // the profiles come last: a caller using mali_compute_phi uploads only [0, hp_phi)
    for (int t = 0; t < d->Ntrans; ++t)
        if (m->trans[(size_t)t * 6 + 3]) hpPhi[t] = htake((int64_t)m->trans[(size_t)t * 6 + 5] * d->Nrays * 2 * N);
    L.hp_wphi = htake((int64_t)d->Ntrans * N);
    L.hostpack = h;

    // ---- per-transition descriptors
    m->transSlot.resize(d->Ntrans);
    for (int t = 0; t < d->Ntrans; ++t) {
        const int32_t *tr = &m->trans[(size_t)t * 6];
        SlotDesc s{};
        s.t = t;
        s.isLine = tr[3];
        s.Nblue = tr[4];
        s.Nlam = tr[5];
        s.atom = tr[0];
        s.rowI = m->lvlOff[tr[0]] + tr[1];
        s.rowJ = m->lvlOff[tr[0]] + tr[2];
        s.toff = m->toff[t];
        s.vOff = -1;
        s.c0 = d->lineconst[3 * t + 0];
        s.c1 = d->lineconst[3 * t + 1];
        s.c2 = d->lineconst[3 * t + 2];
        m->transSlot[t] = s;
    }

    // ---- tiles, slots and the tile-major record layout (mali_types.cuh)
    std::vector<std::vector<int32_t>> trRows(d->Ntrans);
    std::vector<PackTile> ptiles;
    std::vector<TileJ> tileJ;        // per tile: J-dagger field of the depth-0 record, record stride
    std::vector<std::vector<PhiTile>> phiT(d->Ntrans);
    std::vector<std::vector<GijTile>> gijT(d->Ntrans);
    std::vector<int32_t> gijTile0(d->Ntrans, -1);
    std::vector<int32_t> phiTile0(d->Ntrans, -1);
    std::vector<PackSlot> pslots;
    std::vector<PackChunk> pchunks, pchunksRows;   // chunks touching the fields; chunks of Vij rows only
    int partRow = 0;
    int64_t rowOff = 0, rowSum = 0;
    for (int ti = 0; ti < m->ntile; ++ti) {
        const int la0 = ti * Lw, la1 = std::min(d->Nspect, la0 + Lw);
        TileDesc td{};
        td.la0 = la0;
        td.slot0 = (int)m->slots.size();
        td.partRow0 = partRow;
        std::map<std::pair<int, int>, int> lev;
        int nLine = 0;
        for (int t = 0; t < d->Ntrans; ++t) {
            const int32_t *tr = &m->trans[(size_t)t * 6];
            if (!(tr[4] < la1 && tr[4] + tr[5] > la0)) continue;
            SlotDesc s = m->transSlot[t];
            auto slot_of = [&](int level, int bit) {
                auto key = std::make_pair((int)tr[0], level);
                auto it = lev.find(key);
                if (it != lev.end()) return it->second;
                const int id = (int)lev.size();
                lev[key] = id;
                s.flags |= bit;  // first slot of the tile to touch this level: store instead of accumulate
                return id;
            };
            s.flags = 0;
            s.lsI = slot_of(tr[1], 1);
            s.lsJ = slot_of(tr[2], 2);
            if (s.isLine) s.vOff = kVRow * nLine++;
            trRows[t].push_back(partRow);
            partRow += 2;
            m->slots.push_back(s);
            td.nslot++;
        }
        const int vb = kVRow * nLine;            // one direction's Vij rows
        PackTile pt{};
        pt.recOff = (int32_t)rowOff;             // depth-0 record of the tile; records of one tile are contiguous over depth
        // record = [Vij rows dir 0 | fields | Vij rows dir 1]; fields = J-dagger (written by j_finish_kernel; padded to
        // whole 32-byte sectors), bg chi / eta / sca, one per-wavelength field per slot -- padded to whole sectors
        const int jw = (Lw + 3) & ~3;
        // continuum groups of the tile (bound-free transitions sharing their upper level, mali_fs_spec.cuh): one more
        // field each, after the slots' fields
        int ng = 0;
        for (int q = 0; q < td.nslot; ++q) {
            const SlotDesc &sq = m->slots[td.slot0 + q];
            if (sq.isLine) continue;
            bool first = true;
            for (int u = 0; u < q; ++u) {
                const SlotDesc &su = m->slots[td.slot0 + u];
                if (!su.isLine && su.lsJ == sq.lsJ) first = false;
            }
            if (first) ++ng;
        }
        td.ngroup = ng;
        const int sf = (int)align_up(jw + (3 + td.nslot + ng) * Lw, 4);
        pt.recSize = 2 * vb + sf;
        tileJ.push_back(TileJ{(int32_t)rowOff + vb, pt.recSize});
        pt.la0 = la0;
        pt.nslot = td.nslot;
        pt.slot0 = (int32_t)pslots.size();
        pt.vb = vb;
        pt.jw = jw;
        pt.sf = sf;
        int lineIdx = 0;
        for (int q = 0; q < td.nslot; ++q) {
            SlotDesc &s = m->slots[td.slot0 + q];
            s.fOff = vb + jw + (3 + q) * Lw;
            PackSlot ps{};
            ps.isLine = s.isLine;
            ps.Nblue = s.Nblue;
            ps.Nlam = s.Nlam;
            ps.lineIdx = s.isLine ? lineIdx++ : -1;
            ps.toff = s.toff;
            ps.srcOff = s.isLine ? hpPhi[s.t] : hpGij[s.t];
            ps.wphiOff = L.hp_wphi + (int64_t)s.t * N;
            ps.c0 = s.c0;
            pslots.push_back(ps);
            if (!s.isLine) {  // where setup_gij_kernel finds this continuum's g_ij field of this tile
                gijT[s.t].push_back(GijTile{(int32_t)rowOff + s.fOff, pt.recSize});
                if (gijTile0[s.t] < 0) gijTile0[s.t] = ti;
            }
            if (s.isLine) {   // where compute_phi_kernel finds this line's entries of this tile
                phiT[s.t].push_back(PhiTile{(int32_t)rowOff + s.vOff, vb + sf, (int32_t)rowOff + s.fOff, pt.recSize});
                if (phiTile0[s.t] < 0) phiTile0[s.t] = ti;
            }
        }
        // chunks that hold nothing but Vij rows go to the back of the list: the uploads that leave the line profiles to
        // compute_phi_kernel launch only the front part (two thirds of the blocks would return at once otherwise, and
        // the re-layout is bound by the block launch rate, not by bandwidth)
        for (int e0 = 0; e0 < pt.recSize; e0 += 32) {
            const bool rowsOnly = (e0 + 32 <= pt.vb) || (e0 >= pt.vb + pt.sf);
            (rowsOnly ? pchunksRows : pchunks).push_back(PackChunk{ti, e0});
        }
        ptiles.push_back(pt);
        td.recOff = pt.recOff;
        td.bgOff = vb + jw;
        td.vDir = vb + sf;
        td.stride = pt.recSize;
        td.nlevslot = (int)lev.size();
        rowOff += (int64_t)pt.recSize * N;
        rowSum += pt.recSize;
        m->Dmax = std::max(m->Dmax, td.nlevslot);
        m->Tmax = std::max(m->Tmax, td.nslot);
        m->tiles.push_back(td);
    }
    if (rowOff >= (int64_t)1 << 31) {
        delete m;
        return fail(MALI_ELIMIT, "per-column table of %lld doubles exceeds the 32-bit record offsets", (long long)rowOff);
    }
    m->nPartRows = partRow;
    m->rowStride = rowSum;      // doubles of the table per depth point (all tiles)
    m->packChunksFields = (int)pchunks.size();
    pchunks.insert(pchunks.end(), pchunksRows.begin(), pchunksRows.end());
    m->packChunks = (int)pchunks.size();
    std::vector<int32_t> trPartOff(d->Ntrans + 1, 0), trPartRows;
    for (int t = 0; t < d->Ntrans; ++t) {
        trPartOff[t + 1] = trPartOff[t] + (int)trRows[t].size();
        trPartRows.insert(trPartRows.end(), trRows[t].begin(), trRows[t].end());
    }

    // ---- colconst block of one column
    int64_t o = 0;
    auto take = [&](int64_t n) { int64_t r = o; o = align_up(o + n, 16); return r; };
    m->off_z = take(N);
    m->off_bbc = take(2 * (int64_t)d->Nspect);
    m->off_C = take((int64_t)m->sumNlevel2 * N);
    m->off_nTotal = take((int64_t)d->Natom * N);
    m->popsW = (int)align_up(1 + m->sumNlevel, 4);          // popsT row: z | n[all levels] | pad  (mali_types.cuh)
    m->off_popsT = take((int64_t)N * m->popsW);
    m->off_tab = take((int64_t)N * m->rowStride);
    L.colconst = o;
    L.pops = (int64_t)m->sumNlevel * N;
    L.J = (int64_t)N * d->Nspect;
    L.I = (int64_t)d->Nspect * d->Nrays;
    L.Gamma = (int64_t)m->sumNlevel2 * N;
    L.sumNlevel = m->sumNlevel;
    L.sumNlevel2 = m->sumNlevel2;
    L.ntile = m->ntile;
    L.lambda_per_warp = Lw;
    int64_t so = 0;
    m->off_jpart = so;
    so = align_up(so + L.J, 16);
    m->off_part = so;
    so = align_up(so + (int64_t)std::max(partRow, 1) * N, 16);
    m->upOff = so;      // second copy of [Jpart | part] for the up sweep
    L.scratch = 2 * so;
    if (m->Dmax > 255 || m->sumNlevel > 65535) {
        delete m;
        return fail(MALI_ELIMIT, "tile touches %d levels / model has %d levels: beyond the kernel's packed indices", m->Dmax, m->sumNlevel);
    }

    // ---- which tiles have a structure-specialised kernel instance
    auto structure_key = [&](const TileDesc &td) {  // must match tools/gen_spec_instances.py
        int kind[8] = {0}, atom[8] = {0}, lvI[8] = {0}, lvJ[8] = {0}, rowI[8] = {0}, rowJ[8] = {0};
        for (int q = 0; q < td.nslot; ++q) {
            const SlotDesc &sd = m->slots[td.slot0 + q];
            kind[q] = sd.isLine ? 1 : 0;
            atom[q] = sd.atom;
            lvI[q] = sd.lsI;
            lvJ[q] = sd.lsJ;
            rowI[q] = sd.rowI;
            rowJ[q] = sd.rowJ;
        }
        auto arr = [](const int *x) {
            std::string r = "{";
            for (int q = 0; q < 8; ++q) r += std::to_string(x[q]) + (q < 7 ? "," : "}");
            return r;
        };
        return "{" + std::to_string(Lw) + "," + std::to_string(td.nslot) + "," + std::to_string(d->Natom) + "," +
               std::to_string(td.nlevslot) + "," + arr(kind) + "," + arr(atom) + "," + arr(lvI) + "," + arr(lvJ) + "," +
               arr(rowI) + "," + arr(rowJ) + "," + std::to_string(d->Nrays) + "," + std::to_string(m->popsW) + "}";
    };
    auto fill_tile = [&](auto &t, const TileDesc &td, int spec) {
        t.la0 = td.la0;
        t.partRow0 = td.partRow0;
        t.spec = spec;
        t.recOff = td.recOff;
        for (int q = 0; q < td.nslot; ++q) {
            const SlotDesc &sd = m->slots[td.slot0 + q];
            SlotR &r = t.s[q];
            r.Nblue = sd.Nblue;
            r.Nlam = sd.Nlam;
            r.toff = sd.toff;
            r.cA = sd.c2;
            r.cB = sd.c1;
        }
    };
    const bool noSpec = getenv("MALI_NO_SPEC") != nullptr;
    // heaviest tiles first (the light ones fill the tail of a launch), and tiles of one structure next to each other
    // (co-resident blocks then run the same kernel instance: one instruction stream per SM)
    std::vector<const SpecEntry *> specOf(m->ntile, nullptr);
    for (int ti = 0; ti < m->ntile; ++ti) {
        const TileDesc &td = m->tiles[ti];
        if (!noSpec && td.nslot <= kSpecMaxSlots && d->Natom <= 4) specOf[ti] = find_spec(structure_key(td));
    }
    std::vector<int> order(m->ntile);
    for (int ti = 0; ti < m->ntile; ++ti) order[ti] = ti;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        if (m->tiles[a].nslot != m->tiles[b].nslot) return m->tiles[a].nslot > m->tiles[b].nslot;
        const int ia = specOf[a] ? specOf[a]->id : -1, ib = specOf[b] ? specOf[b]->id : -1;
        return ia < ib;
    });
    for (int ti : order) {
        const TileDesc &td = m->tiles[ti];
        const SpecEntry *e = specOf[ti];
        if (!e) {
            m->genericTiles.push_back(ti);
            continue;
        }
        const int sc = spec_class(td.nslot);
        if (sc == 0) {
            TileR<2> t{};
            fill_tile(t, td, e->id);
            m->spec0.push_back(t);
        } else if (sc == 1) {
            TileR<4> t{};
            fill_tile(t, td, e->id);
            m->spec1.push_back(t);
        } else {
            TileR<8> t{};
            fill_tile(t, td, e->id);
            m->spec2.push_back(t);
        }
        m->specTiles++;
    }
    // per-warp shared memory of the specialised kernels, per register class: the largest instance's need
    for (int c = 0; c < 3; ++c) m->smemClass[c] = 0;
    for (size_t ti = 0; ti < ptiles.size(); ++ti) {
        const PackTile &pt = ptiles[ti];
        if (pt.nslot > kSpecMaxSlots) continue;
        int &sm = m->smemClass[spec_class(pt.nslot)];
        sm = std::max(sm, fs_smem_bytes(pt.vb / kVRow, Lw, pt.nslot, m->tiles[ti].ngroup, m->popsW));
    }

    // ---- small copies of the upload path
    auto add_copy = [&](int64_t src, int64_t dst, int64_t len, int toPops, int derived) {
        CopyJob c{};
        c.srcOff = src;
        c.dstOff = dst;
        c.len = len;
        c.toPops = toPops;
        c.pad = derived;
        m->cjobs.push_back(c);
    };
    add_copy(L.hp_height, m->off_z, N, 0, 0);
    add_copy(L.hp_bbc, m->off_bbc, 2 * (int64_t)d->Nspect, 0, 0);
    add_copy(L.hp_nTotal, m->off_nTotal, (int64_t)d->Natom * N, 0, 0);
    add_copy(L.hp_C, m->off_C, (int64_t)m->sumNlevel2 * N, 0, 1);
    add_copy(L.hp_n, 0, (int64_t)m->sumNlevel * N, 1, 1);

    // ---- device copies of the model tables
    std::vector<double> zmu(d->Nrays), hw(d->Nrays);
    for (int q = 0; q < d->Nrays; ++q) {
        zmu[q] = 1.0 / d->muz[q];  // formal_solver.py:92
        hw[q] = 0.5 * d->wmu[q];   // rh_method.py:640,661
    }
    std::vector<double> alpha(d->alpha, d->alpha + ntab), twohc(d->twohc_l3, d->twohc_l3 + ntab),
        wlacont(d->wlacont, d->wlacont + ntab), wlambda(d->wlambda, d->wlambda + ntab);
    cudaError_t e = cudaSuccess;
    auto up = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    up(to_device(m->tiles, &m->d_tiles));
    up(to_device(m->slots, &m->d_slots));
    up(to_device(alpha, &m->d_alpha));
    up(to_device(twohc, &m->d_twohc));
    up(to_device(wlacont, &m->d_wlacont));
    up(to_device(wlambda, &m->d_wlambda));
    up(to_device(zmu, &m->d_zmu));
    up(to_device(hw, &m->d_hw));
    up(to_device(m->Nlevel, &m->d_Nlevel));
    up(to_device(m->lvlOff, &m->d_lvlOff));
    up(to_device(m->g2Off, &m->d_g2Off));
    up(to_device(m->trans, &m->d_trans));
    up(to_device(trPartOff, &m->d_trPartOff));
    up(to_device(trPartRows, &m->d_trPartRows));
    up(to_device(tileJ, &m->d_tileJ));
    {   // tables of the device compute_phi
        std::vector<PhiLine> lines;
        std::vector<PhiTile> tv;
        for (int t = 0; t < d->Ntrans; ++t) {
            const int32_t *tr = &m->trans[(size_t)t * 6];
            if (!tr[3]) continue;
            PhiLine ln{};
            ln.t = t;
            ln.atom = tr[0];
            ln.Nblue = tr[4];
            ln.Nlam = tr[5];
            ln.toff = m->toff[t];
            ln.tile0 = phiTile0[t];
            ln.tab0 = (int32_t)tv.size();
            ln.ntile = (int32_t)phiT[t].size();
            ln.lambda0 = d->lambda0 ? d->lambda0[t] : 0.0;
            ln.c0 = d->lineconst[3 * t + 0];
            lines.push_back(ln);
            tv.insert(tv.end(), phiT[t].begin(), phiT[t].end());
        }
        {   // tables of the device-side g_ij of the continua
            std::vector<GijCont> conts;
            std::vector<GijTile> gts;
            for (int t = 0; t < d->Ntrans; ++t) {
                const int32_t *tr = &m->trans[(size_t)t * 6];
                if (tr[3]) continue;
                GijCont gc{};
                gc.rowI = m->lvlOff[tr[0]] + tr[1];
                gc.rowJ = m->lvlOff[tr[0]] + tr[2];
                gc.Nblue = tr[4];
                gc.Nlam = tr[5];
                gc.tile0 = gijTile0[t];
                gc.toff = m->toff[t];
                gc.tab0 = (int32_t)gts.size();
                conts.push_back(gc);
                gts.insert(gts.end(), gijT[t].begin(), gijT[t].end());
            }
            m->nGijCont = (int)conts.size();
            up(to_device(conts, &m->d_gijCont));
            up(to_device(gts, &m->d_gijTiles));
        }
        m->nPhiLines = (int)lines.size();
        m->phiTilesHost = phiT;
        m->phiTile0Host = phiTile0;
        m->haveLambda0 = d->lambda0 != nullptr;
        up(to_device(lines, &m->d_phiLines));
        up(to_device(tv, &m->d_phiTiles));
        std::vector<double> wl(d->wavelength, d->wavelength + d->Nspect), mz(d->muz, d->muz + d->Nrays),
            wm(d->wmu, d->wmu + d->Nrays);
        up(to_device(wl, &m->d_wavelength));
        up(to_device(mz, &m->d_muz));
        up(to_device(wm, &m->d_wmu));
        std::vector<double> l0(d->Ntrans, 0.0);
        if (d->lambda0) l0.assign(d->lambda0, d->lambda0 + d->Ntrans);
        up(to_device(l0, &m->d_lambda0));
    }
    up(to_device(m->genericTiles, &m->d_genericTiles));
    {
        std::vector<int32_t> gt;
        for (int ti = 0; ti < m->ntile; ++ti)
            if (m->tiles[ti].ngroup > 0) gt.push_back(ti);
        m->nGroupTiles = (int)gt.size();
        up(to_device(gt, &m->d_groupTiles));
    }
    up(to_device(m->cjobs, &m->d_cjobs));
    up(to_device(pchunks, &m->d_pchunks));
    up(to_device(ptiles, &m->d_ptiles));
    up(to_device(pslots, &m->d_pslots));
    if (e != cudaSuccess) {
        mali_model_destroy(m);
        return fail((int)e, "mali_model_create: %s", cudaGetErrorString(e));
    }
    if (!getenv("MALI_SERIAL_CLASSES")) {   // side streams of launch_fs (MALI_SERIAL_CLASSES=1: one stream, for profiling)
        for (int q = 0; q < 2 && e == cudaSuccess; ++q) {
            e = cudaStreamCreateWithFlags(&m->sideStream[q], cudaStreamNonBlocking);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->joinEvent[q], cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->forkEvent, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&m->iterStream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->iterFork, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->iterJoin, cudaEventDisableTiming);
        if (e != cudaSuccess) {
            mali_model_destroy(m);
            return fail((int)e, "mali_model_create: %s", cudaGetErrorString(e));
        }
    }
    *out = m;
    return MALI_OK;
}

void mali_model_destroy(mali_model *m)
{
    if (!m) return;
    cudaSetDevice(m->device);
    void *ptrs[] = {m->d_tiles, m->d_slots, m->d_alpha, m->d_twohc, m->d_wlacont, m->d_wlambda, m->d_zmu, m->d_hw,
                    m->d_Nlevel, m->d_lvlOff, m->d_g2Off, m->d_trans, m->d_trPartOff, m->d_trPartRows,
                    m->d_genericTiles, m->d_cjobs, m->d_pchunks, m->d_ptiles, m->d_pslots, m->d_tileJ, m->d_phiTiles,
                    m->d_phiLines, m->d_wavelength, m->d_muz, m->d_wmu, m->d_gijCont, m->d_gijTiles, m->d_groupTiles, m->d_lambda0};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    for (void *p : m->atomDev)
        if (p) cudaFree(p);
    for (void *p : m->eosDev)
        if (p) cudaFree(p);
    if (m->d_depth) cudaFree(m->d_depth);
    for (auto &g : m->iterGraphs) cudaGraphExecDestroy(g.exec);
    for (cudaEvent_t e : m->profEvents) cudaEventDestroy(e);
    for (int q = 0; q < 2; ++q) {
        if (m->sideStream[q]) cudaStreamDestroy(m->sideStream[q]);
        if (m->joinEvent[q]) cudaEventDestroy(m->joinEvent[q]);
    }
    if (m->forkEvent) cudaEventDestroy(m->forkEvent);
    if (m->iterStream) cudaStreamDestroy(m->iterStream);
    if (m->iterFork) cudaEventDestroy(m->iterFork);
    if (m->iterJoin) cudaEventDestroy(m->iterJoin);
    delete m;
}

int mali_model_set_arith(mali_model *m, int32_t mode)
{
    if (!m || (mode != MALI_ARITH_EXACT && mode != MALI_ARITH_CONTRACTED)) return fail(MALI_EINVAL, "mali_model_set_arith: bad argument");
    m->arith = mode;
    return MALI_OK;
}

int mali_model_get_arith(const mali_model *m) { return m ? m->arith : MALI_EINVAL; }

int mali_model_layout(const mali_model *m, mali_layout *out)
{
    if (!m || !out) return fail(MALI_EINVAL, "mali_model_layout: null argument");
    *out = m->lay;
    return MALI_OK;
}

int mali_model_info(const mali_model *m, int32_t *out8)
{
    if (!m || !out8) return fail(MALI_EINVAL, "mali_model_info: null argument");
    out8[0] = m->ntile;
    out8[1] = m->specTiles;
    out8[2] = (int32_t)m->genericTiles.size();
    out8[3] = m->Tmax;
    out8[4] = m->Dmax;
    out8[5] = (int32_t)m->rowStride;
    out8[6] = std::max(m->smemClass[0], std::max(m->smemClass[1], m->smemClass[2]));
    out8[7] = 1;
    return MALI_OK;
}

static int check_range(const mali_model *m, const mali_buffers *b, int col0, int ncol, const char *who)
{
    if (!m || !b) return fail(MALI_EINVAL, "%s: null argument", who);
    if (col0 < 0 || ncol < 1 || col0 + ncol > b->ncol) return fail(MALI_EINVAL, "%s: columns [%d, %d) outside the batch of %d", who, col0, col0 + ncol, b->ncol);
    return MALI_OK;
}

// the continuum groups' U sums follow from the g_ij fields: called by whichever path has just (re)written those
static void launch_cont_groups(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, cudaStream_t st)
{
    if (m->nGroupTiles == 0) return;
    dim3 grid((m->N * m->Lw + 127) / 128, m->nGroupTiles, ncol);
    cont_group_kernel<<<grid, 128, 0, st>>>(m->d_tiles, m->d_slots, m->d_groupTiles, m->d_twohc, m->N, m->Nspect,
                                            m->Lw, b->colconst, m->lay.colconst, m->off_tab, col0);
    m->launches += 1;
}

// mode 0: whole host-pack blocks; 1: without the line profiles (mali_compute_phi forms them); 2: only the blocks'
// first hp_C doubles -- heights, boundary Planck values, nTotal, background -- (mali_setup_columns forms C, the
// continua's g_ij and the LTE populations as well); 3: only the first hp_bg_chi doubles (mali_background forms the
// background opacities, too)
static int upload_columns(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, const double *host_pack,
                          double *staging_dev, void *stream, int mode)
{
    const bool nophi = mode >= 1;
    if (int r = check_range(m, b, col0, ncol, "mali_upload_columns")) return r;
    if (!staging_dev || !b->colconst || !b->pops || !b->J) return fail(MALI_EINVAL, "mali_upload_columns: null buffer");
    cudaStream_t st = (cudaStream_t)stream;
    const mali_layout &L = m->lay;
    if (host_pack) {
        if (!nophi)
            CU(cudaMemcpyAsync(staging_dev, host_pack, (size_t)ncol * L.hostpack * sizeof(double), cudaMemcpyHostToDevice, st));
        else {  // only the blocks' prefix without the line profiles (/ the derived blocks) crosses the bus
            const size_t pre = (size_t)(mode == 3 ? L.hp_bg_chi : (mode == 2 ? L.hp_C : L.hp_phi)) * sizeof(double);
            CU(cudaMemcpy2DAsync(staging_dev, (size_t)L.hostpack * sizeof(double), host_pack, pre, pre, (size_t)ncol,
                                 cudaMemcpyHostToDevice, st));
        }
    }
    const int nPackChunks = nophi ? m->packChunksFields : m->packChunks;
    if (nPackChunks > 0) {
        dim3 grid(nPackChunks, (m->N + 31) / 32, ncol), block(32, 8);
        pack_tiles_kernel<<<grid, block, 0, st>>>(m->d_pchunks, m->d_ptiles, m->d_pslots, m->d_wlambda, m->d_alpha, m->N, m->Nrays,
                                                  m->Nspect, m->Lw, staging_dev, L.hostpack, L.hp_bg_chi, L.hp_bg_eta,
                                                  L.hp_bg_sca, b->colconst, L.colconst, m->off_tab, col0, mode);
    }
    {
        dim3 grid(32, ncol);
        pack_misc_kernel<<<grid, 256, 0, st>>>(m->d_cjobs, (int)m->cjobs.size(), staging_dev, L.hostpack, b->colconst,
                                               L.colconst, b->pops, L.pops, b->J, L.J, col0, mode >= 2 ? 1 : 0);
    }
    m->launches += 2;
    if (mode < 2) launch_cont_groups(m, b, col0, ncol, st);   // (otherwise mali_setup_columns forms the g_ij fields)
    CU(cudaGetLastError());
    return MALI_OK;
}

int mali_upload_columns(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, const double *host_pack,
                        double *staging_dev, void *stream)
{
    return upload_columns(m, b, col0, ncol, host_pack, staging_dev, stream, 0);
}

int mali_upload_columns_nophi(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol,
                              const double *host_pack_prefix, double *staging_dev, void *stream)
{
    return upload_columns(m, b, col0, ncol, host_pack_prefix, staging_dev, stream, 1);
}

int mali_upload_columns_atmos(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol,
                              const double *host_pack_prefix, double *staging_dev, void *stream)
{
    return upload_columns(m, b, col0, ncol, host_pack_prefix, staging_dev, stream, 2);
}

int mali_upload_columns_thermo(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol,
                               const double *host_pack_prefix, double *staging_dev, void *stream)
{
    return upload_columns(m, b, col0, ncol, host_pack_prefix, staging_dev, stream, 3);
}

int mali_model_set_eos(mali_model *m, const mali_eos_desc *d)
{
    if (!m || !d || !d->tpf || !d->pf || !d->eion || !d->stage_off || !d->abund || d->npf < 2)
        return fail(MALI_EINVAL, "mali_model_set_eos: bad argument");
    CU(cudaSetDevice(m->device));
    for (void *p : m->eosDev)
        if (p) cudaFree(p);
    m->eosDev.clear();
    cudaError_t e = cudaSuccess;
    auto put = [&](const void *src, size_t bytes) -> void * {
        void *dv = nullptr;
        if (e == cudaSuccess) e = cudaMalloc(&dv, std::max<size_t>(bytes, 8));
        if (e == cudaSuccess && bytes) e = cudaMemcpy(dv, src, bytes, cudaMemcpyHostToDevice);
        m->eosDev.push_back(dv);
        return dv;
    };
    const int nst = d->stage_off[eos::kNcontr];
    for (int q = 0; q < eos::kNcontr; ++q) {
        const int ns = d->stage_off[q + 1] - d->stage_off[q];
        if (ns < 2 || ns > eos::kMaxStage) return fail(MALI_ELIMIT, "mali_model_set_eos: element %d has %d stages (2..%d)", q, ns, eos::kMaxStage);
    }
    EosParams &P = m->eos;
    P = EosParams{};
    P.E.npf = d->npf;
    P.E.tpf = (const double *)put(d->tpf, d->npf * sizeof(double));
    P.E.pf = (const double *)put(d->pf, (size_t)nst * d->npf * sizeof(double));
    P.E.eion = (const double *)put(d->eion, nst * sizeof(double));
    P.E.stageOff = (const int32_t *)put(d->stage_off, (eos::kNcontr + 1) * sizeof(int32_t));
    P.E.abund = (const double *)put(d->abund, 99 * sizeof(double));
    P.E.avw = d->avw;
    P.E.rho_from_H = d->rho_from_H;
    P.E.ab_others = d->ab_others;
    P.E.saha_fac = d->saha_fac;
    P.E.prec = d->prec;
    P.amu_wph = d->amu_weight_per_H;
    P.cm3 = d->cm_to_m_cubed;
    P.g_to_kg = 1.0E-03;
    P.cm_to_m = 1.0E-02;
    P.thomson = d->thomson_sigma;
    if (e != cudaSuccess) return fail((int)e, "mali_model_set_eos: %s", cudaGetErrorString(e));
    m->haveEos = true;
    return MALI_OK;
}

int mali_background(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, const double *T,
                    const double *ne, const double *nHTot, const double *cmass, double *work, void *stream)
{
    if (int r = check_range(m, b, col0, ncol, "mali_background")) return r;
    if (!T || !ne || !nHTot || !work || !b->colconst) return fail(MALI_EINVAL, "mali_background: null buffer");
    if (!m->haveEos) return fail(MALI_EINVAL, "mali_background: call mali_model_set_eos first");
    cudaStream_t st = (cudaStream_t)stream;
    const int n = m->N * ncol;
    eos_kernel<<<(n + 63) / 64, 64, 0, st>>>(m->eos, m->N, ncol, T, nHTot, work);
    dim3 grid((m->N + 63) / 64, m->Nspect, ncol);
    background_kernel<<<grid, 64, 0, st>>>(m->eos, m->d_tiles, m->d_wavelength, m->N, m->Nspect, m->Lw, T, ne, work,
                                           b->colconst, m->lay.colconst, m->off_tab, col0);
    m->launches += 2;
    if (cmass) {   // the caller's depth scale is column mass: heights come from here as well (atmosphere.py:94-111)
        double *tau = work + (size_t)n * kEosWork;
        convert_scales_kernel<<<(ncol + 31) / 32, 32, 0, st>>>(m->eos, m->N, ncol, cmass, nHTot, work, b->colconst,
                                                               m->lay.colconst, m->off_z, col0, tau);
        m->launches += 1;
    }
    CU(cudaGetLastError());
    return MALI_OK;
}

int mali_model_set_atoms(mali_model *m, const mali_atom_desc *a)
{
    if (!m || !a) return fail(MALI_EINVAL, "mali_model_set_atoms: null argument");
    if (a->Natom != m->Natom) return fail(MALI_EINVAL, "mali_model_set_atoms: %d atoms, the model has %d", a->Natom, m->Natom);
    for (int q = 0; q < m->Natom; ++q)
        if (a->Nlevel[q] != m->Nlevel[q]) return fail(MALI_EINVAL, "mali_model_set_atoms: atom %d has %d levels, the model %d", q, a->Nlevel[q], m->Nlevel[q]);
    CU(cudaSetDevice(m->device));
    const int nl = m->sumNlevel;
    int nk = 0, ncf = 0;
    for (int c = 0; c < a->Ncoll; ++c) {
        const int32_t *cd = a->coll + 8 * c;
        const bool bad = cd[0] < 0 || cd[0] >= m->Natom || cd[1] < 0 || cd[1] > 2 || cd[2] < 0 || cd[3] < 0 ||
                         cd[2] >= m->Nlevel[cd[0]] || cd[3] >= m->Nlevel[cd[0]] || cd[4] < 2 || cd[5] != nk || cd[6] != ncf ||
                         (cd[7] && cd[4] < 4);
        if (bad) return fail(MALI_EINVAL, "mali_model_set_atoms: collision %d: inconsistent descriptor", c);
        nk += cd[7] ? cd[4] + 4 : cd[4];
        ncf += cd[4];
    }
    for (void *p : m->atomDev)
        if (p) cudaFree(p);
    m->atomDev.clear();
    cudaError_t e = cudaSuccess;
    auto put = [&](const void *src, size_t bytes) -> void * {
        void *d = nullptr;
        if (e == cudaSuccess) e = cudaMalloc(&d, std::max<size_t>(bytes, 8));
        if (e == cudaSuccess && bytes) e = cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice);
        m->atomDev.push_back(d);
        return d;
    };
    AtomLevels &A = m->atoms;
    A = AtomLevels{};
    A.Nlevel = m->d_Nlevel;
    A.lvlOff = m->d_lvlOff;
    A.g2Off = m->d_g2Off;
    A.dE = (const double *)put(a->dE, nl * sizeof(double));
    A.gi0 = (const double *)put(a->gi0, nl * sizeof(double));
    A.nDebye = (const double *)put(a->nDebye, nl * sizeof(double));
    A.g = (const double *)put(a->g, nl * sizeof(double));
    A.dZ = (const int32_t *)put(a->dZ, nl * sizeof(int32_t));
    A.vTherm = (const double *)put(a->vTherm, m->Natom * sizeof(double));
    A.coll = (const int32_t *)put(a->coll, (size_t)a->Ncoll * 8 * sizeof(int32_t));
    A.knots = (const double *)put(a->knots, nk * sizeof(double));
    A.coef = (const double *)put(a->coef, (size_t)ncf * sizeof(double));
    A.fill = (const double *)put(a->fill, (size_t)a->Ncoll * 2 * sizeof(double));
    A.par = (const double *)put(a->par, (size_t)a->Ncoll * sizeof(double));
    A.c1 = a->c1;
    A.c2 = a->c2;
    A.Ncoll = a->Ncoll;
    A.Natom = m->Natom;
    if (e != cudaSuccess) return fail((int)e, "mali_model_set_atoms: %s", cudaGetErrorString(e));
    m->haveAtoms = true;
    return MALI_OK;
}

int mali_setup_columns(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, const double *T,
                       const double *ne, const double *vturb, double *nStar, double *vBroad, int32_t start_from_lte,
                       void *stream)
{
    if (int r = check_range(m, b, col0, ncol, "mali_setup_columns")) return r;
    if (!T || !ne || !vturb || !nStar || !vBroad || !b->colconst || !b->pops) return fail(MALI_EINVAL, "mali_setup_columns: null buffer");
    if (!m->haveAtoms) return fail(MALI_EINVAL, "mali_setup_columns: call mali_model_set_atoms first");
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid((m->N + 63) / 64, m->Natom, ncol);
    double *pops = start_from_lte ? b->pops : nullptr;
    if (m->maxNlevel <= 8)
        setup_levels_kernel<8><<<grid, 64, 0, st>>>(m->atoms, m->N, T, ne, vturb, b->colconst, m->lay.colconst, m->off_C,
                                                    m->off_nTotal, nStar, vBroad, pops, m->lay.pops, m->sumNlevel, col0);
    else
        setup_levels_kernel<16><<<grid, 64, 0, st>>>(m->atoms, m->N, T, ne, vturb, b->colconst, m->lay.colconst, m->off_C,
                                                     m->off_nTotal, nStar, vBroad, pops, m->lay.pops, m->sumNlevel, col0);
    m->launches += 1;
    if (m->nGijCont > 0) {
        dim3 g2(8, m->nGijCont, ncol);
        setup_gij_kernel<<<g2, 256, 0, st>>>(m->d_gijCont, m->d_gijTiles, m->d_wavelength, m->d_alpha, m->N, m->Lw, m->sumNlevel, T, nStar,
                                             b->colconst, m->lay.colconst, m->off_tab, col0);
        m->launches += 1;
        launch_cont_groups(m, b, col0, ncol, st);
    }
    CU(cudaGetLastError());
    return MALI_OK;
}

int mali_compute_phi(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, const double *aDamp,
                     const double *vBroad, const double *vlos, void *stream)
{
    if (int r = check_range(m, b, col0, ncol, "mali_compute_phi")) return r;
    if (!aDamp || !vBroad || !vlos || !b->colconst) return fail(MALI_EINVAL, "mali_compute_phi: null buffer");
    if (!m->haveLambda0) return fail(MALI_EINVAL, "mali_compute_phi: the model was created without lambda0");
    if (m->nPhiLines == 0) return MALI_OK;
    dim3 grid((m->N + 3) / 4, m->nPhiLines, ncol);     // 4 warps per block, one depth point each
    compute_phi_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(
        m->d_phiLines, m->d_phiTiles, m->d_wavelength, m->d_wlambda, m->d_muz, m->d_wmu,
        m->N, m->Nrays, m->Nspect, m->Lw, m->Ntrans, m->Natom, aDamp, vBroad, vlos, b->colconst, m->lay.colconst, m->off_tab,
        col0);
    m->launches += 1;
    CU(cudaGetLastError());
    return MALI_OK;
}

int mali_perturb_columns(const mali_model *m, const mali_buffers *b, int32_t src_col, int32_t col0, int32_t ncol,
                         const mali_perturb_desc *d, void *stream)
{
    if (int r = check_range(m, b, col0, ncol, "mali_perturb_columns")) return r;
    if (src_col < 0 || src_col >= b->ncol) return fail(MALI_EINVAL, "mali_perturb_columns: source column %d outside the batch of %d", src_col, b->ncol);
    if (src_col >= col0 && src_col < col0 + ncol)
        return fail(MALI_EINVAL, "mali_perturb_columns: source column %d inside the range [%d, %d)", src_col, col0, col0 + ncol);
    if (!d || !d->depth || !d->T || !d->ne || !d->nHTot || !d->vturb || !d->vlos || !d->aDamp || !d->pops0 || !d->src_work ||
        !d->src_nStar || !d->src_vBroad || !d->work || !d->nStar || !d->vBroad || !b->colconst || !b->pops || !b->J)
        return fail(MALI_EINVAL, "mali_perturb_columns: null argument");
    if (!m->haveEos || !m->haveAtoms) return fail(MALI_EINVAL, "mali_perturb_columns: call mali_model_set_eos and mali_model_set_atoms first");
    if (m->nPhiLines > 0 && !m->haveLambda0) return fail(MALI_EINVAL, "mali_perturb_columns: the model was created without lambda0");
    for (int c = 0; c < ncol; ++c)
        if (d->depth[c] < 0 || d->depth[c] >= m->N)
            return fail(MALI_EINVAL, "mali_perturb_columns: depth[%d]=%d not in [0, %d)", c, d->depth[c], m->N);
    cudaStream_t st = (cudaStream_t)stream;
    if (ncol > m->depthCap) {
        if (m->d_depth) CU(cudaFree(m->d_depth));
        m->d_depth = nullptr;
        m->depthCap = 0;
        CU(cudaMalloc((void **)&m->d_depth, (size_t)ncol * sizeof(int32_t)));
        m->depthCap = ncol;
    }
    CU(cudaMemcpyAsync(m->d_depth, d->depth, (size_t)ncol * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    PerturbParams p{};
    p.N = m->N;
    p.Nspect = m->Nspect;
    p.Lw = m->Lw;
    p.sumNlevel = m->sumNlevel;
    p.Natom = m->Natom;
    p.col0 = col0;
    p.src = src_col;
    p.colStride = m->lay.colconst;
    p.popStride = m->lay.pops;
    p.JStride = m->lay.J;
    p.off_bbc = m->off_bbc;
    p.off_tab = m->off_tab;
    p.depth = m->d_depth;
    p.T = d->T;
    p.ne = d->ne;
    p.nHTot = d->nHTot;
    p.vturb = d->vturb;
    p.bbc = d->bbc;
    p.pops0 = d->pops0;
    p.srcWork = d->src_work;
    p.srcNStar = d->src_nStar;
    p.srcVBroad = d->src_vBroad;
    p.work = d->work;
    p.nStar = d->nStar;
    p.vBroad = d->vBroad;
    p.colconst = b->colconst;
    p.pops = b->pops;
    p.J = b->J;
    // 1. clone
    const int nb = (int)std::min<int64_t>(64, (m->lay.colconst / 2 + 255) / 256);
    perturb_clone_kernel<<<dim3(nb, ncol), 256, 0, st>>>(p);
    // 2. re-form depth[c]: EOS point, then background and levels (both read it), then g_ij, groups and profiles
    perturb_eos_kernel<<<(ncol + 63) / 64, 64, 0, st>>>(m->eos, p, ncol);
    perturb_background_kernel<<<dim3((m->Nspect + 63) / 64, ncol), 64, 0, st>>>(m->eos, m->d_tiles, m->d_wavelength, d->ne, p);
    const int na = ncol * m->Natom;
    if (m->maxNlevel <= 8)
        perturb_levels_kernel<8><<<(na + 63) / 64, 64, 0, st>>>(m->atoms, p, m->off_C, m->off_nTotal, ncol);
    else
        perturb_levels_kernel<16><<<(na + 63) / 64, 64, 0, st>>>(m->atoms, p, m->off_C, m->off_nTotal, ncol);
    m->launches += 4;
    if (m->nGijCont > 0) {
        perturb_gij_kernel<<<dim3(m->nGijCont, ncol), 64, 0, st>>>(m->d_gijCont, m->d_gijTiles, m->d_wavelength, m->d_alpha, p);
        m->launches += 1;
        if (m->nGroupTiles > 0) {
            perturb_group_kernel<<<dim3(m->nGroupTiles, ncol), m->Lw, 0, st>>>(m->d_tiles, m->d_slots, m->d_groupTiles, m->d_twohc, p);
            m->launches += 1;
        }
    }
    if (m->nPhiLines > 0) {
        perturb_phi_kernel<<<dim3(m->nPhiLines, ncol), 32, 0, st>>>(m->d_phiLines, m->d_phiTiles, m->d_wavelength, m->d_wlambda,
                                                                     m->d_muz, m->d_wmu, m->Nrays, m->Ntrans, d->aDamp, d->vlos, p);
        m->launches += 1;
    }
    // 3. heights from the column mass over the whole range (the recurrence is not local in depth)
    if (d->cmass) {
        double *tau = d->work + (size_t)ncol * m->N * kEosWork;
        convert_scales_kernel<<<(ncol + 31) / 32, 32, 0, st>>>(m->eos, m->N, ncol, d->cmass, d->nHTot, d->work, b->colconst,
                                                               m->lay.colconst, m->off_z, col0, tau);
        m->launches += 1;
    }
    CU(cudaGetLastError());
    return MALI_OK;
}

// The argument checks of mali_compute_rays and mali_compute_rays_depth, and the kernel parameters they share (the
// outputs are left null for the caller to set).
static int rays_params(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, int32_t nmu,
                       const double *mu, const double *aDamp, const double *vBroad, const double *vlos, int32_t *bad,
                       const char *who, RaysParams &p)
{
    if (int r = check_range(m, b, col0, ncol, who)) return r;
    if (!b->colconst || !b->pops || !b->J) return fail(MALI_EINVAL, "%s: null buffer", who);
    if (nmu < 1 || nmu > MALI_RAYS_MAX_MU || !mu)
        return fail(MALI_EINVAL, "%s: nmu=%d not in [1, %d] (or no angles)", who, nmu, MALI_RAYS_MAX_MU);
    for (int q = 0; q < nmu; ++q)
        if (!(mu[q] > 0.0 && mu[q] <= 1.0)) return fail(MALI_EINVAL, "%s: mu[%d]=%g not in (0, 1]", who, q, mu[q]);
    if (m->nPhiLines > 0) {   // the line profiles are formed at the new angles from the per-call inputs
        if (!m->haveLambda0) return fail(MALI_EINVAL, "%s: the model was created without lambda0", who);
        if (!aDamp || !vBroad || !vlos) return fail(MALI_EINVAL, "%s: null aDamp / vBroad / vlos", who);
    }
    static_assert(kRaysMaxMu == MALI_RAYS_MAX_MU, "mali_rays.cuh and mali_b200.h disagree on the angle limit");
    p = RaysParams{};
    p.N = m->N;
    p.Nrays = m->Nrays;
    p.Nspect = m->Nspect;
    p.Natom = m->Natom;
    p.Ntrans = m->Ntrans;
    p.Lw = m->Lw;
    p.ntile = m->ntile;
    p.nchunk = (nmu + m->Nrays - 1) / m->Nrays;
    p.nmu = nmu;
    p.col0 = col0;
    p.ncol = ncol;
    p.colStride = m->lay.colconst;
    p.popStride = m->lay.pops;
    p.JStride = m->lay.J;
    p.off_z = m->off_z;
    p.off_bbc = m->off_bbc;
    p.off_tab = m->off_tab;
    p.tiles = m->d_tiles;
    p.slots = m->d_slots;
    p.alpha = m->d_alpha;
    p.twohc = m->d_twohc;
    p.wavelength = m->d_wavelength;
    p.lambda0 = m->d_lambda0;
    p.colconst = b->colconst;
    p.pops = b->pops;
    p.J = b->J;
    p.aDamp = aDamp;
    p.vBroad = vBroad;
    p.vlos = vlos;
    p.bad = bad;
    for (int q = 0; q < nmu; ++q) {
        p.mu[q] = mu[q];
        p.zmu[q] = 1.0 / mu[q];   // formal_solver.py:92, as mali_model_create forms zmu
    }
    return MALI_OK;
}

static int launch_rays(const mali_model *m, const RaysParams &p, bool depth, void *stream)
{
    const int64_t warps = (int64_t)p.ncol * p.ntile * p.nchunk;
    const int wpb = 4;
    (depth ? rays_kernel<true> : rays_kernel<false>)<<<(unsigned)((warps + wpb - 1) / wpb), 32 * wpb, 0, (cudaStream_t)stream>>>(p);
    m->launches += 1;
    CU(cudaGetLastError());
    return MALI_OK;
}

int mali_compute_rays(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, int32_t nmu, const double *mu,
                      const double *aDamp, const double *vBroad, const double *vlos, double *I_out, int32_t *bad, void *stream)
{
    RaysParams p;
    if (int r = rays_params(m, b, col0, ncol, nmu, mu, aDamp, vBroad, vlos, bad, "mali_compute_rays", p)) return r;
    if (!I_out) return fail(MALI_EINVAL, "mali_compute_rays: null buffer");
    p.I = I_out;
    return launch_rays(m, p, false, stream);
}

int mali_compute_rays_depth(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, int32_t nmu,
                            const double *mu, const double *aDamp, const double *vBroad, const double *vlos,
                            const mali_rays_depth_out *out, int32_t *bad, void *stream)
{
    RaysParams p;
    if (int r = rays_params(m, b, col0, ncol, nmu, mu, aDamp, vBroad, vlos, bad, "mali_compute_rays_depth", p)) return r;
    if (!out || !(out->I || out->chi || out->S || out->tau || out->contrib || out->z_tau1 || out->height))
        return fail(MALI_EINVAL, "mali_compute_rays_depth: no output requested");
    if ((out->contrib || out->z_tau1) && !out->tau)
        return fail(MALI_EINVAL, "mali_compute_rays_depth: contrib and z_tau1 need the tau buffer");
    if (out->height) {   // the heights the sweep reads: colconst's z rows
        const size_t N = (size_t)m->N;
        CU(cudaMemcpy2DAsync(out->height, N * sizeof(double), b->colconst + (size_t)col0 * m->lay.colconst + m->off_z,
                             (size_t)m->lay.colconst * sizeof(double), N * sizeof(double), (size_t)ncol,
                             cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    }
    if (!(out->I || out->chi || out->S || out->tau)) return MALI_OK;
    p.dI = out->I;
    p.dchi = out->chi;
    p.dS = out->S;
    p.dtau = out->tau;
    p.dcontrib = out->contrib;
    p.ztau1 = out->z_tau1;
    return launch_rays(m, p, true, stream);
}

int mali_compute_rates(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, double *Rij_out,
                       double *Rji_out, int32_t *bad, void *stream)
{
    if (int r = check_range(m, b, col0, ncol, "mali_compute_rates")) return r;
    if (!b->colconst || !b->pops || !b->J || !b->scratch) return fail(MALI_EINVAL, "mali_compute_rates: null buffer");
    if (m->Ntrans == 0) return MALI_OK;   // empty outputs (which may be null): nothing to write
    if (!Rij_out || !Rji_out) return fail(MALI_EINVAL, "mali_compute_rates: null output");
    RatesParams p{};
    p.N = m->N;
    p.Nrays = m->Nrays;
    p.Nspect = m->Nspect;
    p.Lw = m->Lw;
    p.ntile = m->ntile;
    p.Ntrans = m->Ntrans;
    p.col0 = col0;
    p.ncol = ncol;
    p.colStride = m->lay.colconst;
    p.popStride = m->lay.pops;
    p.JStride = m->lay.J;
    p.scratchStride = m->lay.scratch;
    p.off_z = m->off_z;
    p.off_bbc = m->off_bbc;
    p.off_tab = m->off_tab;
    p.off_part = m->off_part;
    p.upOff = m->upOff;
    p.tiles = m->d_tiles;
    p.slots = m->d_slots;
    p.alpha = m->d_alpha;
    p.twohc = m->d_twohc;
    p.wlacont = m->d_wlacont;
    p.zmu = m->d_zmu;
    p.hw = m->d_hw;
    p.colconst = b->colconst;
    p.pops = b->pops;
    p.J = b->J;
    p.scratch = b->scratch;
    p.trPartOff = m->d_trPartOff;
    p.trPartRows = m->d_trPartRows;
    p.Rij = Rij_out;
    p.Rji = Rji_out;
    p.bad = bad;
    const cudaStream_t st = (cudaStream_t)stream;
    const int64_t warps = (int64_t)ncol * m->ntile * 2;
    const int wpb = 4;
    rates_kernel<<<(unsigned)((warps + wpb - 1) / wpb), 32 * wpb, 0, st>>>(p);
    rates_finish_kernel<<<dim3((m->N + 127) / 128, m->Ntrans, ncol), 128, 0, st>>>(p);
    m->launches += 2;
    CU(cudaGetLastError());
    return MALI_OK;
}

static FsParams make_fs_params(const mali_model *m, const mali_buffers *b, int col0, int ncol, int wpb)
{
    FsParams p{};
    p.N = m->N;
    p.Nrays = m->Nrays;
    p.Nspect = m->Nspect;
    p.Natom = m->Natom;
    p.Ntrans = m->Ntrans;
    p.Lw = m->Lw;
    p.ntile = m->ntile;
    p.Dmax = std::max(m->Dmax, 1);
    p.col0 = col0;
    p.ncol = ncol;
    p.warpsPerBlock = wpb;
    p.blocksPerCol = (m->ntile + wpb - 1) / wpb;
    p.smemPerWarp = (2 * p.Dmax + m->Natom) * 32;
    p.colStride = m->lay.colconst;
    p.popStride = m->lay.pops;
    p.JStride = m->lay.J;
    p.IStride = m->lay.I;
    p.scratchStride = m->lay.scratch;
    p.off_z = m->off_z;
    p.off_bbc = m->off_bbc;
    p.off_tab = m->off_tab;
    p.off_jpart = m->off_jpart;
    p.off_part = m->off_part;
    p.upOff = m->upOff;
    p.tiles = m->d_tiles;
    p.slots = m->d_slots;
    p.classTiles = m->d_genericTiles;
    p.nClassTiles = (int32_t)m->genericTiles.size();
    p.alpha = m->d_alpha;
    p.twohc = m->d_twohc;
    p.wlacont = m->d_wlacont;
    p.zmu = m->d_zmu;
    p.hw = m->d_hw;
    p.colconst = b->colconst;
    p.pops = b->pops;
    p.J = b->J;
    p.I = b->I;
    p.scratch = b->scratch;
    p.dJbits = reinterpret_cast<unsigned long long *>(b->dJ);
    p.status = b->status;
    p.done = b->done;
    return p;
}

static FsCommon make_fs_common(const mali_model *m, const mali_buffers *b, int col0, int ncol)
{
    FsCommon c{};
    c.N = m->N;
    c.Nrays = m->Nrays;
    c.Nspect = m->Nspect;
    c.Lw = m->Lw;
    c.col0 = col0;
    c.ncol = ncol;
    c.popsW = m->popsW;
    // launch order (mali_fs_class.cu): slabs of 512 columns, the two directions of a tile next to each other: measured
    // 17.2 GB of DRAM traffic per launch instead of 21.7 GB (a column's popsT rows are found in L2 by the later tiles)
    // at the same or slightly better time; slabs of 128 columns cut the traffic to 15.8 GB but put ~14 kernel
    // instances on an SM at once and lose 36 % to instruction-cache misses (profiles/r02_launch_order.txt)
    static const int colChunk = getenv("MALI_COL_CHUNK") ? atoi(getenv("MALI_COL_CHUNK")) : 512;
    static const int dirInter = getenv("MALI_DIR_INTERLEAVE") ? atoi(getenv("MALI_DIR_INTERLEAVE")) : 1;
    c.colChunk = std::max(1, std::min(colChunk, ncol));
    c.dirInterleave = dirInter;
    c.colStride = m->lay.colconst;
    c.IStride = m->lay.I;
    c.scratchStride = m->lay.scratch;
    c.off_bbc = m->off_bbc;
    c.off_tab = m->off_tab;
    c.off_popsT = m->off_popsT;
    c.off_jpart = m->off_jpart;
    c.off_part = m->off_part;
    c.upOff = m->upOff;
    c.alpha = m->d_alpha;
    c.twohc = m->d_twohc;
    c.wlacont = m->d_wlacont;
    c.zmu = m->d_zmu;
    c.hw = m->d_hw;
    c.colconst = b->colconst;
    c.I = b->I;
    c.scratch = b->scratch;
    c.status = b->status;
    c.done = b->done;
    return c;
}

static FinishParams make_finish_params(const mali_model *m, const mali_buffers *b, int col0, int ncol)
{
    FinishParams p{};
    p.N = m->N;
    p.Natom = m->Natom;
    p.Ntrans = m->Ntrans;
    p.col0 = col0;
    p.ncol = ncol;
    p.sumNlevel = m->sumNlevel;
    p.sumNlevel2 = m->sumNlevel2;
    p.colStride = m->lay.colconst;
    p.popStride = m->lay.pops;
    p.gammaStride = m->lay.Gamma;
    p.scratchStride = m->lay.scratch;
    p.off_C = m->off_C;
    p.off_nTotal = m->off_nTotal;
    p.off_part = m->off_part;
    p.upOff = m->upOff;
    p.Nlevel = m->d_Nlevel;
    p.lvlOff = m->d_lvlOff;
    p.g2Off = m->d_g2Off;
    p.trans = m->d_trans;
    p.trPartOff = m->d_trPartOff;
    p.trPartRows = m->d_trPartRows;
    p.colconst = b->colconst;
    p.pops = b->pops;
    p.Gamma = b->Gamma;
    p.scratch = b->scratch;
    p.dPopsBits = reinterpret_cast<unsigned long long *>(b->dPops);
    p.status = b->status;
    p.done = b->done;
    return p;
}

// ctl.on: called from mali_iterate -- the prepare kernel closes the previous iteration, and j_finish_kernel (which only
// the NEXT formal solution and the convergence test depend on) runs on a side stream next to the statistical
// equilibrium; *jJoin then tells the caller to join that stream (event joinEvent[0]) at the end of the iteration.
static int launch_fs(const mali_model *m, const mali_buffers *b, int col0, int ncol, cudaStream_t st, const IterCtl &ctl,
                     bool *jJoin)
{
    fs_prepare_kernel<<<ncol, 128, 0, st>>>(reinterpret_cast<unsigned long long *>(b->dJ), b->done, col0, b->colconst,
                                            m->lay.colconst, m->off_z, m->off_popsT, m->popsW, m->N, m->sumNlevel, b->pops,
                                            m->lay.pops, ctl);
    m->launches += 1;
    const bool rec = m->profOn && m->profUsed + 2 <= (int)m->profEvents.size();
    if (rec) cudaEventRecord(m->profEvents[m->profUsed], st);
    // heaviest work first so that the light tiles fill the tail
    if (!m->genericTiles.empty()) {  // tiles without a specialised instance (any slot count, any number of atoms)
        const int wpb = 1;
        FsParams p = make_fs_params(m, b, col0, ncol, wpb);
        const size_t smem = (size_t)p.smemPerWarp * wpb * sizeof(double);
        if (smem > 227 * 1024) return fail(MALI_ELIMIT, "tile needs %zu B of shared memory", smem);
        const int nt = (int)m->genericTiles.size();
        p.blocksPerCol = (nt + wpb - 1) / wpb;
        fs_gamma_kernel<<<(unsigned)(p.blocksPerCol * ncol), 32 * wpb, smem, st>>>(p);
        m->launches += 1;
    }
    if (m->specTiles > 0) {
        const FsCommon cc = make_fs_common(m, b, col0, ncol);
        size_t smem[3];
        for (int cls = 0; cls < 3; ++cls) {
            smem[cls] = (size_t)m->smemClass[cls];
            if (smem[cls] > 227 * 1024) return fail(MALI_ELIMIT, "a tile needs %zu B of shared memory per warp", smem[cls]);
        }
        // fork: class 2 (heaviest warps) stays on the caller's stream, classes 1 and 0 go to the side streams
        // -- only for small launches (a few waves of warps: single columns, response-function batches), where the
        // serial tails are a large share; big batches fill the machine anyway and keep to one stream
        static const int64_t forkMax = getenv("MALI_FORK_MAX") ? atoll(getenv("MALI_FORK_MAX")) : 16384;
        const bool small = (int64_t)ncol * m->specTiles <= forkMax;
        const bool side1 = small && m->sideStream[0] && !m->spec1.empty() && (!m->spec2.empty());
        const bool side0 = small && m->sideStream[1] && !m->spec0.empty() && (!m->spec2.empty() || !m->spec1.empty());
        if (side1 || side0) CU(cudaEventRecord(m->forkEvent, st));
        cudaStream_t s1 = st, s0 = st;
        if (side1) {
            s1 = m->sideStream[0];
            CU(cudaStreamWaitEvent(s1, m->forkEvent, 0));
        }
        if (side0) {
            s0 = m->sideStream[1];
            CU(cudaStreamWaitEvent(s0, m->forkEvent, 0));
        }
        cudaError_t e = cudaSuccess;
        const bool fast = m->arith == MALI_ARITH_CONTRACTED;
        if (!m->spec2.empty())
            e = (fast ? mali_fs_launch_2_fast : mali_fs_launch_2)(cc, m->spec2.data(), (int)m->spec2.size(), ncol, smem[2], st,
                                                                  &m->launches);
        if (e == cudaSuccess && !m->spec1.empty())
            e = (fast ? mali_fs_launch_1_fast : mali_fs_launch_1)(cc, m->spec1.data(), (int)m->spec1.size(), ncol, smem[1], s1,
                                                                  &m->launches);
        if (e == cudaSuccess && !m->spec0.empty())
            e = (fast ? mali_fs_launch_0_fast : mali_fs_launch_0)(cc, m->spec0.data(), (int)m->spec0.size(), ncol, smem[0], s0,
                                                                  &m->launches);
        if (e != cudaSuccess) return fail((int)e, "fs_gamma_kernel_m: %s", cudaGetErrorString(e));
        if (side1) {   // join
            CU(cudaEventRecord(m->joinEvent[0], s1));
            CU(cudaStreamWaitEvent(st, m->joinEvent[0], 0));
        }
        if (side0) {
            CU(cudaEventRecord(m->joinEvent[1], s0));
            CU(cudaStreamWaitEvent(st, m->joinEvent[1], 0));
        }
    }
    if (rec) {
        cudaEventRecord(m->profEvents[m->profUsed + 1], st);
        m->profUsed += 2;
    }
    FinishParams f = make_finish_params(m, b, col0, ncol);
    dim3 grid((m->N + 31) / 32, m->Natom, ncol);
    cudaStream_t sj = st;
    if (jJoin) {
        *jJoin = false;
        if (ctl.on && m->sideStream[0]) {
            sj = m->sideStream[0];
            CU(cudaEventRecord(m->forkEvent, st));
            CU(cudaStreamWaitEvent(sj, m->forkEvent, 0));
            *jJoin = true;
        }
    }
    gamma_finish_kernel<<<grid, dim3(32, 8), 0, st>>>(f);
    {
        const int nb = std::min(m->N, 41);   // depth rows are dealt round-robin to the blocks of a column
        j_finish_kernel<<<dim3(nb, ncol), 256, 0, sj>>>(b->J, m->lay.J, b->scratch, m->lay.scratch, m->off_jpart, m->upOff, b->colconst, m->lay.colconst, m->off_tab, m->d_tileJ, m->Nspect, m->Lw,
                                                      reinterpret_cast<unsigned long long *>(b->dJ), b->done, col0);
        if (sj != st) CU(cudaEventRecord(m->joinEvent[0], sj));
    }
    m->launches += 2;
    CU(cudaGetLastError());
    return MALI_OK;
}

static int64_t ng_doubles_per_column(const mali_model *m, int order)
{
    // order + 2 ring slots and the start snapshot, each [sumNlevel][Nspace], then one dPops bit pattern per atom
    return (int64_t)(order + 3) * m->lay.pops + m->Natom;
}

// ng != null: the statistical equilibrium also counts the solve (nse), snapshots n and pushes the solution into the
// ring, and the Ng stage follows it (ng_kernel, ng_dpops_kernel).  Without ng the launches are those of before.
static int launch_se(const mali_model *m, const mali_buffers *b, int col0, int ncol, int32_t *iter, int iterMin,
                     cudaStream_t st, const mali_ng_buffers *ng = nullptr, const mali_ng_params *ngp = nullptr)
{
    FinishParams f = make_finish_params(m, b, col0, ncol);
    // inside mali_iterate, columns whose own iteration counter is still <= 3 only iterate J (test.py:27)
    f.iter = iter;
    f.iterMin = iterMin;
    if (ng) {
        f.ngHist = ng->hist;
        f.ngNse = ng->nse;
        f.ngStride = ng_doubles_per_column(m, ngp->order);
        f.ngRing = ngp->order + 2;
    }
    se_prepare_kernel<<<(ncol + 127) / 128, 128, 0, st>>>(f.dPopsBits, b->done, iter, iterMin, iter != nullptr, col0, ncol,
                                                          ng ? ng->nse : nullptr);
    dim3 grid((m->N + 63) / 64, m->Natom, ncol);
    if (m->maxNlevel <= 8)
        stat_equil_kernel<8><<<grid, 64, 0, st>>>(f);
    else
        stat_equil_kernel<16><<<grid, 64, 0, st>>>(f);
    m->launches += 2;
    if (ng) {
        NgParams q{};
        q.N = m->N;
        q.Natom = m->Natom;
        q.col0 = col0;
        q.order = ngp->order;
        q.delay = ngp->delay;
        q.period = ngp->period;
        q.ring = ngp->order + 2;
        q.iterMin = iterMin;
        q.popStride = m->lay.pops;
        q.histStride = f.ngStride;
        q.Nlevel = m->d_Nlevel;
        q.lvlOff = m->d_lvlOff;
        q.pops = b->pops;
        q.hist = ng->hist;
        q.nse = ng->nse;
        q.accepted = ng->accepted;
        q.dPops = b->dPops;
        q.status = b->status;
        q.done = b->done;
        q.iter = iter;
        dim3 g(m->Natom, ncol);
        if (q.order == 1)
            ng_kernel<1><<<g, kNgThreads, 0, st>>>(q);
        else if (q.order == 2)
            ng_kernel<2><<<g, kNgThreads, 0, st>>>(q);
        else
            ng_kernel<3><<<g, kNgThreads, 0, st>>>(q);
        ng_dpops_kernel<<<(ncol + 127) / 128, 128, 0, st>>>(q, ncol);
        m->launches += 2;
    }
    CU(cudaGetLastError());
    return MALI_OK;
}

static int check_ng(const mali_ng_buffers *ng, const mali_ng_params *p, const char *who)
{
    if (!ng || !p || !ng->hist || !ng->nse || !ng->accepted) return fail(MALI_EINVAL, "%s: null Ng buffer or parameters", who);
    if (p->order < 1 || p->order > 3 || p->delay < 0 || p->period < 1)
        return fail(MALI_EINVAL, "%s: Ng order=%d delay=%d period=%d (need 1 <= order <= 3, delay >= 0, period >= 1)", who,
                    p->order, p->delay, p->period);
    return MALI_OK;
}

int mali_formal_sol_gamma(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, void *stream)
{
    if (int r = check_range(m, b, col0, ncol, "mali_formal_sol_gamma")) return r;
    if (!b->colconst || !b->pops || !b->J || !b->I || !b->Gamma || !b->scratch || !b->dJ)
        return fail(MALI_EINVAL, "mali_formal_sol_gamma: null buffer");
    // the done mask belongs to mali_iterate: a per-call formal solution always recomputes, like the reference
    mali_buffers bb = *b;
    bb.done = nullptr;
    bb.iter = nullptr;
    return launch_fs(m, &bb, col0, ncol, (cudaStream_t)stream, IterCtl{}, nullptr);
}

int mali_stat_equil(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, void *stream)
{
    if (int r = check_range(m, b, col0, ncol, "mali_stat_equil")) return r;
    if (!b->colconst || !b->pops || !b->Gamma || !b->dPops || !b->status)
        return fail(MALI_EINVAL, "mali_stat_equil: null buffer");
    mali_buffers bb = *b;
    bb.done = nullptr;
    bb.iter = nullptr;
    return launch_se(m, &bb, col0, ncol, nullptr, 0, (cudaStream_t)stream);
}

int mali_ng_layout(const mali_model *m, int32_t order, int64_t *doubles_per_column)
{
    if (!m || !doubles_per_column || order < 1 || order > 3) return fail(MALI_EINVAL, "mali_ng_layout: bad argument (order %d)", order);
    *doubles_per_column = ng_doubles_per_column(m, order);
    return MALI_OK;
}

int mali_stat_equil_ng(const mali_model *m, const mali_buffers *b, const mali_ng_buffers *ng, const mali_ng_params *p,
                       int32_t col0, int32_t ncol, void *stream)
{
    if (int r = check_range(m, b, col0, ncol, "mali_stat_equil_ng")) return r;
    if (int r = check_ng(ng, p, "mali_stat_equil_ng")) return r;
    if (!b->colconst || !b->pops || !b->Gamma || !b->dPops || !b->status)
        return fail(MALI_EINVAL, "mali_stat_equil_ng: null buffer");
    mali_buffers bb = *b;
    bb.done = nullptr;
    bb.iter = nullptr;
    return launch_se(m, &bb, col0, ncol, nullptr, 0, (cudaStream_t)stream, ng, p);
}

static int iterate_impl(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, int32_t max_iter,
                        double tolJ, double tolPops, void *stream, const mali_ng_buffers *ng, const mali_ng_params *ngp);

int mali_iterate(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, int32_t max_iter, double tolJ,
                 double tolPops, void *stream)
{
    return iterate_impl(m, b, col0, ncol, max_iter, tolJ, tolPops, stream, nullptr, nullptr);
}

int mali_iterate_ng(const mali_model *m, const mali_buffers *b, const mali_ng_buffers *ng, const mali_ng_params *p,
                    int32_t col0, int32_t ncol, int32_t max_iter, double tolJ, double tolPops, void *stream)
{
    if (int r = check_range(m, b, col0, ncol, "mali_iterate_ng")) return r;
    if (int r = check_ng(ng, p, "mali_iterate_ng")) return r;
    return iterate_impl(m, b, col0, ncol, max_iter, tolJ, tolPops, stream, ng, p);
}

// mali_iterate, and with ng: the Ng stage after every statistical equilibrium, inside the same captured graph
static int iterate_impl(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, int32_t max_iter,
                        double tolJ, double tolPops, void *stream, const mali_ng_buffers *ng, const mali_ng_params *ngp)
{
    if (int r = check_range(m, b, col0, ncol, "mali_iterate")) return r;
    if (!b->colconst || !b->pops || !b->J || !b->I || !b->Gamma || !b->scratch || !b->dJ || !b->dPops || !b->status ||
        !b->iter || !b->done)
        return fail(MALI_EINVAL, "mali_iterate: null buffer");
    cudaStream_t caller = (cudaStream_t)stream;
    if (max_iter < 1) return MALI_OK;
    // The legacy default stream cannot be captured into a graph: when the caller works on it (PyTorch's default), the
    // loop runs on a library-owned stream that is forked from and joined back into the caller's stream with events,
    // so the call stays stream-ordered.
    cudaStream_t st = caller;
    const bool detour = (caller == nullptr || caller == cudaStreamLegacy) && m->iterStream != nullptr;
    if (detour) {
        st = m->iterStream;
        CU(cudaEventRecord(m->iterFork, caller));
        CU(cudaStreamWaitEvent(st, m->iterFork, 0));
    }
    IterCtl ctl{};
    ctl.on = 1;
    ctl.tolJ = tolJ;
    ctl.tolPops = tolPops;
    ctl.iter = b->iter;
    ctl.doneW = b->done;
    ctl.status = b->status;
    ctl.dPops = b->dPops;
    // one iteration of test.py:20-29: formal solution + Gamma, then (J finish on a side stream) || (statistical equilibrium)
    auto one_iteration = [&]() -> int {
        bool jJoin = false;
        if (int r = launch_fs(m, b, col0, ncol, st, ctl, &jJoin)) return r;
        if (int r = launch_se(m, b, col0, ncol, b->iter, 4, st, ng, ngp)) return r;
        if (jJoin) CU(cudaStreamWaitEvent(st, m->joinEvent[0], 0));
        return MALI_OK;
    };
    // The iteration is captured ONCE into a CUDA graph and replayed: a column batch of a response function or a single
    // column is bound by launch gaps, not by arithmetic (a CaII/FALC iteration is ~10 short kernels).  The graph is
    // cached per (buffers, column range, tolerances, arithmetic mode).  Profiling and MALI_NO_GRAPH=1 use plain launches.
    static const bool noGraph = getenv("MALI_NO_GRAPH") != nullptr;
    bool done_by_graph = false;
    if (!noGraph && !m->profOn && max_iter >= 2) {
        IterGraphKey key;
        memset(&key, 0, sizeof key);     // the key is compared bytewise: no indeterminate padding
        key.b.ncol = b->ncol;
        key.b.colconst = b->colconst;
        key.b.pops = b->pops;
        key.b.J = b->J;
        key.b.I = b->I;
        key.b.Gamma = b->Gamma;
        key.b.scratch = b->scratch;
        key.b.dJ = b->dJ;
        key.b.dPops = b->dPops;
        key.b.status = b->status;
        key.b.iter = b->iter;
        key.b.done = b->done;
        key.col0 = col0;
        key.ncol = ncol;
        key.tolJ = tolJ;
        key.tolPops = tolPops;
        key.arith = m->arith;
        if (ng) {
            key.ng.hist = ng->hist;
            key.ng.nse = ng->nse;
            key.ng.accepted = ng->accepted;
            key.ngp.order = ngp->order;
            key.ngp.delay = ngp->delay;
            key.ngp.period = ngp->period;
        }
        cudaGraphExec_t exec = nullptr;
        for (auto &g : m->iterGraphs)
            if (memcmp(&g.key, &key, sizeof key) == 0) exec = g.exec;
        if (!exec) {
            const long long l0 = m->launches;
            cudaGraph_t graph = nullptr;
            if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                const int r = one_iteration();
                const cudaError_t e = cudaStreamEndCapture(st, &graph);
                if (r == MALI_OK && e == cudaSuccess && graph && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) {
                    if (m->iterGraphs.size() >= 8) {     // small cache: drop the oldest
                        cudaGraphExecDestroy(m->iterGraphs.front().exec);
                        m->iterGraphs.erase(m->iterGraphs.begin());
                    }
                    m->iterGraphs.push_back(IterGraph{key, exec, m->launches - l0});
                } else {
                    exec = nullptr;
                }
                if (graph) cudaGraphDestroy(graph);
            }
            cudaGetLastError();      // a failed capture falls back to plain launches below
            m->launches = l0;
        }
        if (exec) {
            long long per = 0;
            for (auto &g : m->iterGraphs)
                if (g.exec == exec) per = g.kernels;
            for (int it = 0; it < max_iter; ++it) CU(cudaGraphLaunch(exec, st));
            m->launches += per * max_iter;
            m->graphLaunches += max_iter;
            done_by_graph = true;
        }
    }
    if (!done_by_graph)
        for (int it = 0; it < max_iter; ++it)
            if (int r = one_iteration()) return r;
    iterate_close_kernel<<<(ncol + 127) / 128, 128, 0, st>>>(b->dJ, ctl, col0, ncol);
    m->launches += 1;
    if (detour) {
        CU(cudaEventRecord(m->iterJoin, st));
        CU(cudaStreamWaitEvent(caller, m->iterJoin, 0));
    }
    CU(cudaGetLastError());
    return MALI_OK;
}

int mali_piecewise_linear_1d(int32_t Nspace, int32_t nray, const double *z, const double *muz, const int32_t *toFrom,
                             const double *bbc0, const double *bbc1, const double *chi, const double *S, double *I,
                             double *Psi, void *stream)
{
    if (Nspace < 3) return fail(MALI_ELIMIT, "Nspace=%d: need >= 3 depth points", Nspace);
    if (nray < 1 || !z || !muz || !toFrom || !bbc0 || !bbc1 || !chi || !S || !I || !Psi)
        return fail(MALI_EINVAL, "mali_piecewise_linear_1d: bad argument");
    sweep_hook_kernel<<<(nray + 63) / 64, 64, 0, (cudaStream_t)stream>>>(Nspace, nray, z, muz, toFrom, bbc0, bbc1, chi, S,
                                                                         I, Psi);
    CU(cudaGetLastError());
    return MALI_OK;
}

int mali_profile_begin(const mali_model *m, int32_t max_launches)
{
    if (!m || max_launches < 1) return fail(MALI_EINVAL, "mali_profile_begin: bad argument");
    CU(cudaSetDevice(m->device));
    while ((int)m->profEvents.size() < 2 * max_launches) {
        cudaEvent_t e;
        CU(cudaEventCreate(&e));
        m->profEvents.push_back(e);
    }
    m->profUsed = 0;
    m->profOn = true;
    return MALI_OK;
}

int mali_profile_end(const mali_model *m, double *fs_ms_total, int32_t *fs_launches)
{
    if (!m || !fs_ms_total || !fs_launches) return fail(MALI_EINVAL, "mali_profile_end: bad argument");
    m->profOn = false;
    double tot = 0.0;
    for (int q = 0; q + 1 < m->profUsed; q += 2) {
        CU(cudaEventSynchronize(m->profEvents[q + 1]));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, m->profEvents[q], m->profEvents[q + 1]));
        tot += ms;
    }
    *fs_ms_total = tot;
    *fs_launches = m->profUsed / 2;
    m->profUsed = 0;
    return MALI_OK;
}

long long mali_launch_count(const mali_model *m) { return m ? m->launches : 0; }
long long mali_graph_iterations(const mali_model *m) { return m ? m->graphLaunches : 0; }

int mali_line_layout(const mali_model *m, int32_t t, int32_t *tile0, int32_t *ntile, int32_t *entries, int32_t cap,
                     int64_t *off_tab)
{
    if (!m || !tile0 || !ntile || !off_tab || t < 0 || t >= m->Ntrans) return fail(MALI_EINVAL, "mali_line_layout: bad argument");
    const std::vector<PhiTile> &v = m->phiTilesHost[t];
    *tile0 = m->phiTile0Host[t];
    *ntile = (int32_t)v.size();
    *off_tab = m->off_tab;
    if (entries) {
        if (cap < (int32_t)v.size()) return fail(MALI_EINVAL, "mali_line_layout: room for %d tiles, the line spans %zu", cap, v.size());
        for (size_t q = 0; q < v.size(); ++q) {
            entries[4 * q + 0] = v[q].v0;
            entries[4 * q + 1] = v[q].vDir;
            entries[4 * q + 2] = v[q].f;
            entries[4 * q + 3] = v[q].stride;
        }
    }
    return MALI_OK;
}

int mali_div_hook(int32_t n, const double *a_dev, const double *b_dev, double *q_dev, int32_t *bad_dev, void *stream)
{
    if (n < 1 || !a_dev || !b_dev || !q_dev || !bad_dev) return fail(MALI_EINVAL, "mali_div_hook: bad argument");
    div_hook_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(n, a_dev, b_dev, q_dev, bad_dev);
    CU(cudaGetLastError());
    return MALI_OK;
}

int mali_fp64_peak(int32_t iters, double *scratch_dev, double *ops_per_second)
{
    if (iters < 1 || !scratch_dev || !ops_per_second) return fail(MALI_EINVAL, "mali_fp64_peak: bad argument");
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    int dev = 0, sms = 148;
    CU(cudaGetDevice(&dev));
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int blocks = sms * 8, threads = 256;
    fp64_peak_kernel<<<blocks, threads>>>(iters / 8 + 1, 1.0, scratch_dev);  // warm-up
    CU(cudaEventRecord(e0));
    fp64_peak_kernel<<<blocks, threads>>>(iters, 1.0, scratch_dev);
    CU(cudaEventRecord(e1));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    CU(cudaEventDestroy(e0));
    CU(cudaEventDestroy(e1));
    *ops_per_second = (double)blocks * threads * (double)iters * 16.0 / (ms * 1e-3);  // 8 chains x (mul + add)
    return MALI_OK;
}

int mali_ng_hook(int32_t order, int64_t nvec, const double *hist_dev, double *out_dev, int32_t *accepted_dev, void *stream)
{
    if (order < 1 || order > 3 || nvec < 1 || !hist_dev || !out_dev || !accepted_dev)
        return fail(MALI_EINVAL, "mali_ng_hook: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (order == 1)
        ng_hook_kernel<1><<<1, kNgThreads, 0, st>>>(nvec, hist_dev, out_dev, accepted_dev);
    else if (order == 2)
        ng_hook_kernel<2><<<1, kNgThreads, 0, st>>>(nvec, hist_dev, out_dev, accepted_dev);
    else
        ng_hook_kernel<3><<<1, kNgThreads, 0, st>>>(nvec, hist_dev, out_dev, accepted_dev);
    CU(cudaGetLastError());
    return MALI_OK;
}

int mali_exp_hook(int32_t n, const double *x_dev, double *y_dev, void *stream)
{
    if (n < 1 || !x_dev || !y_dev) return fail(MALI_EINVAL, "mali_exp_hook: bad argument");
    exp_hook_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(n, x_dev, y_dev);
    CU(cudaGetLastError());
    return MALI_OK;
}

int mali_uv(const mali_model *m, const mali_buffers *b, int32_t col, int32_t t, int32_t la, int32_t mu, int32_t toFrom,
            double *Uji, double *Vij, double *Vji, void *stream)
{
    if (int r = check_range(m, b, col, 1, "mali_uv")) return r;
    if (t < 0 || t >= m->Ntrans || mu < 0 || mu >= m->Nrays || !Uji || !Vij || !Vji)
        return fail(MALI_EINVAL, "mali_uv: bad argument");
    const SlotDesc &ts = m->transSlot[t];
    if (la < ts.Nblue || la >= ts.Nblue + ts.Nlam) return fail(MALI_EINVAL, "mali_uv: transition %d is not active at wavelength %d", t, la);
    const int ti = la / m->Lw;
    const TileDesc &td = m->tiles[ti];
    const SlotDesc *sd = nullptr;
    for (int q = 0; q < td.nslot; ++q)
        if (m->slots[td.slot0 + q].t == t) sd = &m->slots[td.slot0 + q];
    if (!sd) return fail(MALI_EINVAL, "mali_uv: internal error, transition %d missing from tile %d", t, ti);
    FsParams p = make_fs_params(m, b, col, 1, 1);
    uv_hook_kernel<<<(m->N + 63) / 64, 64, 0, (cudaStream_t)stream>>>(p, col, *sd, td.recOff, td.stride, td.vDir, la, la - td.la0,
                                                                      mu, toFrom ? 1 : 0, Uji, Vij, Vji);
    CU(cudaGetLastError());
    return MALI_OK;
}

}  // extern "C"
