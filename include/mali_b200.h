/*
 * mali_b200.h -- C ABI of the B200-native MALI hot path (libmali_b200.so).
 *
 * The Lightspinner reference is pure Python and has no FFI layer (SURVEY.md 8b); the boundary it offers is
 * the Python API of rh_method.Context.  Every entry point below is therefore the C-level twin of one
 * reference method, and lightspinner_b200/context.py binds them with ctypes behind the reference's own
 * call signatures (INTEGRATION.md shows the stub a maintainer would add to the reference).
 *
 *   reference (file:line)                                   entry point
 *   ------------------------------------------------------  ---------------------------------
 *   Context.__init__            rh_method.py:531-563        mali_model_create, mali_upload_columns
 *   ComputationalAtom.setup_wavelength  rh_method.py:425-455 (tables built once by mali_upload_columns)
 *   Context.formal_sol_gamma_matrices   rh_method.py:565-708 mali_formal_sol_gamma
 *   ComputationalTransition.uv  rh_method.py:245-288        (fused into mali_formal_sol_gamma); mali_uv = test hook
 *   piecewise_linear_1d         formal_solver.py:144-212    (fused into mali_formal_sol_gamma); mali_piecewise_linear_1d = test hook
 *   planck                      utils.py:17-22              mali_planck_bc (host helper for the lower boundary)
 *   Context.stat_equil          rh_method.py:710-745        mali_stat_equil
 *   test.py:20-29 / response_fn.py:11-21 (the MALI loop)    mali_iterate (device-resident loop, per-column convergence)
 *   (no reference counterpart: opt-in Ng acceleration)      mali_stat_equil_ng, mali_iterate_ng; mali_ng_hook = test hook
 *   lte_pops atomic_set.py:105-145, compute_collisions rh_method.py:474-487, v_broad atomic_model.py:241-245,
 *   continuum g_ij rh_method.py:453-454                     mali_model_set_atoms + mali_setup_columns (device-side set-up)
 *   Background.compute_background_eos background.py:21-53 (witt.py EOS + cop), AtmosphereConstructor.convert_scales
 *   atmosphere.py:70-112 (column mass)                      mali_model_set_eos + mali_background
 *   ComputationalTransition.compute_phi rh_method.py:198-243 mali_compute_phi (device Voigt profiles); mali_line_layout = read-back
 *   (no reference counterpart; Lightweaver's compute_rays) mali_compute_rays (emergent intensity at user angles)
 *
 * Conventions
 *   - plain C, no exceptions; every function returns 0 on success, a negative MALI_E* code on argument
 *     errors, or a positive cudaError_t; mali_last_error() gives the message for the calling thread.
 *   - all `*_dev` / mali_buffers pointers are DEVICE pointers owned by the caller (the Python layer carries
 *     them in torch tensors); the library owns only the model descriptors it uploads in mali_model_create.
 *   - everything is IEEE fp64; the kernels are compiled with --fmad=false and evaluate every expression in
 *     the reference's order (SURVEY.md appendix A).
 *   - all launches are asynchronous on the given stream (a cudaStream_t passed as void*).
 *   - column batches: every per-column array is [ncol][...]; a launch works on columns [col0, col0+ncol).
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef MALI_B200_H
#define MALI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MALI_OK 0
#define MALI_EINVAL (-1)   /* bad argument */
#define MALI_ENOMEM (-2)
#define MALI_ELIMIT (-3)   /* problem exceeds a compiled-in limit (Nrays > 32, Nlevel > 16, Nspace < 3, ...) */

#define MALI_TRANS_STRIDE 6 /* atom, i, j, isLine, Nblue, Nlambda */

typedef struct mali_model mali_model; /* opaque */

/* Host-side description of the radiative model shared by all columns of a batch.
 * trans rows are in the reference's order: atoms as in Context.activeAtoms, within an atom lines then
 * continua (rh_method.py:398-405).  A transition is active on wavelengths [Nblue, Nblue+Nlambda).
 * The per-wavelength tables are concatenated over transitions (offset = running sum of Nlambda). */
typedef struct {
    int32_t Nspace, Nrays, Nspect, Natom, Ntrans;
    const int32_t *Nlevel;     /* [Natom] */
    const int32_t *trans;      /* [Ntrans][MALI_TRANS_STRIDE] */
    const double *wavelength;  /* [Nspect] nm */
    const double *muz, *wmu;   /* [Nrays] */
    const double *lineconst;   /* [Ntrans][3]: hc/4pi*Bij, Aji/Bji, Bji/Bij (lines) */
    const double *wlambda;     /* concat: rh_method.py:157-196 */
    const double *alpha;       /* concat: continuum cross-sections */
    const double *twohc_l3;    /* concat: 2hc/(NM_TO_M lambda)^3 (continua) */
    const double *wlacont;     /* concat: wlambda/lambda/h (continua) */
    const double *lambda0;     /* [Ntrans] line-centre wavelength in nm (lines; read by mali_compute_phi / _rays), may be NULL */
} mali_model_desc;

/* Sizes (in doubles, per column) of every caller-owned array, and the offsets of the reference-layout
 * arrays inside one column's host staging block ("host pack": plain concatenation, no transposition). */
typedef struct {
    int64_t hostpack;  /* staging block: what mali_upload_columns copies host->device */
    int64_t colconst;  /* packed per-column device block: z, planck BC, C, nTotal, then the tile-major table
                          [Nspace][tile records] (see csrc/mali_types.cuh).  Written by mali_upload_columns; the only
                          part that changes afterwards is the J-dagger field of the records, which
                          mali_formal_sol_gamma rewrites (it is the copy of J the next formal solution reads) */
    int64_t pops;      /* sumNlevel * Nspace        n[level][k]            (in/out) */
    int64_t J;         /* Nspace * Nspect           J[k][la]  (depth-major) (out; zeroed by upload) */
    int64_t I;         /* Nspect * Nrays            I[la][mu]               (out) */
    int64_t Gamma;     /* sum Nlevel^2 * Nspace     Gamma[i][j][k] per atom (out) */
    int64_t scratch;   /* library scratch per column */
    /* offsets inside the host pack (reference layouts): */
    int64_t hp_height;   /* [Nspace] */
    int64_t hp_bbc;      /* [Nspect][2]  planck(T[-2:], wav)  (formal_solver.py:206) */
    int64_t hp_bg_chi, hp_bg_eta, hp_bg_sca; /* [Nspect][Nspace] */
    int64_t hp_C;        /* concat atoms [Nlevel][Nlevel][Nspace] */
    int64_t hp_nTotal;   /* [Natom][Nspace] (stored before hp_bg_chi: see mali_upload_columns_atmos / _thermo) */
    int64_t hp_gijcont;  /* concat [offset+lt][Nspace], continua rows only (rh_method.py:453-454) */
    int64_t hp_n;        /* [sumNlevel][Nspace] starting populations */
    /* the line profiles come last, so that a caller who lets the device compute them (mali_compute_phi) uploads
     * only the first hp_phi doubles of every block (mali_upload_columns_nophi): */
    int64_t hp_phi;      /* concat lines, each [Nlambda][Nrays][2][Nspace] (rh_method.py:224) */
    int64_t hp_wphi;     /* [Ntrans][Nspace] */
    int32_t sumNlevel, sumNlevel2, ntile, lambda_per_warp;
} mali_layout;

/* Caller-owned device buffers for a batch of `ncol` columns. */
typedef struct {
    int32_t ncol;
    double *colconst;  /* [ncol][layout.colconst] */
    double *pops;      /* [ncol][layout.pops]     */
    double *J;         /* [ncol][layout.J]        */
    double *I;         /* [ncol][layout.I]        */
    double *Gamma;     /* [ncol][layout.Gamma]    */
    double *scratch;   /* [ncol][layout.scratch]  */
    double *dJ;        /* [ncol] max |1 - Jold/Jnew| of the last formal solution (NaN-propagating) */
    double *dPops;     /* [ncol] max |1 - nold/nnew| of the last stat_equil */
    int32_t *status;   /* [ncol] bit 0: a singular / non-finite statistical-equilibrium system was met;
                          bit 1: an opacity / optical-depth step left [2^-1000, 2^1000] (formal solution invalid) */
    int32_t *iter;     /* [ncol] iterations done by mali_iterate */
    int32_t *done;     /* [ncol] mali_iterate only: 1 = converged, 2 = stopped on a fault (status != 0 or NaN); such
                          columns are skipped by the remaining iterations.  The per-call entry points
                          (mali_formal_sol_gamma, mali_stat_equil) ignore it and always recompute, like the reference */
} mali_buffers;

const char *mali_last_error(void);
int mali_device_count(void);

int mali_model_create(const mali_model_desc *desc, int device, mali_model **out);
void mali_model_destroy(mali_model *m);
/* Arithmetic mode of the structure-specialised formal-solution kernels (csrc/mali_device.cuh, Arith):
 *   MALI_ARITH_EXACT       every operation separately rounded in the reference's evaluation order: one ray's chi, S, I,
 *                          PsiStar and Gamma integrands are bit-identical to the reference's numpy / numba arithmetic;
 *   MALI_ARITH_CONTRACTED  the same expressions with a*b+c fused and quotients by a shared divisor taken as
 *                          a * (1/b): fp64 throughout, every intermediate within ~2 ulp of the exact mode's, about a
 *                          quarter fewer fp64 instructions.
 * Both meet the parity bar (populations, J, I within 1e-10 of the reference after the same number of iterations;
 * identical iteration counts) and both are tested against it.  A new model starts in MALI_ARITH_DEFAULT unless the
 * environment variable MALI_ARITH=exact|contracted says otherwise.  The generic kernel (tiles without a specialised
 * instance), the test hooks and the statistical-equilibrium solve always use the exact form. */
#define MALI_ARITH_EXACT 0
#define MALI_ARITH_CONTRACTED 1
#define MALI_ARITH_DEFAULT MALI_ARITH_CONTRACTED
int mali_model_set_arith(mali_model *m, int32_t mode);
int mali_model_get_arith(const mali_model *m);

int mali_model_layout(const mali_model *m, mali_layout *out);
/* out8: ntile, tiles on structure-specialised kernels, tiles on the generic kernel, max transitions per tile,
 * max levels per tile, doubles per depth row of the tile-major table, shared-memory bytes per warp, TMA staging on/off */
int mali_model_info(const mali_model *m, int32_t *out8);

/* Host helper: out[la][0..1] = planck(T[Nspace-2]), planck(T[Nspace-1]) at wavelength[la]  (utils.py:17-22, glibc exp). */
int mali_planck_bc(const double *wavelength, int32_t Nspect, double Tm2, double Tm1, double *out);

/* Copies ncol host-pack blocks host->device (cudaMemcpyAsync; pin the host memory) into staging_dev
 * ([ncol][layout.hostpack] doubles) and packs them into bufs->colconst / pops for columns [col0, col0+ncol).
 * host_pack may be NULL when staging_dev already holds the blocks.  Also zeroes J for those columns. */
int mali_upload_columns(const mali_model *m, const mali_buffers *bufs, int32_t col0, int32_t ncol,
                        const double *host_pack, double *staging_dev, void *stream);

/* Same, for callers that do not hold the line profiles: host_pack_prefix holds [ncol][layout.hp_phi] doubles (the
 * blocks without their phi / wphi tail; may be NULL when staging_dev already holds them at stride layout.hostpack).
 * The profile entries of the device tables are zeroed; call mali_compute_phi before the first formal solution. */
int mali_upload_columns_nophi(const mali_model *m, const mali_buffers *bufs, int32_t col0, int32_t ncol,
                              const double *host_pack_prefix, double *staging_dev, void *stream);

/* Same again, for callers that let the device form everything it can from the atmosphere: host_pack_prefix holds
 * [ncol][layout.hp_C] doubles (heights, boundary Planck values, background chi / eta / sca, nTotal); call
 * mali_setup_columns and mali_compute_phi before the first formal solution. */
int mali_upload_columns_atmos(const mali_model *m, const mali_buffers *bufs, int32_t col0, int32_t ncol,
                              const double *host_pack_prefix, double *staging_dev, void *stream);

/* And for callers that hand over the thermodynamic state only: host_pack_prefix holds [ncol][layout.hp_bg_chi] doubles
 * (heights -- overwritten by mali_background when it is given a column-mass scale --, boundary Planck values, nTotal);
 * call mali_background, mali_setup_columns and mali_compute_phi before the first formal solution. */
int mali_upload_columns_thermo(const mali_model *m, const mali_buffers *bufs, int32_t col0, int32_t ncol,
                               const double *host_pack_prefix, double *staging_dev, void *stream);

/* State of the reference's EOS object (witt.witt(), witt.py:152-195) and the constants around it, for the device-side
 * Background.compute_background_eos (background.py:21-53) and AtmosphereConstructor.convert_scales (atmosphere.py:70-112,
 * column-mass branch). */
typedef struct {
    int32_t npf;               /* temperatures of the partition-function tables */
    const double *tpf;         /* [npf] */
    const double *pf;          /* [stage_off[28]][npf]: first 28 elements, every ionisation stage */
    const double *eion;        /* [stage_off[28]] ionisation energies in eV */
    const int32_t *stage_off;  /* [29] running sum of the elements' stage counts */
    const double *abund;       /* [99] abundances as the instance holds them (normalised) */
    double avw, rho_from_H, ab_others;   /* witt.py:172-181 */
    double saha_fac;           /* witt.py:52 */
    double prec;               /* witt.py:155 */
    double amu_weight_per_H;   /* Const.Amu * atomicTable.weightPerH   (background.py:33) */
    double cm_to_m_cubed;      /* Const.CM_TO_M**3 as Python evaluates it */
    double thomson_sigma;      /* background.py:11 */
} mali_eos_desc;
int mali_model_set_eos(mali_model *m, const mali_eos_desc *eos);

/* Background.compute_background_eos for columns [col0, col0+ncol): gas / electron pressure from (T, nHTot) through the
 * Wittmann EOS, background opacity chi, emissivity eta = B_nu(T) chi and Thomson scattering on the model's wavelength
 * grid, written into the bg fields of the tile records.  T, ne, nHTot: [ncol][Nspace] device, SI units as
 * Atmosphere holds them after nondimensionalise().  cmass != NULL ([ncol][Nspace], kg m^-2): also the heights of
 * convert_scales' column-mass branch (tau_500 = 1 at height 0) into colconst.  work: device scratch of
 * ncol * Nspace * 21 doubles. */
int mali_background(const mali_model *m, const mali_buffers *bufs, int32_t col0, int32_t ncol, const double *T_dev,
                    const double *ne_dev, const double *nHTot_dev, const double *cmass_dev, double *work_dev, void *stream);

/* Model-level data of the active atoms for the device-side column set-up (mali_setup_columns): what lte_pops
 * (atomic_set.py:105-145), the collisional-rate terms (collisional_rates.py:36-96) and v_broad (atomic_model.py:241-245)
 * read from the atomic-model objects.  Level arrays are concatenated over the atoms in the model's order. */
typedef struct {
    int32_t Natom;
    const int32_t *Nlevel;   /* [Natom], must equal the model's */
    const double *dE;        /* E_SI[l] - E_SI[0]                                  (atomic_set.py:131) */
    const double *gi0;       /* g[l] / g[0]                                        (:132) */
    const int32_t *dZ;       /* stage[l] - stage[0]                                (:133) */
    const double *nDebye;    /* Debye shift count of the level                     (:113-119) */
    const double *g;         /* statistical weights g[l] */
    const double *vTherm;    /* [Natom] 2 k / (amu * atomic weight)                (atomic_model.py:242) */
    double c1, c2;           /* atomic_set.py:107, :111 evaluated by the host */
    int32_t Ncoll;
    const int32_t *coll;     /* [Ncoll][8]: atom, kind (0 Omega, 1 CI, 2 CE), i, j (i < j), table points n, offset into
                                knots, offset into coef, cubic (1) or linear (0); the model's order (rates are added in
                                that order); offsets are running sums */
    const double *knots;     /* the interpolant of collisional_rates.py:15-19 (scipy interp1d) per collision: cubic: the
                                n + 4 knots of its not-a-knot B-spline; linear (2-point tables): the n temperatures */
    const double *coef;      /* cubic: the n B-spline coefficients; linear: the n rates */
    const double *fill;      /* [Ncoll][2]: values below / above the table (rates[0], rates[-1]) */
    const double *par;       /* [Ncoll]: Omega: C0 (collisional_rates.py:35); CI: E_SI[j] - E_SI[i]; CE: g[i] / g[j] */
} mali_atom_desc;
int mali_model_set_atoms(mali_model *m, const mali_atom_desc *atoms);

/* lte_pops + compute_collisions + v_broad + the continua's g_ij (rh_method.py:453-454) for columns [col0, col0+ncol),
 * from T, ne, vturb [ncol][Nspace] (device) and the nTotal the upload put into colconst: writes C and the g_ij fields
 * into colconst, nStar [ncol][sumNlevel][Nspace] and vBroad [ncol][Natom][Nspace] (device, caller-owned; vBroad is what
 * mali_compute_phi takes), and -- start_from_lte != 0 -- the populations n = nStar (rh_method.py:415). */
int mali_setup_columns(const mali_model *m, const mali_buffers *bufs, int32_t col0, int32_t ncol, const double *T_dev,
                       const double *ne_dev, const double *vturb_dev, double *nStar_dev, double *vBroad_dev,
                       int32_t start_from_lte, void *stream);

/* ComputationalTransition.compute_phi (rh_method.py:198-243) on the device, for columns [col0, col0+ncol): Voigt
 * profiles phi[la][mu][toFrom][k] = H(aDamp, v -+ mu vlos / vBroad) / (sqrt(pi) vBroad) of every line and their
 * normalisation wphi, written straight into the device tables (Vij rows and wavelength-weight fields).
 *   aDamp  [ncol][Ntrans][Nspace] device (rows of continua are not read; atomic_model.py:491-502)
 *   vBroad [ncol][Natom][Nspace]  device (atomic_model.py:241-245)      vlos [ncol][Nspace] device
 * Needs mali_model_desc.lambda0.  H comes from csrc/mali_voigt.h (a few ulp; scipy's wofz, which the reference
 * calls, is good to ~1e-13, so profiles agree with the reference's to that level, not bit for bit). */
int mali_compute_phi(const mali_model *m, const mali_buffers *bufs, int32_t col0, int32_t ncol, const double *aDamp,
                     const double *vBroad, const double *vlos, void *stream);

/* Emergent intensity at user angles from the current populations and J, for columns [col0, col0+ncol) (Lightweaver's
 * Context.compute_rays; the reference has no counterpart).  I_out[c][la][m] is what the NEXT mali_formal_sol_gamma would
 * return as I[la][mu] if mu[m] were one of the model's quadrature angles: opacity and emissivity from the current n, the
 * scattering term from the current J (zero after an upload), the line profiles of the up-going direction at mu[m]
 * (rh_method.py:223-231, the device Voigt function of mali_compute_phi), the thermalised lower boundary.  Always the
 * exact arithmetic form.  Writes nothing but I_out and bad: the call can sit between any two iterations.
 *   mu: HOST array [nmu], 0 < mu <= 1, 1 <= nmu <= MALI_RAYS_MAX_MU (carried in the kernel parameters)
 *   aDamp [ncol][Ntrans][Nspace], vBroad [ncol][Natom][Nspace], vlos [ncol][Nspace]: device, per call (the convention
 *   of mali_compute_phi; may be NULL for a model without lines).  Needs mali_model_desc.lambda0 when there are lines.
 *   I_out: device [ncol][Nspect][nmu].  bad: device [ncol] or NULL, bit 1 as in status (the caller zeroes it). */
#define MALI_RAYS_MAX_MU 64
int mali_compute_rays(const mali_model *m, const mali_buffers *b, int32_t col0, int32_t ncol, int32_t nmu,
                      const double *mu, const double *aDamp, const double *vBroad, const double *vlos,
                      double *I_out, int32_t *bad, void *stream);

/* Context.formal_sol_gamma_matrices for columns [col0, col0+ncol): updates J, I, Gamma and dJ.  J-dagger (the
 * previous call's J; zero after an upload, rh_method.py:541) is kept by the library inside colconst.  Work is
 * enqueued on `stream`; small launches also use two library-owned side streams, forked from and joined back into
 * `stream` with events, so the call is stream-ordered like any other. */
int mali_formal_sol_gamma(const mali_model *m, const mali_buffers *bufs, int32_t col0, int32_t ncol, void *stream);

/* Context.stat_equil for columns [col0, col0+ncol): updates pops in place, writes dPops and status. */
int mali_stat_equil(const mali_model *m, const mali_buffers *bufs, int32_t col0, int32_t ncol, void *stream);

/* The loop of test.py:20-29 kept on the device: up to max_iter iterations of formal solution (+ stat_equil once
 * a column's own iteration counter exceeds 3); a column whose (dJ, dPops) satisfy dJ <= tolJ && dPops <= tolPops
 * is flagged done and no longer touched.  tolJ < 0 disables the convergence test (fixed iteration count).
 * One iteration is captured into a CUDA graph (cached per buffers / range / tolerances / arithmetic mode) and replayed;
 * a caller on the legacy default stream is served on a library-owned stream forked from / joined into it with events.
 * All launches are asynchronous and ordered on `stream`; no host synchronisation happens inside.  bufs->iter / done must be
 * zeroed and bufs->dPops set to 1.0 by the caller first (dPops stays 1.0 until a column's first stat_equil). */
int mali_iterate(const mali_model *m, const mali_buffers *bufs, int32_t col0, int32_t ncol, int32_t max_iter,
                 double tolJ, double tolPops, void *stream);

/* Ng acceleration of the population iteration (Auer 1987), opt-in; the reference has no such option, so with it on the
 * iteration counts differ from the reference's.  Per column and active atom, the vector x = n[level][k] (flattened
 * over level, depth) is pushed into a ring of the last order + 2 solved vectors after every statistical-equilibrium
 * solve, and nse counts the column's solves since the caller last zeroed it.  When nse > delay, nse >= order + 2 and
 * (nse - delay) % period == 0, with x0 the newest vector, d_i = x_i - x_{i+1} (i = 0..order) and w = 1/x0^2:
 *     A_ij = sum w (d0 - d_{i+1})(d0 - d_{j+1}),  b_i = sum w d0 (d0 - d_{i+1}),  A c = b,
 *     x* = (1 - sum c) x0 + sum_i c_i x_{i+1},
 * accepted (replacing the populations and the newest ring entry) only if A is non-singular and every entry of x* is
 * finite and > 0.  dPops of such an iteration is max |1 - n_start / n_final| over the column's atoms (n_start: what the
 * solve started from).  1 <= order <= 3, delay >= 0, period >= 1 (else MALI_EINVAL); (2, 3, 3) is the measured default,
 * (2, 2, 2) did not converge on CaII+H/FALC (DESIGN.md section 4).  The sums over (level, depth) are fixed-order block
 * reductions: results do not depend on the batch or the column range. */
typedef struct { int32_t order, delay, period; } mali_ng_params;
typedef struct {
    double *hist;      /* [ncol][mali_ng_layout doubles]: order+2 ring slots + 1 start snapshot, each sumNlevel*Nspace,
                          then Natom doubles of library scratch */
    int32_t *nse;      /* [ncol] solves since reset (caller zeroes; zero it again after editing a column's populations) */
    int32_t *accepted; /* [ncol][Natom] extrapolations applied (caller zeroes) */
} mali_ng_buffers;
int mali_ng_layout(const mali_model *m, int32_t order, int64_t *doubles_per_column);
/* mali_stat_equil followed by the Ng stage for columns [col0, col0+ncol). */
int mali_stat_equil_ng(const mali_model *m, const mali_buffers *b, const mali_ng_buffers *ng, const mali_ng_params *p,
                       int32_t col0, int32_t ncol, void *stream);
/* mali_iterate with the Ng stage after every statistical equilibrium (same captured graph, cached per Ng buffers and
 * parameters as well).  With delay >= max_iter no extrapolation is due and the results are bit-identical to
 * mali_iterate's. */
int mali_iterate_ng(const mali_model *m, const mali_buffers *b, const mali_ng_buffers *ng, const mali_ng_params *p,
                    int32_t col0, int32_t ncol, int32_t max_iter, double tolJ, double tolPops, void *stream);

/* Measurement: between begin and end every fs_gamma_kernel launch made through this model is bracketed by CUDA
 * events on its stream; end() returns their summed device time and the launch count (bench.py's roofline).
 * mali_launch_count: kernels launched through this model since creation (bench.py's gpu_launches). */
int mali_profile_begin(const mali_model *m, int32_t max_launches);
int mali_profile_end(const mali_model *m, double *fs_ms_total, int32_t *fs_launches);
long long mali_launch_count(const mali_model *m);
/* iterations of mali_iterate that were replayed from a captured CUDA graph since the model was created */
long long mali_graph_iterations(const mali_model *m);

/* Where the profile of line t lives inside a column's device table (read-back of ComputationalTransition.phi / wphi,
 * rh_method.py:224,235): the line spans *ntile wavelength tiles starting at tile *tile0 (tile = lambda_per_warp
 * consecutive wavelengths); for the q-th of them entries[4q..4q+3] = {v0, vDir, f, stride}: at depth k the row of 32
 * doubles hc/4pi*Bij*phi[(lambda, mu) in lane order] of direction 0 starts at colconst + *off_tab + v0 + k*stride (direction
 * 1: + vDir), and the field wlambda*wphi/HC [lambda_per_warp] at colconst + *off_tab + f + k*stride.  entries may be NULL
 * (query *ntile first). */
int mali_line_layout(const mali_model *m, int32_t t, int32_t *tile0, int32_t *ntile, int32_t *entries, int32_t cap,
                     int64_t *off_tab);

/* fp64 CUDA-core peak probe: unfused mul + add operations per second on the current device (roofline denominator;
 * MEASURED_PEAKS.json has no fp64 entry). */
int mali_fp64_peak(int32_t iters, double *scratch_dev, double *ops_per_second);

/* Test hooks ---------------------------------------------------------------------------------------------- */
/* piecewise_linear_1d for nray independent rays: chi, S, I, Psi are [nray][Nspace]; muz, bbc0/bbc1 (planck at
 * T[-2], T[-1]) and toFrom are per ray; z is [Nspace] (shared). */
int mali_piecewise_linear_1d(int32_t Nspace, int32_t nray, const double *z_dev, const double *muz_dev,
                             const int32_t *toFrom_dev, const double *bbc0_dev, const double *bbc1_dev,
                             const double *chi_dev, const double *S_dev, double *I_dev, double *Psi_dev,
                             void *stream);
/* y[i] = exp(x[i]) with the kernel's own exp (valid for 2^-54 <= |x| < 512): must equal libm's exp bit for bit,
 * which is what numba calls in formal_solver.py:41. */
int mali_exp_hook(int32_t n, const double *x_dev, double *y_dev, void *stream);
/* q[i] = a[i] / b[i] with the kernels' shared-reciprocal division; bad[i] != 0 where (a, b) is outside its domain.
 * Must equal the IEEE quotient bit for bit inside the domain. */
int mali_div_hook(int32_t n, const double *a_dev, const double *b_dev, double *q_dev, int32_t *bad_dev, void *stream);
/* One Ng extrapolation of hist_dev [order+2][nvec] (newest first) with the kernel's own code: out_dev = x* if accepted,
 * else the newest vector; *accepted_dev = 1 / 0. */
int mali_ng_hook(int32_t order, int64_t nvec, const double *hist_dev, double *out_dev, int32_t *accepted_dev, void *stream);
/* ComputationalTransition.uv(la, mu, toFrom) for transition t of column col: writes Uji, Vij, Vji [Nspace]. */
int mali_uv(const mali_model *m, const mali_buffers *bufs, int32_t col, int32_t t, int32_t la, int32_t mu,
            int32_t toFrom, double *Uji_dev, double *Vij_dev, double *Vji_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MALI_B200_H */
