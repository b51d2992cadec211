"""compute_rates on the GPU (mali_compute_rates): the radiative rates R_ij, R_ji of every transition from the current
state.

They must agree with the oracle construction of tests/rates_reference.py, satisfy the J identity with the J of the next
formal solution, make the populations solve the plain statistical-equilibrium equations at a tight fixed point, change
nothing the iteration uses, and not depend on the batch, the column range, the kernel path or the library build.  Every
achieved error is printed."""
import ctypes as C
import os

import numpy as np
import pytest

from helpers import fake_reference_objects, load_golden, select_rays, only_transitions
from rates_reference import net_rates, reference_rates, se_residual
from test_gpu_rays import advance, make_engine, thermo_problems

pytestmark = pytest.mark.gpu

MALI_EINVAL = -1
# Both sides take the same n, J and line profiles (host-profile uploads) and evaluate the same separately rounded
# expressions; only the order of the sums over wavelength, angle and direction differs.
TOL_R = 1e-12
TOL_J_IDENTITY = 1e-13
# The plain statistical-equilibrium residual (rates_reference.se_residual) at tolJ = tolPops = 1e-9: the oracle loop on
# c1_falc_ca measured 1.3e-8 (tests/test_rates_host.py), the same bar applies to the device loop.
SE_BAR = 5e-8
# Context forms its line profiles on the device (mali_compute_phi, ~1e-13 from scipy's wofz, which the reference uses);
# carried through a converged, optically thick line this is the bar of the compute_rays suite.
TOL_R_DEVICE_PHI = 5e-11

FIXTURES = ['c1_falc_ca', 'c2_falc_cah', 'c2v_jitter_cah_0', 'stress_r10_d512']


def converge(eng, tol=(2e-3, 1e-3), max_iter=400):
    import torch
    eng.reset_iteration_state()
    eng.iterate_async(max_iter, *tol)
    torch.cuda.synchronize()
    eng.raise_on_faults()
    assert (eng.t_done.cpu().numpy() == 1).all()


def to_state(eng, k):
    converge(eng) if k == 'conv' else advance(eng, k)


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    nz = b != 0
    assert np.array_equal(a == 0, b == 0)
    return float(np.max(np.abs(a[nz] - b[nz]) / np.abs(b[nz]))) if nz.any() else 0.0


def check_reference(eng, p, label, col=0, tol=TOL_R):
    r = eng.compute_rates(col, 1)
    Rij, Rji = reference_rates(p, eng.n(col), eng.J(col))
    e = max(rel(r.Rij[0], Rij), rel(r.Rji[0], Rji))
    print('%s: compute_rates vs oracle construction: max rel err %.3e (%d values)' % (label, e, 2 * Rij.size))
    # the terms are non-negative wherever the sweep's I is: the reference's last-point quirk gives negative I at the top
    # of the 512-depth fixture's first wavelengths, and so R_ij < 0 at k = 0 for the continua there, on both sides
    neg = (Rij < 0).sum() + (Rji < 0).sum()
    assert np.array_equal(r.Rij[0] < 0, Rij < 0) and np.array_equal(r.Rji[0] < 0, Rji < 0)
    if neg:
        print('  %d negative entries, all at the top (k = 0), on both sides' % neg)
        assert not (Rij[:, 1:] < 0).any() and not (Rji[:, 1:] < 0).any()
    assert np.array_equal(r.net[0], net_rates(p, eng.n(col), r.Rij[0], r.Rji[0]))
    assert e <= tol
    return r


# ---------------------------------------------------------------------------------------------------- 1. oracle
MODES = [('stock', 'exact'), ('stock', 'contracted'), ('nospec', 'exact')]
CASES = [(n, path, arith, k) for n in FIXTURES for path, arith in MODES for k in (0, 6, 'conv')
         if not (n == 'stress_r10_d512' and k == 'conv')]


@pytest.mark.parametrize('name,path,arith,k', CASES)
def test_against_reference(oracle, name, path, arith, k):
    p, _ = load_golden(name)
    eng = make_engine(p, path=path, arith=arith)
    eng.upload([p])
    to_state(eng, k)
    check_reference(eng, p, '%s %s %s k=%s' % (name, path, arith, k))
    eng.close()


# ---------------------------------------------------------------------------------------------------- 2. J identity
def j_identity(eng, col, J):
    """R_ij = 4 pi sum_la wla V_ij J, R_ji = 4 pi sum_la wla (U_ji + V_ji J) [Ntrans, Nspace] from the device tables
    (mali_uv at angle 0, direction 0), and the transitions for which it holds: continua, and lines when the column's
    profiles do not depend on the angle (vlos = 0)."""
    mt = eng.mt
    N = mt.Nspace
    static = not np.any(eng.t_vlos[col].cpu().numpy()) if eng._has_profile[col] else False
    Rij, Rji = np.zeros((mt.Ntrans, N)), np.zeros((mt.Ntrans, N))
    mask = np.zeros(mt.Ntrans, bool)
    from lightspinner_b200.tables import HC
    for t in range(mt.Ntrans):
        atom, i, j, isLine, Nblue, Nlam = (int(x) for x in mt.trans[t])
        if isLine and not static:
            continue
        mask[t] = True
        wphi = eng.line_profile(col, t)[1] if isLine else None
        for la in range(Nblue, Nblue + Nlam):
            U, Vij, Vji = eng.uv(col, t, la, 0, 0)
            w = mt.wlambda[mt.toff[t] + la - Nblue]
            w = w * wphi / HC if isLine else mt.wlacont[mt.toff[t] + la - Nblue]
            w = w * 4 * np.pi
            Rij[t] += w * Vij * J[la]
            Rji[t] += w * (U + Vji * J[la])
    return Rij, Rji, mask


def check_j_identity(eng, label, cols=(0,)):
    r = eng.compute_rates()
    eng.formal_sol_gamma_matrices()
    lines = eng.mt.trans[:, 3] != 0
    for c in cols:
        Iij, Iji, mask = j_identity(eng, c, eng.J(c))
        cont, lin = ~lines, mask & lines
        e_c = max(rel(r.Rij[c][cont], Iij[cont]), rel(r.Rji[c][cont], Iji[cont]))
        e_l = max(rel(r.Rij[c][lin], Iij[lin]), rel(r.Rji[c][lin], Iji[lin])) if lin.any() else None
        print('%s col %d: J identity: continua %.3e, lines %s' % (label, c, e_c, 'n/a' if e_l is None else '%.3e' % e_l))
        assert e_c <= TOL_J_IDENTITY
        if e_l is not None:
            assert e_l <= TOL_J_IDENTITY


@pytest.mark.parametrize('name', FIXTURES)
def test_j_identity(name):
    p, _ = load_golden(name)
    eng = make_engine(p, arith='exact')
    eng.upload_device_phi([p])
    advance(eng, 6)
    check_j_identity(eng, name)
    eng.close()


# ---------------------------------------------------------------------------------------------------- 3. fixed point
@pytest.mark.parametrize('ng', [False, True])
def test_statistical_equilibrium_at_the_fixed_point(ng):
    from lightspinner_b200 import NgOptions
    p, _ = load_golden('c1_falc_ca')
    res = {}
    for tol in ((2e-3, 1e-3), (1e-9, 1e-9)):
        eng = make_engine(p, ng=NgOptions() if ng else None)
        eng.upload([p])
        converge(eng, tol, max_iter=1000)
        r = eng.compute_rates()
        res[tol] = se_residual(p, eng.n(0), r.Rij[0], r.Rji[0])
        print('c1_falc_ca ng=%s tol %s: %d iterations, plain statistical-equilibrium residual %.3e'
              % (ng, tol, int(eng.t_iter[0]), res[tol]))
        eng.close()
    assert res[(1e-9, 1e-9)] < 1e-3 * res[(2e-3, 1e-3)]
    assert res[(1e-9, 1e-9)] <= SE_BAR


# ---------------------------------------------------------------------------------------------------- 4. model shapes
@pytest.mark.parametrize('model', ['c2x5', 'c1x5', 'merged12', 'merged16'])
def test_model_shapes(oracle, model):
    import model_shapes as ms
    q = ms.build(model)
    eng = make_engine(q)
    eng.upload([q])
    advance(eng, 6)
    info = eng.model_info()
    check_reference(eng, q, '%s (max %d slots per tile, max %d levels)' % (model, info['max_slots'], info['max_levels']))
    eng.close()


# ---------------------------------------------------------------------------------------------------- 5. rays, thermo
@pytest.mark.parametrize('rays', [[2], [0, 2, 4]])
def test_ray_counts(oracle, rays):
    p = select_rays(load_golden('c1_falc_ca')[0], rays)
    eng = make_engine(p)
    eng.upload([p])
    advance(eng, 6)
    check_reference(eng, p, 'c1_falc_ca with %d rays' % len(rays))
    eng.close()


@pytest.mark.parametrize('path', ['stock', 'nospec'])
def test_upload_thermo_columns(path):
    base, probs, eos, atoms = thermo_problems(3)
    eng = make_engine(base, 3, path=path, arith='exact')
    eng.set_eos(eos)
    eng.set_atoms(atoms)
    eng.upload_thermo(probs)
    advance(eng, 6)
    full = eng.compute_rates()
    for c in range(3):
        assert np.array_equal(eng.compute_rates(c, 1).Rij[0], full.Rij[c])
    check_j_identity(eng, 'config-4 x3 upload_thermo %s' % path, cols=(0, 1, 2))
    eng.close()


# ---------------------------------------------------------------------------------------------------- 6. bit identity
BATCH = ['c2_falc_cah', 'c2v_jitter_cah_0', 'c2v_jitter_cah_1', 'c2v_jitter_cah_0', 'c2_falc_cah', 'c2v_jitter_cah_1',
         'c2v_jitter_cah_0']


def test_batch_and_column_ranges_bitwise():
    probs = [load_golden(n)[0] for n in BATCH]
    eng = make_engine(probs[0], len(probs), arith=None)
    eng.upload_device_phi(probs)
    advance(eng, 6)
    full = eng.compute_rates()
    for c0, nc in ((0, 2), (2, 3), (5, 2), (6, 1), (1, 5)):
        part = eng.compute_rates(c0, nc)
        for f in ('Rij', 'Rji', 'net'):
            assert np.array_equal(getattr(part, f), getattr(full, f)[c0:c0 + nc]), (f, c0, nc)
    for c in (0, 3, 6):
        one = make_engine(probs[c], arith=None)
        one.upload_device_phi([probs[c]])
        advance(one, 6)
        r = one.compute_rates()
        assert np.array_equal(r.Rij[0], full.Rij[c]) and np.array_equal(r.Rji[0], full.Rji[c]), c
        one.close()
    print('7-column batch: equal to column ranges and single-column engines, %d values' % (2 * full.Rij.size))
    eng.close()


def test_checked_library_gives_the_same_bits():
    from lightspinner_b200 import build
    assert os.path.isfile(build.CHECK_LIB)
    p, _ = load_golden('c2v_jitter_cah_0')
    out = []
    for lib in (None, build.CHECK_LIB):
        eng = make_engine(p, library=lib)
        eng.upload_device_phi([p])
        advance(eng, 6)
        r = eng.compute_rates()
        out.append((r.Rij, r.Rji))
        assert not eng.t_status.cpu().numpy().any()
        eng.close()
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


def test_stock_and_generic_paths_given_the_same_state():
    p, _ = load_golden('c2v_jitter_cah_0')
    a, b = make_engine(p), make_engine(p, path='nospec')
    assert a.model_info()['spec_tiles'] > 0 and b.model_info()['spec_tiles'] == 0
    for e in (a, b):
        e.upload_device_phi([p])
        advance(e, 6)
    b.t_pops.copy_(a.t_pops)
    b.t_J.copy_(a.t_J)
    ra, rb = a.compute_rates(), b.compute_rates()
    assert np.array_equal(ra.Rij, rb.Rij) and np.array_equal(ra.Rji, rb.Rji) and np.array_equal(ra.net, rb.net)
    a.close()
    b.close()


# ---------------------------------------------------------------------------------------------------- 7. no side effects
def engine_state(eng):
    import torch
    return {k: v.cpu().numpy().copy() for k, v in vars(eng).items()
            if isinstance(v, torch.Tensor) and k not in ('_rays_bad', 't_scratch')}


def test_no_side_effects_on_engine_tensors():
    from lightspinner_b200 import NgOptions
    p, _ = load_golden('c2_falc_cah')
    eng = make_engine(p, ng=NgOptions())
    eng.upload_device_phi([p])
    eng.reset_iteration_state()
    eng.iterate_async(10)
    before = engine_state(eng)
    assert 't_ng_hist' in before and 't_Gamma' in before
    eng.compute_rates()
    after = engine_state(eng)
    for key in before:
        assert np.array_equal(before[key].view(np.uint8), after[key].view(np.uint8)), key
    print('%d engine tensors unchanged (%s)' % (len(before), ', '.join(sorted(before))))
    eng.close()


@pytest.mark.parametrize('ng', [False, True])
def test_free_running_loop_is_unchanged(ng):
    import torch
    from lightspinner_b200 import NgOptions
    p, _ = load_golden('c2v_jitter_cah_0')
    res = []
    for with_rates in (False, True):
        eng = make_engine(p, arith=None, ng=NgOptions() if ng else None)
        eng.upload_device_phi([p])
        eng.reset_iteration_state()
        for _ in range(40):
            eng.iterate_async(2)
            if with_rates:
                eng.compute_rates_async()
        eng.iterate_async(400)
        torch.cuda.synchronize()
        res.append((eng.t_iter.cpu().numpy().copy(), eng.n(0), eng.J(0), eng.I(0), eng.Gamma(0)))
        eng.close()
    print('ng=%s: %d iterations with and without a compute_rates call between every two iterations' % (ng, res[0][0][0]))
    for a, b in zip(res[0], res[1]):
        assert np.array_equal(a, b)


# ---------------------------------------------------------------------------------------------------- 8. Python API
def test_context_after_the_test_py_loop(oracle):
    from lightspinner_b200 import Context, RadiativeRates
    p, _ = load_golden('c1_falc_ca')
    atmos, spect, eqPops, bg = fake_reference_objects(p)
    ctx = Context(atmos, spect, eqPops, bg)
    trans = [t for a in ctx.activeAtoms for t in a.trans]
    assert all(not t.Rij.any() and not t.Rji.any() for t in trans)     # zeros before any call
    dJ, dPops, it = 1.0, 1.0, 0
    while dJ > 2e-3 or dPops > 1e-3:                # test.py:20-29
        it += 1
        dJ = ctx.formal_sol_gamma_matrices()
        if it > 3:
            dPops = ctx.stat_equil()
    J_before = ctx.J.copy()
    r = ctx.compute_rates()
    assert isinstance(r, RadiativeRates) and r.Rij.shape == (len(trans), int(p['Nspace']))
    eng = ctx._engine.compute_rates(0, 1)
    assert np.array_equal(r.Rij, eng.Rij[0]) and np.array_equal(r.Rji, eng.Rji[0]) and np.array_equal(r.net, eng.net[0])
    for t in trans:
        assert np.array_equal(t.Rij, r.Rij[t.index]) and np.array_equal(t.Rji, r.Rji[t.index])
    assert np.array_equal(ctx.J, J_before)          # cached results stay valid
    # edits through the eqPops alias are honoured
    n = ctx.activeAtoms[0].n
    n[1] *= 1.05
    r2 = ctx.compute_rates()
    Rij, Rji = reference_rates(p, n, ctx.J)
    e = max(rel(r2.Rij, Rij), rel(r2.Rji, Rji))
    print('Context after %d iterations: edited populations, compute_rates vs oracle %.3e' % (it, e))
    assert not np.array_equal(r2.Rij, r.Rij) and e <= TOL_R_DEVICE_PHI
    assert np.array_equal(r2.net, net_rates(p, n, r2.Rij, r2.Rji))
    for t in trans:
        assert np.array_equal(t.Rij, r2.Rij[t.index])
    ctx.close()


def test_batch_context_rows():
    from lightspinner_b200 import BatchContext
    cols = [fake_reference_objects(load_golden(n)[0]) for n in ('c2_falc_cah', 'c2v_jitter_cah_0', 'c2v_jitter_cah_1')]
    batch = BatchContext(cols)
    batch.iterate()
    B = batch.compute_rates()
    mt = batch[0]._engine.mt
    assert B.Rij.shape == B.Rji.shape == B.net.shape == (3, mt.Ntrans, mt.Nspace)
    for k in range(3):
        one = batch[k].compute_rates()
        assert np.array_equal(B.Rij[k], one.Rij) and np.array_equal(B.Rji[k], one.Rji) and np.array_equal(B.net[k], one.net)
        t = batch[k].activeAtoms[1].trans[0]
        assert np.array_equal(t.Rij, B.Rij[k][t.index])
    batch.close()


def test_out_tensors_and_shapes():
    import torch
    p, _ = load_golden('c1_falc_ca')
    eng = make_engine(p, 3)
    eng.upload([p, p, p])
    advance(eng, 4)
    T, N = eng.mt.Ntrans, eng.mt.Nspace
    f64 = dict(dtype=torch.float64, device=eng.device)
    out = (torch.full((2, T, N), -1.0, **f64), torch.full((2, T, N), -1.0, **f64))
    Rij, Rji = eng.compute_rates_async(1, 2, out=out)
    assert Rij is out[0] and Rji is out[1]
    ref = eng.compute_rates(1, 2)
    assert np.array_equal(Rij.cpu().numpy(), ref.Rij) and np.array_equal(Rji.cpu().numpy(), ref.Rji)
    assert eng.compute_rates().Rij.shape == (3, T, N)
    good = torch.empty(2, T, N, **f64)
    bad = [good, (good,), (good, good, good), (good, torch.empty(2, T, N, dtype=torch.float32, device=eng.device)),
           (good, torch.empty(2, T, N + 1, **f64)), (good, torch.empty(2, N, T, **f64).transpose(1, 2)),
           (good, torch.empty(2, T, N, dtype=torch.float64))]
    for o in bad:
        with pytest.raises(ValueError):
            eng.compute_rates_async(1, 2, out=o)
    for c0, nc in ((-1, 1), (0, 0), (2, 2), (3, None)):
        with pytest.raises(ValueError):
            eng.compute_rates(c0, nc)
    eng.close()


def test_model_without_transitions():
    p, _ = load_golden('c1_falc_ca')
    q = only_transitions(p, [])
    eng = make_engine(q)
    eng.upload([q])
    advance(eng, 2)
    r = eng.compute_rates()
    assert r.Rij.shape == r.Rji.shape == r.net.shape == (1, 0, int(p['Nspace']))
    import torch
    sentinel = torch.full((4,), 7.0, dtype=torch.float64, device=eng.device)
    P = lambda t: C.c_void_p(t.data_ptr())
    assert eng.lib.mali_compute_rates(eng._handle, C.byref(eng.bufs), 0, 1, P(sentinel), P(sentinel), None,
                                      eng._stream()) == 0
    assert (sentinel.cpu().numpy() == 7.0).all()
    eng.close()


def test_c_entry_point_rejects_bad_arguments():
    import torch
    from lightspinner_b200 import _capi
    p, _ = load_golden('c1_falc_ca')
    eng = make_engine(p)
    eng.upload([p])
    L, h = eng.lib, eng._handle
    n = eng.mt.Ntrans * eng.mt.Nspace
    Rij, Rji = (torch.zeros(n, dtype=torch.float64, device=eng.device) for _ in range(2))
    P = lambda t: C.c_void_p(t.data_ptr())

    def call(col0=0, ncol=1, rij=None, rji=None, bufs=None, handle=None):
        return L.mali_compute_rates(handle if handle is not None else h, C.byref(bufs or eng.bufs), col0, ncol,
                                    P(Rij) if rij is None else rij, P(Rji) if rji is None else rji, None, eng._stream())

    assert call() == 0
    for kw in (dict(col0=-1), dict(ncol=0), dict(ncol=2), dict(col0=1), dict(rij=C.c_void_p(0)), dict(rji=C.c_void_p(0))):
        assert call(**kw) == MALI_EINVAL, kw
        print('MALI_EINVAL for %s: %s' % (kw, L.mali_last_error().decode()))
    for field in ('colconst', 'pops', 'J', 'scratch'):
        b = _capi.Buffers.from_buffer_copy(eng.bufs)
        setattr(b, field, None)
        assert call(bufs=b) == MALI_EINVAL, field
        print('MALI_EINVAL for a null %s: %s' % (field, L.mali_last_error().decode()))
    assert L.mali_compute_rates(None, C.byref(eng.bufs), 0, 1, P(Rij), P(Rji), None, eng._stream()) == MALI_EINVAL
    assert L.mali_compute_rates(h, None, 0, 1, P(Rij), P(Rji), None, eng._stream()) == MALI_EINVAL
    eng.close()
