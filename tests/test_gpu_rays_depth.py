"""compute_rays_depth on the GPU (mali_compute_rays_depth): chi, S, I, tau, the contribution function and the tau = 1
heights along the up-going rays of compute_rays.

The oracle's own formal solver, fed the device's chi and S, must reproduce the device's I at every depth bit for bit,
and the header's formulas in numpy must reproduce tau, contrib and z_tau1 bit for bit; I[0] is compute_rays' result;
chi, S and I agree with the oracle construction of tests/rays_depth_reference.py at new angles; and the result does not
depend on the selection of quantities, the batch, the column range, the angle chunking or the library build.  Every
achieved error is printed."""
import ctypes as C
import os

import numpy as np
import pytest

from helpers import load_golden
from rays_depth_reference import ray_terms, reference_rays_depth
from test_gpu_rays import (BATCH, MALI_EINVAL, TOL_I, TOL_I_CONVERGED, advance, engine_state, make_engine,
                           next_formal_solution_I, rel, thermo_problems, to_state)

pytestmark = pytest.mark.gpu

MU = [1.0, 0.6, 0.1]
QUANTITIES = ('I', 'chi', 'S', 'tau', 'contrib', 'z_tau1', 'height')


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def oracle_sweep(z, mu, chi, S, Istart):
    """The oracle's formal solver (formal_solver.py:46-142) of one up-going ray from a given lower-boundary intensity."""
    from oracle import mali_oracle as O
    z, chi, S = (np.ascontiguousarray(a, dtype=np.float64) for a in (z, chi, S))
    I, Psi = np.zeros(chi.shape[0]), np.zeros(chi.shape[0])
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    O.lib().lso_piecewise_1d_impl(float(mu), 1, float(Istart), dp(z), dp(chi), dp(S), chi.shape[0], dp(I), dp(Psi))
    return I


def check_sweep_bits(d, p, mus, label, device_boundary=False):
    """Criterion 1 and 4 on one column's RayDepthData: the oracle's piecewise_linear_1d on the device's chi and S gives
    the device's I; the header's formulas on the device's arrays give its tau, contrib and z_tau1; contrib telescopes.
    device_boundary: start the oracle's sweep from the device's I[N-1] (columns whose boundary Planck values were
    formed on the device) instead of the oracle's own thermalised boundary."""
    from oracle import mali_oracle as O
    N, Ns, nmu = d.I.shape
    z, T, wav = d.height, np.asarray(p['temperature'], dtype=np.float64), np.asarray(p['wavelength'])
    I_o = np.zeros_like(d.I)
    for la in range(Ns):
        for m in range(nmu):
            if device_boundary:
                I_o[:, la, m] = oracle_sweep(z, mus[m], d.chi[:, la, m], d.S[:, la, m], d.I[N - 1, la, m])
            else:
                I_o[:, la, m] = O.piecewise_linear_1d(z, T, mus[m], 1, wav[la], d.chi[:, la, m], d.S[:, la, m])[0]
    tau, contrib, zt = ray_terms(z, d.chi, d.S, d.I, mus)
    gap = np.abs(d.contrib.sum(axis=0) - d.I[0]) / np.abs(d.contrib).sum(axis=0)
    nan = int(np.isnan(d.z_tau1).sum())
    print('%s: oracle sweep on device chi/S: I max rel diff %.3e; tau %.3e, contrib %.3e, z_tau1 %.3e (%d NaN); '
          'telescoping gap %.3e; %d rays x %d depths'
          % (label, rel(d.I, I_o), rel(d.tau, tau), rel(d.contrib, contrib),
             rel(np.nan_to_num(d.z_tau1), np.nan_to_num(zt)), nan, float(gap.max()), Ns * nmu, N))
    assert same_bits(d.I, I_o)
    assert same_bits(d.tau, tau)
    assert same_bits(d.contrib, contrib)
    assert same_bits(d.z_tau1, zt)
    assert np.all(gap <= 1e-13)


# ---------------------------------------------------------------------------------------------------- 1, 2, 4. bits
CASES = [(n, path, k) for n in ('c1_falc_ca', 'c2_falc_cah', 'c2v_jitter_cah_0', 'stress_r10_d512')
         for path in ('stock', 'nospec') for k in (0, 6, 'conv') if not (n == 'stress_r10_d512' and k == 'conv')]


@pytest.mark.parametrize('name,path,k', CASES)
def test_sweep_bits_and_compute_rays(name, path, k):
    p, _ = load_golden(name)
    eng = make_engine(p, path=path)
    eng.upload_device_phi([p])
    to_state(eng, k)
    label = '%s %s k=%s' % (name, path, k)
    d = eng.compute_rays_depth(MU).column(0)
    check_sweep_bits(d, p, MU, label)
    assert same_bits(d.I[0], eng.compute_rays(MU)[0])
    # at the quadrature's angles I[0] is the next exact formal solution's I
    muz = np.asarray(p['muz'])
    q = eng.compute_rays_depth(muz, quantities=['I'])
    assert same_bits(q.I[:, 0], eng.compute_rays(muz))
    assert same_bits(q.I[:, 0], next_formal_solution_I(eng))
    print('%s: I[0] bit-identical to compute_rays at %s and at the quadrature angles (= next formal solution)'
          % (label, MU))
    eng.close()


@pytest.mark.parametrize('path', ['stock', 'nospec'])
def test_sweep_bits_upload_thermo_and_heights(path):
    """Columns set up from the thermodynamic state: the heights are formed on the device and returned by the call."""
    base, probs, eos, atoms = thermo_problems(3)
    eng = make_engine(base, 3, path=path)
    eng.set_eos(eos)
    eng.set_atoms(atoms)
    eng.upload_thermo(probs)
    advance(eng, 6)
    d = eng.compute_rays_depth(MU)
    colconst = eng.t_colconst.cpu().numpy().reshape(3, -1)
    N = d.height.shape[1]
    for c in range(3):
        # the heights are the run of colconst upload_thermo wrote, at the same offset in every column
        at = [o for o in np.nonzero(colconst[c] == d.height[c, 0])[0] if same_bits(colconst[c, o:o + N], d.height[c])]
        assert len(at) >= 1, c
        if c == 0:
            off = at[0]
        assert off in at
        q = dict(probs[c], wavelength=base['wavelength'])
        check_sweep_bits(d.column(c), q, MU, 'config-4 upload_thermo column %d %s' % (c, path), device_boundary=True)
    assert np.all(np.diff(d.height, axis=1) < 0)        # heights fall with depth index
    eng.close()


# ---------------------------------------------------------------------------------------------------- 3. oracle
@pytest.mark.parametrize('name', ['c1_falc_ca', 'c2_falc_cah', 'c2v_jitter_cah_0'])
@pytest.mark.parametrize('k', [6, 'conv'])
def test_oracle_at_new_angles(oracle, name, k):
    p, _ = load_golden(name)
    eng = make_engine(p, arith=None)
    eng.upload_device_phi([p])
    to_state(eng, k)
    d = eng.compute_rays_depth(MU).column(0)
    ref = reference_rays_depth(p, eng.n(0), eng.J(0), MU)
    bar = TOL_I_CONVERGED if k == 'conv' else TOL_I
    errs = {q: rel(getattr(d, q), ref[q]) for q in ('chi', 'S', 'I')}
    print('%s k=%s at %s vs oracle: %s' % (name, k, MU, ', '.join('%s %.3e' % kv for kv in errs.items())))
    assert same_bits(d.height, ref['height'])
    for q, e in errs.items():
        assert np.all(np.isfinite(getattr(d, q))) and e <= bar, q
    eng.close()


# ---------------------------------------------------------------------------------------------------- 5. physics
def test_physics_sanity():
    p, _ = load_golden('c2_falc_cah')
    eng = make_engine(p)
    eng.upload_device_phi([p])
    advance(eng, 6)
    mus = [1.0, 0.5, 0.1]
    d = eng.compute_rays_depth(mus).column(0)
    trans = np.asarray(p['trans']).reshape(-1, 6)
    Ns = d.I.shape[1]
    line = np.zeros(Ns, dtype=bool)
    for atom, i, j, isLine, Nblue, Nlam in trans:
        if isLine:
            line[Nblue:Nblue + Nlam] = True
    cont = np.nonzero(~line)[0]
    assert cont.size > 0
    t1 = d.tau[1:, cont, 0]
    worst = 0.0
    for m in (1, 2):
        tm = d.tau[1:, cont, m] * mus[m]
        worst = max(worst, float(np.max(np.abs(tm - t1) / t1)))
    print('continuum (%d wavelengths without an active line): max |tau(mu) mu - tau(1)| / tau(1) = %.3e'
          % (cont.size, worst))
    assert worst <= 1e-14
    zc1, zc01 = d.z_tau1[cont, 0], d.z_tau1[cont, 2]
    assert np.all(np.isfinite(zc1)) and np.all(zc01 >= zc1)
    # Ca II K: the line with lambda0 nearest 393.4 nm, at the wavelength nearest its centre
    lam0 = np.asarray(p['linepar'])[:, 3]
    t = min((t for t in range(trans.shape[0]) if trans[t, 3]), key=lambda t: abs(lam0[t] - 393.4))
    wl = np.asarray(p['wavelength'])
    la = int(np.argmin(np.abs(wl - lam0[t])))
    lc = int(cont[np.argmin(np.abs(wl[cont] - lam0[t]))])     # the nearest wavelength without an active line
    print('Ca II K (lambda0 %.4f nm, wavelength %d = %.4f nm): z_tau1 %.4e m; continuum at %.4f nm: %.4e m'
          % (lam0[t], la, wl[la], d.z_tau1[la, 0], wl[lc], d.z_tau1[lc, 0]))
    assert d.z_tau1[la, 0] > d.z_tau1[lc, 0]
    eng.close()


# ---------------------------------------------------------------------------------------------------- 6. invariance
def test_quantity_subsets_give_the_same_bits():
    p, _ = load_golden('c2v_jitter_cah_0')
    eng = make_engine(p)
    eng.upload_device_phi([p])
    advance(eng, 6)
    full = eng.compute_rays_depth_async(MU)
    full = {k: v.cpu().numpy() for k, v in full.items()}
    subsets = [(q,) for q in QUANTITIES] + [('I', 'z_tau1'), ('contrib',), ('chi', 'S', 'height'), ('tau', 'contrib')]
    for sub in subsets:
        got = eng.compute_rays_depth_async(MU, quantities=sub)
        assert tuple(got) == sub
        for k, v in got.items():
            assert same_bits(v.cpu().numpy(), full[k]), (sub, k)
    d = eng.compute_rays_depth(MU, quantities=['z_tau1'])
    assert d.I is None and d.tau is None and same_bits(d.z_tau1, full['z_tau1']) and same_bits(d.height, full['height'])
    # caller-owned outputs
    import torch
    out = {'I': torch.empty_like(torch.from_numpy(full['I'])).to(eng.device)}
    got = eng.compute_rays_depth_async(MU, quantities=['I', 'contrib'], out=out)
    assert got['I'] is out['I'] and same_bits(got['I'].cpu().numpy(), full['I'])
    print('%d quantity selections bit-identical to the full call' % (len(subsets) + 2))
    eng.close()


def test_batch_and_column_ranges_bitwise():
    probs = [load_golden(n)[0] for n in BATCH]
    eng = make_engine(probs[0], len(probs), arith=None)
    eng.upload_device_phi(probs)
    advance(eng, 6)
    full = eng.compute_rays_depth(MU)
    for c0, nc in ((0, 2), (2, 3), (5, 2), (6, 1), (1, 5)):
        part = eng.compute_rays_depth(MU, c0, nc)
        for q in QUANTITIES:
            assert same_bits(getattr(part, q), getattr(full, q)[c0:c0 + nc]), (c0, nc, q)
    for c in (0, 3, 6):
        one = make_engine(probs[c], arith=None)
        one.upload_device_phi([probs[c]])
        advance(one, 6)
        d = one.compute_rays_depth(MU)
        for q in QUANTITIES:
            assert same_bits(getattr(d, q)[0], getattr(full, q)[c]), (c, q)
        one.close()
    print('7-column batch: every quantity equal to column ranges and single-column engines')
    eng.close()


def test_angle_chunks():
    """nmu = 70 runs as 64 + 6 angles: the same bits as two calls, and as the reversed list."""
    p, _ = load_golden('c1_falc_ca')
    eng = make_engine(p)
    eng.upload_device_phi([p])
    advance(eng, 5)
    rng = np.random.default_rng(70)
    mus = np.concatenate([[1.0], 1.0 - rng.random(69)])
    d = eng.compute_rays_depth(mus)
    a, b = eng.compute_rays_depth(mus[:64]), eng.compute_rays_depth(mus[64:])
    r = eng.compute_rays_depth(mus[::-1])
    for q in ('I', 'chi', 'S', 'tau', 'contrib', 'z_tau1'):
        v = getattr(d, q)
        assert v.shape[-1] == 70
        assert same_bits(v, np.concatenate([getattr(a, q), getattr(b, q)], axis=-1)), q
        assert same_bits(v, getattr(r, q)[..., ::-1]), q
    assert same_bits(d.I[:, 0], eng.compute_rays(mus))
    print('70 angles: equal to 64 + 6 and to the reversed list')
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
        out.append(eng.compute_rays_depth(MU + list(np.asarray(p['muz']))))
        assert not eng.t_status.cpu().numpy().any()
        eng.close()
    for q in QUANTITIES:
        assert same_bits(getattr(out[0], q), getattr(out[1], q)), q


def test_no_side_effects_on_engine_tensors():
    from lightspinner_b200 import NgOptions
    p, _ = load_golden('c2_falc_cah')
    eng = make_engine(p, ng=NgOptions())
    eng.upload_device_phi([p])
    eng.reset_iteration_state()
    eng.iterate_async(10)
    before = engine_state(eng)
    assert 't_ng_hist' in before and 't_aDamp' in before
    eng.compute_rays_depth(MU)
    eng.compute_rays_depth(np.linspace(0.01, 1.0, 70), quantities=['contrib', 'z_tau1'])
    after = engine_state(eng)
    for key in before:
        assert np.array_equal(before[key].view(np.uint8), after[key].view(np.uint8)), key
    print('%d engine tensors unchanged' % len(before))
    eng.close()


# ---------------------------------------------------------------------------------------------------- Python API
def test_context_and_batch_context():
    from helpers import fake_reference_objects
    from lightspinner_b200 import BatchContext, Context, RayDepthData
    p, _ = load_golden('c1_falc_ca')
    ctx = Context(*fake_reference_objects(p))
    for it in range(1, 7):
        ctx.formal_sol_gamma_matrices()
        if it > 3:
            ctx.stat_equil()
    d = ctx.compute_rays_depth([1.0, 0.5])
    N, Ns = int(p['Nspace']), int(p['Nspect'])
    assert isinstance(d, RayDepthData)
    assert d.I.shape == (N, Ns, 2) and d.z_tau1.shape == (Ns, 2) and d.height.shape == (N,)
    assert same_bits(d.I[0], ctx.compute_rays([1.0, 0.5]))
    n = ctx.activeAtoms[0].n                          # edits through the eqPops alias are honoured
    n[1] *= 1.05
    d2 = ctx.compute_rays_depth([1.0, 0.5], quantities=['chi'])
    assert d2.I is None and not same_bits(d2.chi, d.chi)
    ctx.close()
    cols = [fake_reference_objects(load_golden(nm)[0]) for nm in ('c2_falc_cah', 'c2v_jitter_cah_0')]
    batch = BatchContext(cols)
    batch.iterate()
    B = batch.compute_rays_depth(MU)
    assert B.I.shape[0] == 2
    for c in range(2):
        one = batch[c].compute_rays_depth(MU)
        for q in QUANTITIES:
            assert same_bits(getattr(one, q), getattr(B, q)[c]), (c, q)
    batch.close()


# ---------------------------------------------------------------------------------------------------- 7. errors
def test_c_entry_point_rejects_bad_arguments():
    import torch
    from lightspinner_b200 import _capi
    p, _ = load_golden('c1_falc_ca')
    eng = make_engine(p)
    eng.upload_device_phi([p])
    L, h, b = eng.lib, eng._handle, C.byref(eng.bufs)
    N, S = int(p['Nspace']), int(p['Nspect'])
    buf = {k: torch.zeros(N * S * 64, dtype=torch.float64, device=eng.device) for k in QUANTITIES}
    P = lambda t: C.c_void_p(t.data_ptr())
    prof = [P(eng.t_aDamp), P(eng.t_vBroad), P(eng.t_vlos)]

    def call(col0=0, ncol=1, mus=(1.0,), nmu=None, prof_=None, outs=QUANTITIES, desc=True):
        m = np.asarray(mus, dtype=np.float64)
        mp = m.ctypes.data_as(C.POINTER(C.c_double)) if m.size else None
        o = _capi.RaysDepthOut(**{k: P(buf[k]) for k in outs})
        return L.mali_compute_rays_depth(h, b, col0, ncol, len(m) if nmu is None else nmu, mp, *(prof_ or prof),
                                         C.byref(o) if desc else None, None, eng._stream())

    assert call() == 0
    assert call(outs=('height',)) == 0 and call(outs=('tau',)) == 0 and call(outs=('I', 'chi')) == 0
    bad = [dict(col0=-1), dict(ncol=0), dict(ncol=2), dict(col0=1), dict(mus=()), dict(mus=[0.5] * 65),
           dict(mus=[0.0]), dict(mus=[-0.2]), dict(mus=[1.5]), dict(mus=[float('nan')]), dict(mus=[float('inf')]),
           dict(mus=[0.5, 0.0]), dict(prof_=[None, prof[1], prof[2]]), dict(prof_=[prof[0], prof[1], None]),
           dict(outs=()), dict(desc=False), dict(outs=('contrib',)), dict(outs=('z_tau1',)),
           dict(outs=('I', 'contrib', 'z_tau1'))]
    for kw in bad:
        assert call(**kw) == MALI_EINVAL, kw
        print('MALI_EINVAL for %s: %s' % (kw, L.mali_last_error().decode()))
    torch.cuda.synchronize()
    eng.close()


def test_python_layer_errors():
    import torch
    p, _ = load_golden('c1_falc_ca')
    eng = make_engine(p, 3)
    eng.upload_device_phi([p, p])
    for bad in (0.0, 1.5, float('nan'), [], [[0.5]]):
        with pytest.raises(ValueError):
            eng.compute_rays_depth(bad, 0, 2)
    with pytest.raises(ValueError):
        eng.compute_rays_depth(0.5, 2, 2)
    for q in (['I', 'J'], [], ['tau', 'tau']):
        with pytest.raises(ValueError):
            eng.compute_rays_depth(0.5, 0, 1, quantities=q)
    with pytest.raises(ValueError):        # an out tensor of the wrong shape, or for a quantity not requested
        eng.compute_rays_depth_async(0.5, 0, 1, quantities=['I'],
                                     out={'I': torch.empty(1, 2, 3, dtype=torch.float64, device=eng.device)})
    with pytest.raises(ValueError):
        eng.compute_rays_depth_async(0.5, 0, 1, quantities=['I'],
                                     out={'tau': torch.empty(1, 2, 3, dtype=torch.float64, device=eng.device)})
    # column 2 was never given profile inputs; columns uploaded with host profiles lose theirs
    with pytest.raises(ValueError, match=r'\[2\]'):
        eng.compute_rays_depth(0.5)
    hp = eng.hostpack_size()
    from lightspinner_b200.tables import pack_column
    pinned = torch.empty(hp, dtype=torch.float64, pin_memory=True)
    pack_column(eng.mt, eng.lay, p, out=pinned.numpy())
    eng.upload_packed(pinned, 1, 1)
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match=r'\[1\]'):
        eng.compute_rays_depth(0.5, 0, 2)
    assert eng.compute_rays_depth(0.5, 0, 1).I.shape == (1, int(p['Nspace']), int(p['Nspect']), 1)
    eng.close()
