"""compute_rays on the GPU (mali_compute_rays): the emergent intensity at user angles from the current state.

It must be exactly the I of the next formal solution when it is given the quadrature's own angles (exact arithmetic),
agree with the oracle construction of tests/rays_reference.py at new angles, change nothing the iteration uses, and not
depend on the batch, the column range, the angle chunking or the library build.  Every achieved error is printed."""
import os
import warnings

import numpy as np
import pytest

from helpers import fake_reference_objects, load_golden, load_setup_inputs, select_rays
from rays_reference import reference_rays

pytestmark = pytest.mark.gpu

MU_NEW = [1.0, 0.9, 0.6, 0.33, 0.1, 0.05]
MALI_EINVAL = -1
TOL_I = 1e-11          # the I bar of the parity suite; the device and scipy Voigt functions differ by <= 3e-14
# At convergence on CaII+H/FALC the oracle comparison measured 2.0e-11 (B200).  Both sides get the same n and J and
# evaluate the same exact arithmetic (test 1 shows the sweep bit-identical to the formal solution), so the difference
# is that of the two Voigt functions carried through the converged, optically thick line profiles.
TOL_I_CONVERGED = 5e-11


def make_engine(p, ncol=1, path='stock', arith='exact', **kw):
    """MaliEngine on the stock library ('stock') or with every tile on the generic kernel ('nospec')."""
    from lightspinner_b200.engine import MaliEngine
    if path == 'nospec':
        os.environ['MALI_NO_SPEC'] = '1'
    try:
        with warnings.catch_warnings():
            warnings.simplefilter('ignore', RuntimeWarning)     # the generic-fallback notice
            return MaliEngine(p, ncol, arith=arith, **kw)
    finally:
        os.environ.pop('MALI_NO_SPEC', None)


def advance(eng, k):
    """k iterations of the loop of test.py:20-29 through the per-call entry points."""
    for it in range(1, k + 1):
        eng.formal_sol_gamma_matrices()
        if it > 3:
            eng.stat_equil()


def converge(eng):
    import torch
    eng.reset_iteration_state()
    eng.iterate_async(400)
    torch.cuda.synchronize()
    eng.raise_on_faults()
    assert (eng.t_done.cpu().numpy() == 1).all()


def to_state(eng, k):
    converge(eng) if k == 'conv' else advance(eng, k)


def next_formal_solution_I(eng):
    eng.formal_sol_gamma_matrices()
    return np.stack([eng.I(c) for c in range(eng.ncol)])


def rel(a, b):
    b = np.asarray(b)
    nz = b != 0
    return float(np.max(np.abs(a[nz] - b[nz]) / np.abs(b[nz]))) if nz.any() else 0.0


def check_self_consistency(eng, p, label):
    R = eng.compute_rays(np.asarray(p['muz']))
    I = next_formal_solution_I(eng)
    print('%s: compute_rays(muz) vs next formal solution: max rel diff %.3e, %d values' % (label, rel(R, I), R.size))
    assert R.shape == I.shape
    assert np.array_equal(R, I)


# ---------------------------------------------------------------------------------------------------- 1. exact bits
CASES = [(n, path, k) for n in ('c1_falc_ca', 'c2_falc_cah', 'c2v_jitter_cah_0', 'stress_r10_d512')
         for path in ('stock', 'nospec') for k in (1, 6, 'conv') if not (n == 'stress_r10_d512' and k == 'conv')]


@pytest.mark.parametrize('name,path,k', CASES)
def test_self_consistency_exact(name, path, k):
    p, _ = load_golden(name)
    eng = make_engine(p, path=path)
    eng.upload_device_phi([p])
    to_state(eng, k)
    check_self_consistency(eng, p, '%s %s k=%s' % (name, path, k))
    eng.close()


def thermo_problems(ncol):
    """config-4 columns set up from the thermodynamic state (the recipe of tools/ng_converge.py)."""
    from lightspinner_b200 import synth
    from lightspinner_b200.atoms import AtomTables
    from lightspinner_b200.eos import EosTables
    zeos = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'eos.npz'))
    base, _ = load_golden('c2_falc_cah')
    atoms4, _ = load_setup_inputs('c2_falc_cah')
    names = [str(x).strip().upper() for x in base['atom_names']]
    probs = []
    for c in range(ncol):
        T, ne, vl = synth.jitter_atmosphere(c, zeos['falc_T'], zeos['falc_ne'])
        probs.append(dict(temperature=T, ne=ne, vlos=vl, nHTot=zeos['falc_nHTot'], cmass=zeos['falc_cmass'],
                          vturb=base['vturb'], nTotal=np.stack([atoms4[nm]['abundance'] * zeos['falc_nHTot'] for nm in names]),
                          aDamp=base['aDamp']))
    return base, probs, EosTables.from_arrays(zeos), AtomTables.from_arrays([dict(atoms4[nm]) for nm in names])


@pytest.mark.parametrize('path', ['stock', 'nospec'])
def test_self_consistency_upload_thermo(path):
    """The Doppler widths formed on the device by mali_setup_columns are the ones compute_rays reads."""
    base, probs, eos, atoms = thermo_problems(3)
    eng = make_engine(base, 3, path=path)
    eng.set_eos(eos)
    eng.set_atoms(atoms)
    eng.upload_thermo(probs)
    advance(eng, 6)
    check_self_consistency(eng, base, 'config-4 x3 upload_thermo %s' % path)
    eng.close()


def test_self_consistency_tiles_with_more_than_8_slots():
    import model_shapes as ms
    q = ms.build('c2x5')
    eng = make_engine(q)
    assert eng.model_info()['max_slots'] > 8
    eng.upload_device_phi([q])
    advance(eng, 6)
    check_self_consistency(eng, q, 'c2x5 (max %d slots per tile)' % eng.model_info()['max_slots'])
    eng.close()


# ---------------------------------------------------------------------------------------------------- 2. contracted
@pytest.mark.parametrize('name', ['c1_falc_ca', 'c2_falc_cah', 'c2v_jitter_cah_0'])
def test_contracted_formal_solution(name):
    p, _ = load_golden(name)
    eng = make_engine(p, arith='contracted')
    eng.upload_device_phi([p])
    advance(eng, 6)
    R = eng.compute_rays(np.asarray(p['muz']))
    I = next_formal_solution_I(eng)
    e = rel(R, I)
    print('%s: exact compute_rays vs contracted formal solution: %.3e' % (name, e))
    assert e <= TOL_I


# ---------------------------------------------------------------------------------------------------- 3. oracle
@pytest.mark.parametrize('name', ['c1_falc_ca', 'c2_falc_cah', 'c2v_jitter_cah_0'])
@pytest.mark.parametrize('k', [6, 'conv'])
def test_oracle_at_new_angles(oracle, name, k):
    p, _ = load_golden(name)
    eng = make_engine(p, arith=None)
    eng.upload_device_phi([p])
    to_state(eng, k)
    R = eng.compute_rays(MU_NEW)[0]
    ref = reference_rays(p, eng.n(0), eng.J(0), MU_NEW)
    e = rel(R, ref)
    nz = ref != 0
    err = np.zeros_like(R)
    err[nz] = np.abs(R[nz] - ref[nz]) / np.abs(ref[nz])
    la, m = np.unravel_index(np.argmax(err), err.shape)
    print('%s k=%s: compute_rays at %s vs oracle: max rel err %.3e (wavelength %d, mu %g, I %.3e)'
          % (name, k, MU_NEW, e, la, MU_NEW[m], ref[la, m]))
    assert np.all(np.isfinite(R)) and np.array_equal(R == 0, ref == 0)
    assert e <= (TOL_I_CONVERGED if k == 'conv' else TOL_I)
    eng.close()


# ---------------------------------------------------------------------------------------------------- 4. no side effects
def engine_state(eng):
    import torch
    return {k: v.cpu().numpy().copy() for k, v in vars(eng).items() if isinstance(v, torch.Tensor) and k != '_rays_bad'}


def test_no_side_effects_on_engine_tensors():
    from lightspinner_b200 import NgOptions
    p, _ = load_golden('c2_falc_cah')
    eng = make_engine(p, ng=NgOptions())
    eng.upload_device_phi([p])
    eng.reset_iteration_state()
    eng.iterate_async(10)
    before = engine_state(eng)
    assert 't_ng_hist' in before and 't_aDamp' in before
    eng.compute_rays(MU_NEW)
    eng.compute_rays(np.linspace(0.01, 1.0, 100))
    after = engine_state(eng)
    for key in before:
        assert np.array_equal(before[key].view(np.uint8), after[key].view(np.uint8)), key
    print('%d engine tensors unchanged (%s)' % (len(before), ', '.join(sorted(before))))


@pytest.mark.parametrize('ng', [False, True])
def test_free_running_loop_is_unchanged(ng):
    import torch
    from lightspinner_b200 import NgOptions
    p, _ = load_golden('c2v_jitter_cah_0')
    res = []
    for with_rays in (False, True):
        eng = make_engine(p, arith=None, ng=NgOptions() if ng else None)
        eng.upload_device_phi([p])
        eng.reset_iteration_state()
        eng.iterate_async(7)
        if with_rays:
            eng.compute_rays_async(MU_NEW)
        eng.iterate_async(400)
        torch.cuda.synchronize()
        res.append((eng.t_iter.cpu().numpy().copy(), eng.n(0), eng.J(0), eng.I(0)))
        eng.close()
    print('ng=%s: %d iterations with and without a compute_rays call between the chunks' % (ng, res[0][0][0]))
    for a, b in zip(res[0], res[1]):
        assert np.array_equal(a, b)


# ---------------------------------------------------------------------------------------------------- 5. invariance
BATCH = ['c2_falc_cah', 'c2v_jitter_cah_0', 'c2v_jitter_cah_1', 'c2v_jitter_cah_0', 'c2_falc_cah', 'c2v_jitter_cah_1',
         'c2v_jitter_cah_0']


def test_batch_and_column_ranges_bitwise():
    probs = [load_golden(n)[0] for n in BATCH]
    eng = make_engine(probs[0], len(probs), arith=None)
    eng.upload_device_phi(probs)
    advance(eng, 6)
    full = eng.compute_rays(MU_NEW)
    for c0, nc in ((0, 2), (2, 3), (5, 2), (6, 1), (1, 5)):
        assert np.array_equal(eng.compute_rays(MU_NEW, c0, nc), full[c0:c0 + nc]), (c0, nc)
    for c in (0, 3, 6):
        one = make_engine(probs[c], arith=None)
        one.upload_device_phi([probs[c]])
        advance(one, 6)
        assert np.array_equal(one.compute_rays(MU_NEW)[0], full[c]), c
        one.close()
    print('7-column batch: equal to column ranges and single-column engines, %d values' % full.size)


RAY_MODELS = [('c1_falc_ca', [2]), ('c1_falc_ca', [0, 4]), ('c1_falc_ca', [0, 2, 4]), ('c1_falc_ca', None),
              ('stress_r10_d512', None)]


@pytest.mark.parametrize('name,rays', RAY_MODELS)
def test_angle_counts_and_chunks(name, rays):
    p, _ = load_golden(name)
    if rays is not None:
        p = select_rays(p, rays)
    R = int(p['Nrays'])
    eng = make_engine(p)
    eng.upload_device_phi([p])
    advance(eng, 5)
    rng = np.random.default_rng(R)
    pool = np.concatenate([[1.0], 1.0 - rng.random(63)])
    for nmu in sorted({1, R, R + 1, 64}):
        mus = pool[:nmu]
        got = eng.compute_rays(mus)
        assert got.shape == (1, int(p['Nspect']), nmu)
        singles = np.concatenate([eng.compute_rays(m) for m in mus], axis=2)
        rev = eng.compute_rays(mus[::-1])[:, :, ::-1]
        assert np.array_equal(got, singles), nmu
        assert np.array_equal(got, rev), nmu
    check_self_consistency(eng, p, '%s with %d rays' % (name, R))
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
        out.append(eng.compute_rays(MU_NEW + list(np.asarray(p['muz']))))
        assert not eng.t_status.cpu().numpy().any()
        eng.close()
    assert np.array_equal(out[0], out[1])


# ---------------------------------------------------------------------------------------------------- 6. Python API
def test_context_after_the_test_py_loop(oracle):
    from lightspinner_b200 import Context
    p, _ = load_golden('c1_falc_ca')
    atmos, spect, eqPops, bg = fake_reference_objects(p)
    ctx = Context(atmos, spect, eqPops, bg)
    dJ, dPops, it = 1.0, 1.0, 0
    while dJ > 2e-3 or dPops > 1e-3:                # test.py:20-29
        it += 1
        dJ = ctx.formal_sol_gamma_matrices()
        if it > 3:
            dPops = ctx.stat_equil()
    I_before = ctx.I.copy()
    r = ctx.compute_rays([1.0, 0.5])
    assert r.shape == (int(p['Nspect']), 2)
    assert np.array_equal(r, ctx._engine.compute_rays([1.0, 0.5], 0, 1)[0])
    assert np.array_equal(ctx.compute_rays(0.5), r[:, 1:])
    assert np.array_equal(ctx.I, I_before)          # cached results stay valid
    # edits through the eqPops alias are honoured
    n = ctx.activeAtoms[0].n
    n[1] *= 1.05
    r2 = ctx.compute_rays([1.0, 0.5])
    ref = reference_rays(p, n, ctx.J, [1.0, 0.5])
    e = rel(r2, ref)
    print('Context after %d iterations: edited populations, compute_rays vs oracle %.3e' % (it, e))
    assert not np.array_equal(r2, r) and e <= TOL_I
    ctx.close()


def test_batch_context_rows_and_long_lists():
    from lightspinner_b200 import BatchContext
    cols = [fake_reference_objects(load_golden(n)[0]) for n in ('c2_falc_cah', 'c2v_jitter_cah_0', 'c2v_jitter_cah_1')]
    batch = BatchContext(cols)
    batch.iterate()
    B = batch.compute_rays(MU_NEW)
    assert B.shape == (3, batch[0]._engine.mt.Nspect, len(MU_NEW))
    for k in range(3):
        assert np.array_equal(B[k], batch[k].compute_rays(MU_NEW))
    mus = np.linspace(0.01, 1.0, 100)
    L = batch._engine.compute_rays(mus)
    assert L.shape[2] == 100
    parts = np.concatenate([batch._engine.compute_rays(mus[a:b]) for a, b in ((0, 30), (30, 64), (64, 100))], axis=2)
    assert np.array_equal(L, parts)
    batch.close()


# ---------------------------------------------------------------------------------------------------- 7. errors
def test_c_entry_point_rejects_bad_arguments():
    import ctypes as C
    import torch
    from lightspinner_b200 import _capi
    p, _ = load_golden('c1_falc_ca')
    eng = make_engine(p)
    eng.upload_device_phi([p])
    L, h, b = eng.lib, eng._handle, C.byref(eng.bufs)
    S = int(p['Nspect'])
    out = torch.zeros(S * 64, dtype=torch.float64, device=eng.device)
    P = lambda t: C.c_void_p(t.data_ptr())
    prof = [P(eng.t_aDamp), P(eng.t_vBroad), P(eng.t_vlos)]

    def call(col0=0, ncol=1, mus=(1.0,), nmu=None, prof_=None, I=None, handle=None):
        m = np.asarray(mus, dtype=np.float64)
        mp = m.ctypes.data_as(C.POINTER(C.c_double)) if m.size else None
        return L.mali_compute_rays(handle or h, b, col0, ncol, len(m) if nmu is None else nmu, mp,
                                   *(prof_ or prof), P(out) if I is None else I, None, eng._stream())

    assert call() == 0
    bad = [dict(col0=-1), dict(ncol=0), dict(ncol=2), dict(col0=1), dict(mus=()), dict(mus=[0.5] * 65),
           dict(mus=[0.0]), dict(mus=[-0.2]), dict(mus=[1.5]), dict(mus=[float('nan')]), dict(mus=[float('inf')]),
           dict(mus=[0.5, 0.0]), dict(I=C.c_void_p(0)), dict(prof_=[None, prof[1], prof[2]]),
           dict(prof_=[prof[0], prof[1], None])]
    for kw in bad:
        assert call(**kw) == MALI_EINVAL, kw
        print('MALI_EINVAL for %s: %s' % (kw, L.mali_last_error().decode()))
    # a model created without lambda0 cannot form line profiles
    desc = eng.mt.desc()
    desc.lambda0 = None
    h2 = C.c_void_p()
    _capi.check(L.mali_model_create(C.byref(desc), eng.device.index, C.byref(h2)), L)
    assert call(handle=h2) == MALI_EINVAL
    assert b'lambda0' in L.mali_last_error()
    L.mali_model_destroy(h2)
    eng.close()


def test_python_layer_errors():
    import torch
    p, _ = load_golden('c1_falc_ca')
    eng = make_engine(p, 3)
    eng.upload_device_phi([p, p])
    for bad in (0.0, 1.5, float('nan'), [], [[0.5]]):
        with pytest.raises(ValueError):
            eng.compute_rays(bad)
    with pytest.raises(ValueError):
        eng.compute_rays(0.5, 2, 2)
    # column 2 was never given profile inputs; columns uploaded with host profiles lose theirs
    with pytest.raises(ValueError, match=r'\[2\]'):
        eng.compute_rays(0.5)
    hp = eng.hostpack_size()
    from lightspinner_b200.tables import pack_column
    pinned = torch.empty(hp, dtype=torch.float64, pin_memory=True)
    pack_column(eng.mt, eng.lay, p, out=pinned.numpy())
    eng.upload_packed(pinned, 1, 1)
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match=r'\[1\]'):
        eng.compute_rays(0.5, 0, 2)
    assert eng.compute_rays(0.5, 0, 1).shape == (1, int(p['Nspect']), 1)
    # upload() of dicts that carry the inputs keeps them
    eng.upload([p], col0=2)
    assert eng.compute_rays([1.0], 2, 1).shape == (1, int(p['Nspect']), 1)
    eng.close()
