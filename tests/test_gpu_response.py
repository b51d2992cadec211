"""MaliEngine.compute_response and mali_perturb_columns on the device (definition in include/mali_b200.h).

- Set-up identity: a column cloned from the set-up base and re-formed at one depth holds bit for bit what the full
  set-up (upload_thermo) forms from the host-built perturbed problem (lightspinner_b200.response.perturbed_problem).
- End-to-end identity against the hand-built batch (host problems -> upload_thermo -> the device loop), reference
  parity against the two response-function fixtures the unmodified reference produced, invariance under the
  workspace, the depth order, the column range and the checked build, the angles, a physics check and the errors.
CaII / FALC from its thermodynamic state: the recipe of test_gpu_background.py (eos.npz, setup_inputs.npz)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from helpers import load_golden, load_setup_inputs
from lightspinner_b200.response import perturbed_problem

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
STEP = {'temperature': 25.0, 'vturb': 500.0, 'vlos': 1000.0}


def engine(p, ncol, library=None, arith=None, ng=None, eos=True, atoms=True):
    from lightspinner_b200.atoms import AtomTables
    from lightspinner_b200.engine import MaliEngine
    from lightspinner_b200.eos import EosTables
    z = np.load(os.path.join(HERE, 'golden', 'eos.npz'))
    at, _ = load_setup_inputs('c1_falc_ca')
    eng = MaliEngine(p, ncol, library=library, arith=arith, ng=ng)
    if eos:
        eng.set_eos(EosTables.from_arrays(z))
    if atoms:
        eng.set_atoms(AtomTables.from_arrays([dict(at['CA'])]))
    return eng


def c1_base(depth_scale='cmass'):
    p, r = load_golden('c1_falc_ca')
    z = np.load(os.path.join(HERE, 'golden', 'eos.npz'))
    at, _ = load_setup_inputs('c1_falc_ca')
    q = {k: p[k] for k in ('vturb', 'vlos', 'aDamp')}
    q['temperature'], q['ne'], q['nHTot'] = z['falc_T'], z['falc_ne'], z['falc_nHTot']
    q['nTotal'] = (at['CA']['abundance'] * q['nHTot'])[None, :]
    if depth_scale == 'cmass':
        q['cmass'] = z['falc_cmass']
    else:
        q['height'] = z['falc_height']
    return p, r, q


def damping(q):
    """Stand-ins for the damping of the shifted atmospheres: the base's, scaled (only the rows of the perturbed depths
    are read)."""
    a = np.asarray(q['aDamp'], dtype=np.float64)
    return a * (1.0 - 1e-3), a * (1.0 + 2e-3)


# ------------------------------------------------------------------------------------------------ set-up identity
@pytest.mark.parametrize('depth_scale', ['cmass', 'height'])
@pytest.mark.parametrize('param', ['temperature', 'vturb', 'vlos'])
def test_perturbed_setup_is_the_full_setup(param, depth_scale):
    from lightspinner_b200.response import base_arrays
    p, r, q = c1_base(depth_scale)
    N = int(p['Nspace'])
    adm, adp = damping(q)
    cols = [(k, s) for k in (0, 1, 10, 40, N - 2, N - 1) for s in (-1, 1)]
    M = len(cols)
    eng = engine(p, 1 + 2 * M)
    b = base_arrays(q, N, 1, eng.mt.Ntrans)
    eng.upload_thermo([b], 0)
    src_work = eng._last_work
    pops0 = torch.as_tensor(r['final_n'], dtype=torch.float64, device=eng.device).reshape(-1)
    eng.t_J.fill_(1.0)          # what an earlier solve left: the call must zero J
    eng.t_pops.fill_(2.0)
    eng._perturb_chunk(b, param, STEP[param], cols, adm, adp, 0, src_work, pops0, 1)
    probs = []
    for k, s in cols:
        pq = perturbed_problem(b, param, STEP[param], k, s, adm, adp)
        pq['n'] = r['final_n']
        probs.append(pq)
    eng.upload_thermo(probs, 1 + M, start_from_lte=False)
    torch.cuda.synchronize()
    L = eng.lay
    SN = int(L.sumNlevel) * N

    def rows(t, per, c0):
        return t[c0 * per:(c0 + M) * per].cpu().numpy().reshape(M, per)

    for name, t, per in (('colconst', eng.t_colconst, L.colconst), ('pops', eng.t_pops, L.pops), ('J', eng.t_J, L.J),
                         ('nStar', eng.nStar, SN)):
        got, want = rows(t, per, 1), rows(t, per, 1 + M)
        bad = [cols[c] for c in range(M) if not np.array_equal(got[c], want[c])]
        assert not bad, '%s differs for columns (k, s) %s' % (name, bad)
    for name, t in (('aDamp', eng.t_aDamp), ('vBroad', eng.t_vBroad), ('vlos', eng.t_vlos)):
        assert np.array_equal(t[1:1 + M].cpu().numpy(), t[1 + M:].cpu().numpy()), name
    assert eng._has_profile[1:].all()
    # the perturbation is real: every column differs from the source somewhere in its tables
    src = eng.t_colconst[:L.colconst].cpu().numpy()
    got = rows(eng.t_colconst, L.colconst, 1)
    assert all(not np.array_equal(got[c], src) for c in range(M))
    eng.close()


# ------------------------------------------------------------------------------------------------ end to end
def hand_built(p, q, param, depths, adm, adp, mus, arith=None, ng=None):
    """The response function the long way: the base solved by upload_thermo + the device loop, then every perturbed
    column as a host problem -> upload_thermo (warm start) -> the device loop; I, iterations, I0."""
    from lightspinner_b200.response import base_arrays
    N = int(p['Nspace'])
    cols = [(int(k), s) for k in depths for s in (-1, 1)]
    eng = engine(p, len(cols) + 1, arith=arith, ng=ng)
    b = base_arrays(q, N, 1, eng.mt.Ntrans)
    eng.upload_thermo([b], 0)
    eng._solve_range(0, 1, 500, 2e-3, 1e-3)
    I0 = eng.compute_rays(mus, 0, 1)[0] if mus is not None else eng.I(0)
    n = eng.n(0)
    probs = []
    for k, s in cols:
        pq = perturbed_problem(b, param, STEP[param], k, s, adm, adp)
        pq['n'] = n
        probs.append(pq)
    eng.upload_thermo(probs, 1, start_from_lte=False)
    eng._solve_range(1, len(cols), 500, 2e-3, 1e-3)
    I = eng.compute_rays(mus, 1, len(cols)) if mus is not None else np.stack([eng.I(1 + c) for c in range(len(cols))])
    its = eng.t_iter[1:].cpu().numpy()
    eng.close()
    return I.reshape(len(depths), 2, *I.shape[1:]), its.reshape(len(depths), 2), I0


@pytest.mark.parametrize('arith,ng', [('exact', False), ('contracted', False), ('contracted', True)])
def test_compute_response_is_the_hand_built_batch(arith, ng):
    from lightspinner_b200.ng import NgOptions
    p, _, q = c1_base()
    adm, adp = damping(q)
    depths = [0, 10, 40, 80, 81]
    ngo = NgOptions() if ng else None
    eng = engine(p, 7, arith=arith, ng=ngo)
    res = eng.compute_response(q, 'temperature', 25.0, aDamp_minus=adm, aDamp_plus=adp, depths=depths)
    I, its, I0 = hand_built(p, q, 'temperature', depths, adm, adp, None, arith=arith, ng=ngo)
    assert np.array_equal(res.I_minus, I[:, 0]) and np.array_equal(res.I_plus, I[:, 1])
    assert np.array_equal(res.iterations, its) and res.converged.all()
    assert np.array_equal(res.I0, I0) and res.base_converged
    assert np.array_equal(res.rf, (I[:, 1] - I[:, 0]) / 50.0)
    assert res.depths.tolist() == depths and res.mu is None and res.param == 'temperature' and res.step == 25.0
    eng.close()


def test_reference_parity():
    """Columns (40, +25 K) and (10, -25 K) with the fixtures' damping rows: the reference's 5 iterations and its final I
    within 1e-10; the base takes the reference's 46."""
    p, r, q = c1_base()
    g40, r40 = load_golden('rf_k40p')
    g10, r10 = load_golden('rf_k10m')
    adm, adp = np.array(q['aDamp']), np.array(q['aDamp'])
    adp[:, 40] = g40['aDamp'][:, 40]
    adm[:, 10] = g10['aDamp'][:, 10]
    eng = engine(p, 6)
    res = eng.compute_response(q, 'temperature', 25.0, aDamp_minus=adm, aDamp_plus=adp, depths=[10, 40])
    assert res.base_iterations == int(r['niter'])
    assert res.iterations[1, 1] == int(r40['niter']) == 5 and res.iterations[0, 0] == int(r10['niter']) == 5
    e40 = np.max(np.abs(res.I_plus[1] - r40['final_I']) / np.abs(r40['final_I']))
    e10 = np.max(np.abs(res.I_minus[0] - r10['final_I']) / np.abs(r10['final_I']))
    print('rel err I: (40, +) %.2e  (10, -) %.2e' % (e40, e10))
    assert e40 < 1e-10 and e10 < 1e-10
    eng.close()


def test_invariance():
    """Bit-identical across workspace sizes (3, 7, all), depth subsets and orders, col0 != 0 and the checked build."""
    from lightspinner_b200.build import CHECK_LIB
    p, _, q = c1_base()
    adm, adp = damping(q)
    N = int(p['Nspace'])
    full = [81, 0, 40, 3, 80, 12]
    runs = []
    for ncol, col0, depths, lib in ((3, 0, full, None), (7, 0, full, None), (14, 0, full, None), (9, 2, full[::-1], None),
                                    (5, 1, [40, 3], None), (7, 0, full, CHECK_LIB)):
        eng = engine(p, col0 + ncol + 1, library=lib)
        res = eng.compute_response(q, 'vturb', STEP['vturb'], aDamp_minus=adm, aDamp_plus=adp, depths=depths,
                                   col0=col0, ncol=ncol, mus=[1.0, 0.5])
        runs.append({int(k): (res.I_minus[i], res.I_plus[i], tuple(res.iterations[i])) for i, k in enumerate(depths)})
        runs[-1]['I0'] = res.I0
        eng.close()
    ref = runs[0]
    for run in runs[1:]:
        for k, v in run.items():
            if k == 'I0':
                assert np.array_equal(v, ref['I0'])
            else:
                assert np.array_equal(v[0], ref[k][0]) and np.array_equal(v[1], ref[k][1]) and v[2] == ref[k][2], k
    assert N - 1 in ref


@pytest.mark.parametrize('param', ['vturb', 'vlos'])
def test_angles_are_compute_rays_of_each_column(param):
    p, _, q = c1_base()
    adm, adp = damping(q)
    mus = np.concatenate([[1.0], p['muz'], [0.3]])
    depths = [2, 41, 81]
    eng = engine(p, 4)
    res = eng.compute_response(q, param, STEP[param], aDamp_minus=adm, aDamp_plus=adp, depths=depths, mus=mus)
    I, its, I0 = hand_built(p, q, param, depths, adm, adp, mus)
    assert np.array_equal(res.I_minus, I[:, 0]) and np.array_equal(res.I_plus, I[:, 1])
    assert np.array_equal(res.I0, I0) and np.array_equal(res.iterations, its)
    assert np.array_equal(res.mu, mus) and res.rf.shape == (3, int(p['Nspect']), mus.shape[0])
    eng.close()


def test_temperature_response_peaks_near_tau_one():
    """In a continuum window the temperature RF at mu = 1 peaks within a few depth points of tau_mu = 1."""
    p, _, q = c1_base()
    adm, adp = damping(q)
    trans = np.asarray(p['trans']).reshape(-1, 6)
    S = int(p['Nspect'])
    inline = np.zeros(S, dtype=bool)
    for t in trans:
        if t[3]:
            inline[t[4]:t[4] + t[5]] = True
    la = int(np.nonzero(~inline)[0][-1])           # 500 nm
    assert p['wavelength'][la] == 500.0
    eng = engine(p, 2 + 2 * int(p['Nspace']))
    res = eng.compute_response(q, 'temperature', 25.0, aDamp_minus=adm, aDamp_plus=adp, mus=[1.0])
    d = eng.compute_rays_depth([1.0], col0=1, ncol=1, quantities=('tau',))
    tau = d.tau[0, :, la, 0]
    k1 = int(np.argmax(tau >= 1.0))
    kmax = int(np.argmax(res.rf[:, la, 0]))
    print('wavelength %.3f nm: RF peak at k=%d, tau=1 at k=%d' % (p['wavelength'][la], kmax, k1))
    assert abs(kmax - k1) <= 3
    assert res.converged.all()
    eng.close()


# ------------------------------------------------------------------------------------------------ errors
def test_value_errors():
    p, _, q = c1_base()
    adm, adp = damping(q)
    eng = engine(p, 4)
    bad = [
        (dict(param='pressure'), 'param'),
        (dict(step=0.0), 'step'),
        (dict(step=float('nan')), 'step'),
        (dict(depths=[82]), 'depths'),
        (dict(depths=[3, 3]), 'unique'),
        (dict(aDamp_minus=None), 'aDamp_minus'),
        (dict(aDamp_plus=adp[:, :5]), 'aDamp_plus'),
        (dict(ncol=2), 'at least 3'),
        (dict(col0=2, ncol=3), 'outside'),
        (dict(max_iter=0), 'max_iter'),
        (dict(mus=[1.5]), 'mu'),
        (dict(base={k: v for k, v in q.items() if k != 'nHTot'}), 'nHTot'),
    ]
    for kw, what in bad:
        args = dict(base=q, param='temperature', step=25.0, aDamp_minus=adm, aDamp_plus=adp, depths=[1])
        args.update(kw)
        with pytest.raises(ValueError, match=what):
            eng.compute_response(args.pop('base'), args.pop('param'), args.pop('step'), **args)
    eng.close()
    for missing in ('eos', 'atoms'):
        e2 = engine(p, 3, **{missing: False})
        with pytest.raises(ValueError, match='set_eos'):
            e2.compute_response(q, 'vlos', 100.0, depths=[1])
        e2.close()


def test_c_abi_rejects_bad_arguments():
    from lightspinner_b200 import _capi
    from lightspinner_b200.response import base_arrays
    p, r, q = c1_base()
    eng = engine(p, 4)
    N = int(p['Nspace'])
    b = base_arrays(q, N, 1, eng.mt.Ntrans)
    eng.upload_thermo([b], 0)
    f64 = dict(dtype=torch.float64, device=eng.device)
    x = {k: torch.as_tensor(b[k], **f64).reshape(1, N).repeat(2, 1).contiguous()
         for k in ('temperature', 'ne', 'nHTot', 'vturb', 'vlos', 'cmass')}
    aD = torch.as_tensor(b['aDamp'], **f64).reshape(1, -1, N).repeat(2, 1, 1).contiguous()
    SN = int(eng.lay.sumNlevel) * N
    nStar, vBroad, work = torch.empty(2 * SN, **f64), torch.empty(2, 1, N, **f64), torch.empty(2 * N * 21, **f64)
    P = lambda t: C.c_void_p(t.data_ptr())
    depth = np.array([3, 7], dtype=np.int32)

    def desc(**over):
        d = dict(T=P(x['temperature']), ne=P(x['ne']), nHTot=P(x['nHTot']), vturb=P(x['vturb']), vlos=P(x['vlos']),
                 cmass=P(x['cmass']), aDamp=P(aD), bbc=None, pops0=P(eng.t_pops[:eng.lay.pops]), src_work=P(eng._last_work),
                 src_nStar=P(eng.nStar[:SN]), src_vBroad=P(eng.t_vBroad[0]), work=P(work), nStar=P(nStar),
                 vBroad=P(vBroad))
        d.update(over)
        dd = _capi.PerturbDesc(**{k: v for k, v in d.items() if k != 'depth'})
        dd.depth = over.get('depth', depth).ctypes.data_as(C.POINTER(C.c_int32))
        return dd

    def call(src, c0, nc, d, e=eng):
        return e.lib.mali_perturb_columns(e._handle, C.byref(e.bufs), src, c0, nc, C.byref(d), e._stream())

    keep = depth
    assert call(0, 1, 2, desc()) == 0
    torch.cuda.synchronize()
    EINVAL = -1
    assert call(0, 3, 2, desc()) == EINVAL                 # range past the batch
    assert call(0, 1, 0, desc()) == EINVAL                 # empty range
    assert call(1, 1, 2, desc()) == EINVAL                 # source inside the range
    assert call(4, 1, 2, desc()) == EINVAL                 # source outside the batch
    assert call(-1, 1, 2, desc()) == EINVAL
    for bad in ([3, N], [-1, 2]):
        d = desc(depth=np.array(bad, dtype=np.int32))
        assert call(0, 1, 2, d) == EINVAL
        assert b'depth' in eng.lib.mali_last_error()
    for k in ('T', 'ne', 'nHTot', 'vturb', 'vlos', 'aDamp', 'pops0', 'src_work', 'src_nStar', 'src_vBroad', 'work',
              'nStar', 'vBroad'):
        assert call(0, 1, 2, desc(**{k: None})) == EINVAL, k
    nd = desc()
    nd.depth = C.POINTER(C.c_int32)()
    assert call(0, 1, 2, nd) == EINVAL
    assert call(0, 1, 2, desc(cmass=None, bbc=None)) == 0     # the optional pointers
    torch.cuda.synchronize()
    for missing in ('eos', 'atoms'):
        e2 = engine(p, 3, **{missing: False})
        assert call(0, 1, 2, desc(), e=e2) == EINVAL
        assert b'mali_model_set_eos' in e2.lib.mali_last_error()
        e2.close()
    del keep
    eng.close()
