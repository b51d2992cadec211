"""GPU parity on the derived models of tests/model_shapes.py: many-level atoms (12 and 16 levels), 3, 4, 5 and 10
atoms, tiles with up to 40 transitions, launches that mix specialised and generic tiles, and model-specific kernel
instances built at run time.  No committed fixture reaches these shapes; the checker is the C oracle (general in the
atom and level counts, pinned to the reference on the fixtures).

Lock-step runs feed both sides the oracle's populations every iteration, so that errors do not compound.  The bars on
J, I, Gamma and dJ are those of tests/test_gpu_parity.py.  The bar on n is max(1e-9, 10 x the population floor):
the largest difference between two correct solvers (the oracle's LU and scipy's LAPACK) on the same Gamma, measured
in the same run (tests/test_model_shapes_host.py prints it): these systems reach cond ~ 1e11."""
import functools
import os
import warnings

import numpy as np
import pytest

import model_shapes as ms
from helpers import load_golden, load_setup_inputs, only_transitions, relerr

pytestmark = pytest.mark.gpu

TOL_G = 1e-11
TOL_FINAL = 1e-10
SPEC_MODELS = ['c1x2', 'c2x2', 'merged12']       # models that also run on a model-specific library (nvcc at run time)


@functools.lru_cache(maxsize=None)
def model(name):
    return ms.build(name)


def gamma_err(G, Gref):
    scale = np.max(np.abs(Gref), axis=1, keepdims=True)
    scale[scale == 0] = 1.0
    return float(np.max(np.abs(G - Gref) / scale))


def engine(q, path, arith=None, ncol=1):
    """MaliEngine on one of three paths: the stock library ('stock'), every tile on the generic kernel ('nospec'),
    or a model-specific library built for q ('specialize')."""
    from lightspinner_b200.engine import MaliEngine
    if path == 'nospec':
        os.environ['MALI_NO_SPEC'] = '1'
    try:
        with warnings.catch_warnings():
            warnings.simplefilter('ignore', RuntimeWarning)     # the generic-fallback notice
            return MaliEngine(q, ncol, arith=arith, specialize=(path == 'specialize'))
    finally:
        os.environ.pop('MALI_NO_SPEC', None)


def expected_tiles(q, path):
    """(spec_tiles, generic_tiles) the library must report, from the Python structure keys."""
    from lightspinner_b200 import specialize
    keys = specialize.tile_structures(q)
    ntile = -(-int(q['Nspect']) // (32 // int(q['Nrays'])))
    if path == 'nospec':
        nspec = 0
    elif path == 'specialize':
        nspec = len(keys)
    else:
        stock = set(specialize.stock_keys())
        nspec = sum(k in stock for k in keys)
    return nspec, ntile - nspec


def lockstep(eng, oracle, q, niter):
    oc = oracle.OracleContext(q)
    worst = dict(J=0.0, I=0.0, G=0.0, dJ=0.0, n=0.0, floor=0.0)
    for it in range(1, niter + 1):
        eng.set_n(0, oc.n)
        dJ = float(eng.formal_sol_gamma_matrices()[0])
        dJo = oc.formal_sol_gamma_matrices()
        worst['dJ'] = max(worst['dJ'], abs(dJ - dJo) / max(1.0, abs(dJo)))
        worst['J'] = max(worst['J'], relerr(eng.J(0), oc.J))
        worst['I'] = max(worst['I'], relerr(eng.I(0), oc.I))
        worst['G'] = max(worst['G'], gamma_err(eng.Gamma(0), oc.Gamma))
        if it > 3:
            eng.stat_equil()
            worst['floor'] = max(worst['floor'], ms.stat_equil_both(oc))
            worst['n'] = max(worst['n'], relerr(eng.n(0), oc.n))
    return worst


PATHS = [(nm, 'stock') for nm in ms.MODELS] + [(nm, 'nospec') for nm in ms.MODELS] + \
        [(nm, 'specialize') for nm in SPEC_MODELS]


@pytest.mark.parametrize('arith', ['exact', 'contracted'])
@pytest.mark.parametrize('name,path', PATHS)
def test_lockstep_parity(oracle, name, path, arith):
    """Per-call parity over 6 iterations, and the tile counts of model_info(): a structure key that differs between
    specialize.tile_structures and the library's structure_key() fails here instead of slowing the model down."""
    q = model(name)
    eng = engine(q, path, arith)
    info = eng.model_info()
    eng.upload([q])
    w = lockstep(eng, oracle, q, 6)
    eng.close()
    tol_ji = 1e-13 if arith == 'exact' else 1e-12
    tol_n = max(1e-9, 10 * w['floor'])
    print('%s %s %s: J %.1e I %.1e Gamma %.1e dJ %.1e n %.1e (bar %.1e)  tiles %d spec / %d generic, max slots %d, '
          'smem/warp %d B' % (name, path, arith, w['J'], w['I'], w['G'], w['dJ'], w['n'], tol_n, info['spec_tiles'],
                              info['generic_tiles'], info['max_slots'], info['smem_per_warp']))
    assert (info['spec_tiles'], info['generic_tiles']) == expected_tiles(q, path), info
    if path == 'specialize':
        assert info['generic_tiles'] == {'c1x2': 2, 'c2x2': 36, 'merged12': 2}[name]
    assert w['J'] < tol_ji and w['I'] < tol_ji and w['G'] < TOL_G and w['dJ'] < 1e-11, w
    assert w['n'] < tol_n, w


@pytest.mark.parametrize('name', ms.MODELS)
def test_rate_and_particle_conservation(name):
    """Every column of every atom's Gamma sums to zero (rh_method.py:698-703); after stat_equil each atom's
    populations sum to its nTotal, and an atom of one level holds exactly nTotal."""
    q = model(name)
    eng = engine(q, 'stock')
    eng.upload([q])
    N = int(q['Nspace'])
    NL = [int(x) for x in q['Nlevel']]
    nTotal = np.asarray(q['nTotal'])
    for it in range(1, 7):
        eng.formal_sol_gamma_matrices()
        for a in range(len(NL)):
            G = eng.atom_Gamma(0, a)
            assert np.max(np.abs(G.sum(axis=0))) <= 1e-9 * np.max(np.abs(G)), (name, it, a)
        if it > 3:
            eng.stat_equil()
            for a in range(len(NL)):
                n = eng.atom_n(0, a)
                assert np.all(n > 0)
                assert relerr(n.sum(axis=0), nTotal[a]) < 1e-12, (name, it, a)
                if NL[a] == 1:
                    assert np.array_equal(n[0], nTotal[a]), (name, a)
    assert eng.n(0).shape == (sum(NL), N)
    eng.close()


@functools.lru_cache(maxsize=None)
def oracle_free_run(oracle, name):
    """The reference's loop (test.py:20-29) on the oracle with scipy's solve: (iterations, dJ/dPops history, n, J, I)."""
    oc = oracle.OracleContext(model(name))
    dJ, dPops, i, hist = 1.0, 1.0, 0, []
    while (dJ > 2e-3 or dPops > 1e-3) and i < 200:
        i += 1
        dJ = oc.formal_sol_gamma_matrices()
        if i > 3:
            dPops = oc.stat_equil(use_scipy=True)
        hist.append((dJ, dPops))
    return i, np.array(hist), oc.n.copy(), oc.J.copy(), oc.I.copy()


@pytest.mark.parametrize('loop', ['host', 'device'])
@pytest.mark.parametrize('arith', ['exact', 'contracted'])
@pytest.mark.parametrize('name', ['merged12', 'merged16'])
def test_many_level_atom_free_running(oracle, name, arith, loop):
    """A 12- and a 16-level atom iterated to convergence by the host loop and by mali_iterate: the oracle's iteration
    count, its dJ / dPops history to rtol 1e-6 (host loop), final n, J and I within 1e-10."""
    niter, hist_o, n_o, J_o, I_o = oracle_free_run(oracle, name)
    q = model(name)
    eng = engine(q, 'stock', arith)
    eng.upload([q])
    if loop == 'host':
        dJ, dPops, i, hist = 1.0, 1.0, 0, []
        while (dJ > 2e-3 or dPops > 1e-3) and i < 200:
            i += 1
            dJ = float(eng.formal_sol_gamma_matrices()[0])
            if i > 3:
                dPops = float(eng.stat_equil()[0])
            hist.append((dJ, dPops))
        assert i == niter, (i, niter)
        # rtol 1e-6 as in test_c1_free_running_to_convergence, plus an absolute 1e-13: dJ = max |1 - J_old / J_new| is
        # formed from J's that agree to ~1e-15, and with the populations held over iterations 1-3 dJ of iteration 4 is
        # ~1e-10 on these models -- there one ulp of J moves dJ by 2e-6 of itself
        hist = np.array(hist)
        e_hist = np.abs(hist - hist_o) / np.abs(hist_o)
        print('%s %s history: largest relative difference dJ %.1e dPops %.1e' % ((name, arith) + tuple(e_hist.max(0))))
        assert np.all(np.abs(hist - hist_o) <= 1e-6 * np.abs(hist_o) + 1e-13), np.column_stack([hist, hist_o, e_hist])
    else:
        eng.reset_iteration_state()
        eng.iterate_async(60)
        eng.raise_on_faults()
        assert int(eng.t_iter.cpu()[0]) == niter and int(eng.t_done.cpu()[0]) == 1
    e = (relerr(eng.n(0), n_o), relerr(eng.J(0), J_o), relerr(eng.I(0), I_o))
    print('%s %s %s loop: %d iterations, final n %.1e J %.1e I %.1e' % ((name, arith, loop, niter) + e))
    assert max(e) < TOL_FINAL, e
    eng.close()


@pytest.mark.parametrize('name', ['c2x2', 'merged12'])
def test_device_loop_and_batch_bitwise(name):
    """On the model-specific library (a launch that mixes specialised and generic tiles; the 16-level solve inside the
    captured iteration graph): mali_iterate equals the host loop bit for bit, and a batch of 3 jittered columns
    equals the 3 single-column runs bit for bit."""
    from lightspinner_b200 import synth
    q = model(name)
    cols = [synth.jitter_problem(q, c) for c in range(3)]
    niter = 8

    def result(eng, c):
        return eng.J(c), eng.I(c), eng.Gamma(c), eng.n(c)

    singles = []
    for p in cols:
        eng = engine(q, 'specialize')
        info = eng.model_info()
        assert info['spec_tiles'] > 0 and info['generic_tiles'] > 0, info
        eng.upload([p])
        for i in range(1, niter + 1):
            eng.formal_sol_gamma_matrices()
            if i > 3:
                eng.stat_equil()
        singles.append(result(eng, 0))
        eng.close()
    eng = engine(q, 'specialize', ncol=3)
    eng.upload(cols)
    eng.reset_iteration_state()
    eng.iterate_async(niter, tolJ=-1.0)
    eng.raise_on_faults()
    assert eng.t_iter.cpu().tolist() == [niter] * 3
    assert eng.graph_iterations() == niter
    for c in range(3):
        for a, b in zip(singles[c], result(eng, c)):
            assert np.array_equal(a, b), (name, c)
    assert not np.array_equal(singles[0][3], singles[1][3])     # the columns do differ
    eng.close()


def test_device_setup_with_replicated_atoms(oracle):
    """LTE populations, collisional rates and Doppler widths formed on the device for 4 atoms (H, CaII and copies of
    both with a tenth of the abundance) against oracle/setup_oracle.py; the whole column table against a host upload
    of those values (the line profiles, formed on the device too, carry the Voigt function's 1e-12)."""
    from lightspinner_b200.atoms import AtomTables
    from oracle import setup_oracle as so
    q = dict(model('c2x2'))
    atoms, col = load_setup_inputs('c2_falc_cah')
    names = [str(s).strip().rstrip("'").upper() for s in q['atom_names']]
    assert names == ['H', 'CA', 'H', 'CA']
    T, ne, N = np.asarray(q['temperature']), col['ne'], int(q['Nspace'])
    nStar, C, vB = [], [], []
    for a, nm in enumerate(names):
        A = atoms[nm]
        ns = so.lte_pops(A['E_SI'], A['g'], A['stage'], T, ne, np.asarray(q['nTotal'][a]))
        nStar.append(ns)
        C.append(so.compute_collisions(A['E_SI'], A['g'], A['coll'], A['coll_T'], A['coll_rates'], T, ne,
                                       ns).reshape(-1, N))
        vB.append(so.v_broad(A['weight'], T, q['vturb']))
    q['ne'] = ne
    q['nStar'] = q['n'] = np.concatenate(nStar)
    q['C'] = np.concatenate(C)
    q['vBroad'] = np.stack(vB)
    at = AtomTables.from_arrays([dict(atoms[nm]) for nm in names])
    ref = engine(q, 'stock')
    ref.upload([q])
    want = ref.t_colconst.cpu().numpy().copy()
    ref.close()
    eng = engine(q, 'stock')
    eng.set_atoms(at)
    eng.upload_atmos([q])
    got = eng.t_colconst.cpu().numpy()
    e_ns = relerr(eng.nStar.cpu().numpy().reshape(-1, N), q['nStar'])
    e_vb = relerr(eng._last_vBroad.cpu().numpy()[0], q['vBroad'])
    nz = want != 0
    e_all = float(np.max(np.abs(got[nz] - want[nz]) / np.abs(want[nz])))
    eng.close()
    # C alone, through Gamma of a model without radiative transitions (Gamma = C off the diagonal)
    q0 = only_transitions(q, [])
    eng = engine(q0, 'stock')
    eng.set_atoms(at)
    eng.upload_atmos([q0])
    eng.formal_sol_gamma_matrices()
    e_C = 0.0
    for a in range(4):
        off = ~np.eye(6, dtype=bool)
        e_C = max(e_C, relerr(eng.atom_Gamma(0, a)[off], C[a].reshape(6, 6, N)[off]))
    eng.close()
    print('4 atoms: nStar %.1e  vBroad %.1e  C %.1e  column table %.1e' % (e_ns, e_vb, e_C, e_all))
    assert e_ns < 1e-13 and e_vb < 1e-13 and e_C < 1e-13
    assert np.array_equal(got[~nz], want[~nz])
    assert e_all < 1e-12


def test_limits_are_reported_not_crashed():
    """17 levels and 33 rays are refused with a MaliError that says why."""
    from lightspinner_b200 import _capi
    from lightspinner_b200.engine import MaliEngine
    p, _ = load_golden('c1_falc_ca')
    ca = ms.atom_blocks(p)[0]
    q17 = ms.assemble(p, [ms.merge([ca, ms.scaled(ca, 0.1), ms.scaled(ms.sub_atom(ca, range(5), 'CA'), 0.05)], 'CA')])
    assert q17['Nlevel'].tolist() == [17]
    with pytest.raises(_capi.MaliError, match=r'Nlevel=17 not in \[1, 16\]'):
        MaliEngine(q17, 1)
    q33 = dict(p)
    q33['Nrays'] = 33
    q33['muz'] = np.linspace(0.03, 1.0, 33)
    q33['wmu'] = np.full(33, 1.0 / 33)
    with pytest.raises(_capi.MaliError, match=r'Nrays=33 not in \[1, 32\]'):
        MaliEngine(q33, 1)
