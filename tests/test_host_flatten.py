"""Host-side logic of the drop-in Context (no GPU): the mirror of the reference's per-Context set-up (damping
parameters and Doppler widths asked of the model objects, collisions rh_method.py:474-487, activity ranges :122-127)
and the flattening / host-pack layout must reproduce what the reference computed, bit for bit.  The line profiles
themselves (rh_method.py:198-243) are formed on the device; tests/test_gpu_device_phi.py checks them."""
import numpy as np
import pytest

from helpers import fake_reference_objects, load_golden, select_rays

KEYS = ['wavelength', 'muz', 'wmu', 'Nlevel', 'trans', 'linepar', 'alpha', 'height', 'temperature', 'bg_chi', 'bg_eta',
        'bg_sca', 'nStar', 'nTotal', 'C', 'n', 'aDamp', 'vBroad', 'vlos']


@pytest.mark.parametrize('name', ['c1_falc_ca', 'c2_falc_cah', 'c1v_jitter_ca3', 'rf_k40p'])
def test_context_flattening_reproduces_reference_arrays(name):
    """Drive lightspinner_b200.Context's host mirror with fixture-backed stand-ins of the reference objects."""
    from lightspinner_b200.context import Context
    p, r = load_golden(name)
    atmos, spect, eqPops, bg = fake_reference_objects(p)
    ctx = Context(atmos, spect, eqPops, bg, _host_only=True)
    q = ctx._problem
    for k in KEYS:
        assert np.array_equal(np.asarray(q[k]), np.asarray(p[k])), (name, k)
    # aliasing contract of rh_method.py:411-416
    for atom in ctx.activeAtoms:
        assert eqPops[atom.atomicModel.name].pops is atom.n
    with pytest.raises(Exception):
        ctx.formal_sol_gamma_matrices()      # no engine: the host-only object cannot compute (no CPU fallback)


def test_model_tables_match_oracle_tables(oracle):
    from lightspinner_b200 import tables
    for name in ['c1_falc_ca', 'c2_falc_cah']:
        p, r = load_golden(name)
        mt = tables.ModelTables(p)
        ot = oracle.model_tables(p)
        assert np.array_equal(mt.lineconst, ot['lineconst'])
        assert np.array_equal(mt.wlambda, ot['wlambda'])
        assert np.array_equal(mt.twohc_l3, ot['twohc_l3'])
        assert np.array_equal(mt.wlacont, ot['wlacont'])
        g = tables.gij_continuum(mt, p['nStar'], p['temperature'])
        og = oracle.column_tables(p)['gijcont']
        rows = np.concatenate([np.arange(ot['toff'][t], ot['toff'][t + 1]) for t in range(mt.Ntrans)
                               if not p['trans'][t, 3]])
        assert np.array_equal(g, og[rows])


def test_synthetic_jitter_is_deterministic_and_mild():
    from lightspinner_b200 import synth
    p, r = load_golden('c1_falc_ca')
    a, b = synth.jitter_problem(p, 7), synth.jitter_problem(p, 7)
    assert np.array_equal(a['phi'], b['phi']) and np.array_equal(a['bg_chi'], b['bg_chi'])
    c = synth.jitter_problem(p, 8)
    assert not np.array_equal(a['bg_chi'], c['bg_chi'])
    assert np.all(np.abs(np.log(a['bg_chi'] / p['bg_chi'])) < 0.25)


def _recorded_reference_objects(p):
    """fake_reference_objects(p) whose model objects check each call the drop-in makes against the call the
    reference's Context made when the fixture was recorded (tests/golden/make_golden.py stores its hGround, the
    atoms' Doppler widths and LTE populations): v_broad, damping and compute_rates are asked with the
    nondimensionalised atmosphere, damping with the atom's vBroad and the H ground population, compute_rates with the
    atom's nStar and a zeroed C [Nlevel, Nlevel, Nspace].  Each is asked once per model object."""
    atmos, spect, eqPops, bg = fake_reference_objects(p)
    N = int(p['Nspace'])
    lvloff = np.concatenate([[0], np.cumsum(p['Nlevel'])]).astype(int)
    calls = []

    def v_broad(at, atom):
        assert at is atmos and not at.dimensioned
        calls.append(('v_broad', atom.name))
        return atom._vBroad

    def damping(at, vBroad, hGround, line, atom):
        assert at is atmos and not at.dimensioned
        assert np.array_equal(vBroad, atom._vBroad) and np.array_equal(hGround, p['hGround'])
        calls.append(('damping', id(line)))
        return line._aDamp, None

    def compute_rates(at, nStar, C, coll, a):
        assert at is atmos and not at.dimensioned
        NL = int(p['Nlevel'][a])
        assert np.array_equal(nStar, p['nStar'][lvloff[a]:lvloff[a + 1]])
        assert C.shape == (NL, NL, N) and not C.any()
        calls.append(('compute_rates', a))
        C += coll._C

    for a, atom in enumerate(spect.radSet.activeAtoms):
        atom.v_broad = lambda at, atom=atom: v_broad(at, atom)
        for line in atom.lines:
            line.damping = lambda at, vB, hG, line=line, atom=atom: damping(at, vB, hG, line, atom)
        for coll in atom.collisions:
            coll.compute_rates = lambda at, nStar, C, coll=coll, a=a: compute_rates(at, nStar, C, coll, a)
    return (atmos, spect, eqPops, bg), calls


def test_context_host_mirror_against_live_reference():
    """The drop-in fed stand-ins of the reference's model objects that answer, and expect, what the reference's own
    objects answered and were asked when the fixtures were recorded: it must ask each object the same question and
    flatten the answers to exactly what the reference's Context held (C, Nblue, damping parameters, ...)."""
    from lightspinner_b200.context import Context
    for name in ['c1_falc_ca', 'c2_falc_cah', 'c1v_jitter_ca3', 'rf_k40p']:
        p, _ = load_golden(name)
        (atmos, spect, eqPops, bg), calls = _recorded_reference_objects(p)
        ctx = Context(atmos, spect, eqPops, bg, _host_only=True)
        natom = len(p['Nlevel'])
        nline = int(np.asarray(p['trans'])[:, 3].sum())
        assert sorted(c[0] for c in calls) == sorted(['v_broad'] * natom + ['damping'] * nline + ['compute_rates'] * natom)
        assert len(set(calls)) == len(calls), name
        for k in KEYS:
            assert np.array_equal(np.asarray(ctx._problem[k]), np.asarray(p[k])), (name, k)


def test_stock_kernel_instances_cover_the_fixture_models():
    """tools/gen_spec_instances.py and mali_api.cu must agree on the structure keys: every tile of the fixture
    models has an ahead-of-time instance (the GPU twin checks model_info()['generic_tiles'] == 0)."""
    from lightspinner_b200 import specialize
    have = set(specialize.stock_keys())
    assert len(have) >= 40
    for name in ['c1_falc_ca', 'c2_falc_cah', 'c1v_jitter_ca3', 'rf_k40p']:
        p, _ = load_golden(name)
        assert set(specialize.tile_structures(p)) <= have, name
        assert specialize.library_for(p) is None


def test_batch_context_rejects_columns_of_different_models():
    """BatchContext checks, before touching the GPU, that its columns share one radiative model."""
    from lightspinner_b200.context import BatchContext
    p, _ = load_golden('c1_falc_ca')
    q = select_rays(p, [0, 2, 4])
    with pytest.raises(ValueError, match='share'):
        BatchContext([fake_reference_objects(p), fake_reference_objects(q)])
    with pytest.raises(ValueError):
        BatchContext([])


def test_atom_and_eos_tables_from_live_reference_objects():
    """The model-level tables of the device-side set-up built from stand-ins of the reference's objects
    (AtomTables.from_models: atomic models with levels and collision terms, and the atomic table; EosTables.from_witt:
    a witt instance) equal the ones built from the committed fixtures (tests/golden/setup_inputs.npz, eos.npz) --
    the path a user of the reference takes and the path the GPU tests take are the same data.  The stand-ins carry
    the attributes the reference's objects held when the fixtures were recorded, under the reference's names."""
    import os
    from types import SimpleNamespace as NS
    from helpers import GOLDEN, load_setup_inputs
    from lightspinner_b200.atoms import AtomTables
    from lightspinner_b200.eos import NCONTR, EosTables
    atoms, _ = load_setup_inputs('c2_falc_cah')
    kinds = [type(nm, (), {}) for nm in ('Omega', 'CI', 'CE')]     # collisional_rates.py's class names

    def model(name, a):
        levels = [NS(E_SI=e, g=g, stage=st) for e, g, st in zip(a['E_SI'], a['g'], a['stage'])]
        colls, o = [], 0
        for kind, i, j, n in a['coll']:
            c = kinds[kind]()
            c.i, c.j, c.temperature, c.rates = int(i), int(j), a['coll_T'][o:o + n], a['coll_rates'][o:o + n]
            colls.append(c)
            o += n
        return NS(name=name, levels=levels, collisions=colls)

    models = [model('H', atoms['H']), model('CA', atoms['CA'])]
    table = {'H': NS(weight=atoms['H']['weight']), 'CA': NS(weight=atoms['CA']['weight'])}
    live = AtomTables.from_models(models, table)
    fix = AtomTables.from_arrays([dict(atoms['H']), dict(atoms['CA'])])
    for k in ('Nlevel', 'dE', 'gi0', 'dZ', 'nDebye', 'g', 'vTherm', 'coll', 'knots', 'coef', 'fill', 'par'):
        assert np.array_equal(getattr(live, k), getattr(fix, k)), k
    assert live.c1 == fix.c1 and live.c2 == fix.c2
    z = np.load(os.path.join(GOLDEN, 'eos.npz'))
    off = z['stage_off']
    el = [NS(pf=z['pf'][off[i]:off[i + 1]], eion=z['eion'][off[i]:off[i + 1]], nstage=int(off[i + 1] - off[i]))
          for i in range(NCONTR)]
    witt = NS(el=el, tpf=z['tpf'], ABUND=z['ABUND'], avw=float(z['avw']), rho_from_H=float(z['rho_from_H']),
              ab_others=float(z['ab_others']), prec=1.e-5)
    e_live = EosTables.from_witt(witt, float(z['weightPerH']))
    e_fix = EosTables.from_arrays(z)
    for k in ('tpf', 'pf', 'eion', 'stage_off'):
        assert np.array_equal(getattr(e_live, k), getattr(e_fix, k)), k
    assert np.allclose(e_live.abund, e_fix.abund, rtol=1e-14, atol=0)
    for k in ('avw', 'rho_from_H', 'ab_others', 'saha_fac', 'amu_wph', 'cm3', 'thomson'):
        assert abs(getattr(e_live, k) / getattr(e_fix, k) - 1.0) < 1e-14, k
