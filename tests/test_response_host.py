"""compute_response on the CPU: the host builder of the perturbed columns (lightspinner_b200.response, the reference the
device path is tested against) and the argument checks.  The builder must reproduce exactly what the unmodified
reference changed for the two response-function fixtures (tests/golden/rf_k40p.npz: T[40] + 25 K, rf_k10m.npz: T[10] -
25 K, both CaII/FALC).  No GPU needed."""
import os

import numpy as np
import pytest

from helpers import load_golden, load_setup_inputs
from lightspinner_b200.response import (RESPONSE_PARAMS, base_arrays, perturbed_bbc, perturbed_problem, response_args)

HERE = os.path.dirname(os.path.abspath(__file__))


def c1_base():
    """CaII/FALC in upload_thermo form, the column test_gpu_background.py solves from its thermodynamic state."""
    p, _ = load_golden('c1_falc_ca')
    z = np.load(os.path.join(HERE, 'golden', 'eos.npz'))
    atoms, _ = load_setup_inputs('c1_falc_ca')
    q = {k: p[k] for k in ('vturb', 'vlos', 'aDamp')}
    q['temperature'], q['ne'], q['nHTot'], q['cmass'] = (z['falc_%s' % k] for k in ('T', 'ne', 'nHTot', 'cmass'))
    q['nTotal'] = (atoms['CA']['abundance'] * q['nHTot'])[None, :]
    return p, q


@pytest.mark.parametrize('fixture,k,s', [('rf_k40p', 40, 1), ('rf_k10m', 10, -1)])
def test_builder_reproduces_the_reference_columns(fixture, k, s):
    p, base = c1_base()
    g, _ = load_golden(fixture)
    assert np.array_equal(base['temperature'], p['temperature'])
    # the fixture's damping rows stand for the damping of the shifted atmosphere (only row k is used)
    q = perturbed_problem(base, 'temperature', 25.0, k, s, aDamp_minus=g['aDamp'], aDamp_plus=g['aDamp'])
    assert np.array_equal(q['temperature'], g['temperature'])
    assert np.array_equal(q['aDamp'], g['aDamp'])
    for key in ('vturb', 'vlos'):
        assert np.array_equal(q[key], g[key])
    for key in ('ne', 'nHTot', 'cmass', 'nTotal'):
        assert q[key] is base[key]
    assert not np.shares_memory(q['temperature'], base['temperature'])


@pytest.mark.parametrize('param', RESPONSE_PARAMS)
def test_builder_changes_one_entry(param):
    _, base = c1_base()
    N, T = 82, base['aDamp'].shape[0]
    adm, adp = base['aDamp'] * 0.5, base['aDamp'] * 2.0
    for k in (0, 37, N - 1):
        for s in (-1, 1):
            q = perturbed_problem(base, param, 7.5, k, s, aDamp_minus=adm, aDamp_plus=adp)
            d = np.nonzero(q[param] != np.asarray(base[param]))[0]
            assert d.tolist() == [k] and q[param][k] == base[param][k] + s * 7.5
            want = np.array(base['aDamp'])
            if param != 'vlos':
                want[:, k] = (adp if s > 0 else adm)[:, k]
            assert np.array_equal(q['aDamp'], want)
            assert q['aDamp'].shape == (T, N)


def test_boundary_planck_pair_only_for_the_last_two_depths():
    from lightspinner_b200.tables import planck_bc
    p, base = c1_base()
    T, wav = base['temperature'], p['wavelength']
    N = T.shape[0]
    for k in range(N):
        for s in (-1, 1):
            got = perturbed_bbc(wav, T, 'temperature', 25.0, k, s)
            if k < N - 2:
                assert got is None
            else:
                q = perturbed_problem(base, 'temperature', 25.0, k, s, base['aDamp'], base['aDamp'])
                assert np.array_equal(got, planck_bc(wav, q['temperature']))
                assert not np.array_equal(got, planck_bc(wav, T))
    for param in ('vturb', 'vlos'):
        assert perturbed_bbc(wav, T, param, 25.0, N - 1, 1) is None


def test_argument_checks():
    _, base = c1_base()
    N, Nt = 82, base['aDamp'].shape[0]
    ad = base['aDamp']
    step, d, m, pl = response_args('temperature', 25, ad, ad, None, N, Nt)
    assert step == 25.0 and d.dtype == np.int32 and d.tolist() == list(range(N)) and m is not None and pl is not None
    step, d, m, pl = response_args('vlos', 100.0, None, None, [5, 2], N, Nt)
    assert d.tolist() == [5, 2] and m is None and pl is None
    assert response_args('vturb', 1.0, ad, ad, 3, N, Nt)[1].tolist() == [3]
    bad = [
        (('pressure', 1.0, ad, ad, None), 'param'),
        (('temperature', 0.0, ad, ad, None), 'step'),
        (('temperature', -1.0, ad, ad, None), 'step'),
        (('temperature', float('nan'), ad, ad, None), 'step'),
        (('temperature', float('inf'), ad, ad, None), 'step'),
        (('temperature', 'x', ad, ad, None), 'step'),
        (('temperature', 1.0, ad, ad, [0, N]), 'depths'),
        (('temperature', 1.0, ad, ad, [-1]), 'depths'),
        (('temperature', 1.0, ad, ad, [3, 3]), 'unique'),
        (('temperature', 1.0, ad, ad, []), 'depths'),
        (('temperature', 1.0, ad, ad, [1.5]), 'depths'),
        (('temperature', 1.0, None, ad, None), 'aDamp_minus'),
        (('vturb', 1.0, ad, None, None), 'aDamp_plus'),
        (('temperature', 1.0, ad[:, :-1], ad, None), 'aDamp_minus'),
        (('vturb', 1.0, ad, ad[:-1], None), 'aDamp_plus'),
    ]
    for args, what in bad:
        with pytest.raises(ValueError, match=what):
            response_args(*args, N, Nt)
    arrs = base_arrays(base, N, 1, Nt)
    assert arrs['nTotal'].shape == (1, N) and arrs['aDamp'].shape == (Nt, N) and 'height' not in arrs
    with pytest.raises(ValueError, match='cmass'):
        base_arrays({k: v for k, v in base.items() if k != 'cmass'}, N, 1, Nt)
    with pytest.raises(ValueError, match='ne'):
        base_arrays({k: v for k, v in base.items() if k != 'ne'}, N, 1, Nt)
    with pytest.raises(ValueError, match='vturb'):
        base_arrays(dict(base, vturb=base['vturb'][:-1]), N, 1, Nt)
    with pytest.raises(ValueError, match='param'):
        perturbed_problem(base, 'ne', 1.0, 3, 1)
