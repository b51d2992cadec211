"""compute_rays on the CPU: the oracle construction of its contract (tests/rays_reference.py) reproduces, bit for bit,
the I of the oracle's own next formal solution when it is given the quadrature's angles; and the Python layer validates
the angles.  No GPU needed."""
import numpy as np
import pytest

from helpers import load_golden, recompute_phi
from rays_reference import reference_rays


@pytest.mark.parametrize('name', ['c1_falc_ca', 'c2v_jitter_cah_0'])
def test_reference_rays_is_the_next_formal_solution(oracle, name):
    p, _ = load_golden(name)
    # the construction re-forms the profiles: at the fixture's own angles they must be the fixture's
    phi, wphi = recompute_phi(p)
    lines = np.asarray(p['trans'])[:, 3] != 0
    assert np.array_equal(phi, p['phi'])
    assert np.array_equal(wphi[lines], np.asarray(p['wphi'])[lines])
    oc = oracle.OracleContext(p)
    for it in range(1, 7):                     # the loop of test.py:20-29, 6 iterations
        oc.formal_sol_gamma_matrices()
        if it > 3:
            oc.stat_equil(use_scipy=False)
    got = reference_rays(p, oc.n, oc.J, p['muz'])
    oc.formal_sol_gamma_matrices()
    diff = float(np.max(np.abs(got - oc.I) / np.where(oc.I != 0, np.abs(oc.I), 1.0)))
    print('%s: reference_rays vs the next formal solution after 6 iterations: max rel diff %.3e (%d values)'
          % (name, diff, got.size))
    assert np.array_equal(got, oc.I)


def test_reference_rays_at_new_angles_is_finite_and_positive(oracle):
    p, _ = load_golden('c1_falc_ca')
    mus = [1.0, 0.9, 0.6, 0.33, 0.1, 0.05]
    I = reference_rays(p, p['n'], np.zeros((int(p['Nspect']), int(p['Nspace']))), mus)
    assert I.shape == (int(p['Nspect']), len(mus))
    assert np.all(np.isfinite(I)) and np.all(I > 0)


@pytest.mark.parametrize('bad', [0.0, -0.5, 1.0 + 1e-12, float('nan'), float('inf'), [], [[1.0, 0.5]], [0.5, 0.0]])
def test_angles_are_validated_without_a_gpu(bad):
    from lightspinner_b200.engine import rays_angles
    with pytest.raises(ValueError):
        rays_angles(bad)


def test_scalar_and_list_angles():
    from lightspinner_b200.engine import rays_angles
    a = rays_angles(0.5)
    assert a.shape == (1,) and a.dtype == np.float64 and a[0] == 0.5
    b = rays_angles([1.0, 0.25, 1e-3])
    assert b.shape == (3,) and np.array_equal(b, [1.0, 0.25, 1e-3])
    assert rays_angles(np.float32(1.0))[0] == 1.0
