"""compute_rays_depth on the CPU: the oracle construction of its contract (tests/rays_depth_reference.py) ends in the
emergent intensity of rays_reference, its contribution function telescopes to that intensity, tau grows with depth, the
k = 0 step carries the reference's stale-w quirk, z_tau1 is NaN where tau = 1 is never reached; and the Python layer
validates its arguments.  No GPU needed."""
import numpy as np
import pytest

from helpers import load_golden
from rays_depth_reference import _w2, ray_terms, reference_rays_depth, z_tau1
from rays_reference import reference_rays

MU = [1.0, 0.6, 0.1]


def state_after_6(oracle, p):
    oc = oracle.OracleContext(p)
    for it in range(1, 7):                     # the loop of test.py:20-29, 6 iterations
        oc.formal_sol_gamma_matrices()
        if it > 3:
            oc.stat_equil(use_scipy=False)
    return oc.n.copy(), oc.J.copy()


@pytest.fixture(scope='module', params=['c1_falc_ca', 'c2v_jitter_cah_0'])
def case(request, oracle):
    p, _ = load_golden(request.param)
    n, J = state_after_6(oracle, p)
    return request.param, p, n, J, reference_rays_depth(p, n, J, MU)


def test_surface_intensity_is_reference_rays(case):
    name, p, n, J, d = case
    ref = reference_rays(p, n, J, MU)
    I0 = d['I'][0]
    e = float(np.max(np.abs(I0 - ref) / np.abs(ref)))
    print('%s: I[0] of the depth construction vs reference_rays: max rel diff %.3e, %d of %d values bit-identical'
          % (name, e, int(np.sum(I0 == ref)), ref.size))
    assert e <= 1e-14
    assert np.array_equal(I0, ref)          # chi and eta are summed in the oracle's order


def test_contributions_telescope_to_the_emergent_intensity(case):
    name, p, n, J, d = case
    c, I0 = d['contrib'], d['I'][0]
    gap = np.abs(c.sum(axis=0) - I0)
    scale = np.abs(c).sum(axis=0)
    print('%s: max |sum contrib - I[0]| / sum |contrib| = %.3e' % (name, float(np.max(gap / scale))))
    assert np.all(gap <= 1e-13 * scale)


def test_tau_starts_at_zero_and_grows(case):
    name, p, n, J, d = case
    tau = d['tau']
    assert np.all(tau[0] == 0.0)
    assert np.all(np.diff(tau, axis=0) >= 0.0)
    # on a plane-parallel atmosphere the optical depth scales as 1 / mu wherever the opacity does not depend on mu
    print('%s: tau at the bottom spans %.3e .. %.3e' % (name, float(tau[-1].min()), float(tau[-1].max())))


def test_k0_step_applies_the_stale_weights(case):
    """I[0] = a[0] I[1] + delta[0] with the w of the step into 1 and S[1] (formal_solver.py:137-139); with the step's own
    w and S[0] the recurrence would not reproduce the sweep's I[0]."""
    name, p, n, J, d = case
    z, chi, S, I = d['height'], d['chi'], d['S'], d['I']
    zmu = 1.0 / np.asarray(MU)
    dtau = [0.5 * (chi[j] + chi[j + 1]) * zmu * np.abs(z[j] - z[j + 1]) for j in (0, 1)]
    w0, w1 = _w2(dtau[1])
    stale = (1.0 - w0) * I[1] + (w0 * S[1] + w1 * (S[1] - S[0]) / dtau[0])
    v0, v1 = _w2(dtau[0])
    fresh = (1.0 - v0) * I[1] + (v0 * S[0] + v1 * (S[1] - S[0]) / dtau[0])
    e_stale = float(np.max(np.abs(stale - I[0]) / np.abs(I[0])))
    e_fresh = float(np.max(np.abs(fresh - I[0]) / np.abs(I[0])))
    print('%s: k = 0 recurrence vs I[0]: stale w %.3e, own w %.3e' % (name, e_stale, e_fresh))
    assert e_stale <= 1e-14 and e_fresh > 1e-10
    # and contrib[0] is that delta (T[0] = 1)
    assert np.array_equal(d['contrib'][0], w0 * S[1] + w1 * ((S[1] - S[0]) / dtau[0]))


def test_z_tau1_is_nan_where_tau_stays_below_one():
    z = np.linspace(2.0e6, -1.0e5, 8)
    tau = np.zeros((8, 3))
    tau[:, 0] = np.linspace(0.0, 0.9, 8)               # never reaches 1
    tau[:, 1] = np.linspace(0.0, 7.7, 8)               # passes 1 between k = 0 and k = 1
    tau[:, 2] = [0.0, 0.2, 0.5, 1.0, 1.0, 2.0, 3.0, 4.0]   # exactly 1 at k = 3
    zt = z_tau1(z, tau)
    assert np.isnan(zt[0])
    assert zt[1] == z[0] + (z[1] - z[0]) * ((1.0 - tau[0, 1]) / (tau[1, 1] - tau[0, 1]))
    assert z[1] < zt[1] < z[0]
    assert zt[2] == z[3]


def test_ray_terms_on_a_synthetic_thin_column():
    """A column too thin to reach tau = 1: z_tau1 is NaN on every ray, and the contributions still telescope."""
    N = 6
    z = np.linspace(1.0e6, 0.0, N)
    chi = np.full((N, 1, 2), 1e-8)
    S = np.linspace(1.0, 2.0, N)[:, None, None] * np.ones((1, 1, 2))
    I = np.zeros_like(chi)
    I[-1] = 3.0
    tau, contrib, zt = ray_terms(z, chi, S, I, [1.0, 0.5])
    assert np.all(np.isnan(zt))
    assert tau[-1, 0, 1] == pytest.approx(2.0 * tau[-1, 0, 0], rel=1e-14)
    assert np.all(tau[-1] < 1.0)


@pytest.mark.parametrize('bad', [['I', 'J'], ['tau', 'tau'], [], 'Z', ['I', None]])
def test_quantities_are_validated_without_a_gpu(bad):
    from lightspinner_b200.engine import rays_depth_quantities
    with pytest.raises(ValueError):
        rays_depth_quantities(bad)


def test_quantity_selection_order():
    from lightspinner_b200 import RayDepthData
    from lightspinner_b200.engine import RAYS_DEPTH_QUANTITIES, rays_depth_quantities
    assert rays_depth_quantities(None) == RAYS_DEPTH_QUANTITIES
    assert RAYS_DEPTH_QUANTITIES == ('I', 'chi', 'S', 'tau', 'contrib', 'z_tau1', 'height')
    assert rays_depth_quantities(['z_tau1', 'I']) == ('I', 'z_tau1')
    assert rays_depth_quantities('contrib') == ('contrib',)
    d = RayDepthData(mu=np.array([1.0]), height=np.zeros((2, 4)), I=np.ones((2, 4, 3, 1)))
    one = d.column(1)
    assert one.height.shape == (4,) and one.I.shape == (4, 3, 1) and one.tau is None
