"""Ng acceleration on the CPU: the numpy restatement of the step (tests/ng_reference.py) on the C oracle's MALI loop
reproduces the measured iteration counts, converges to the plain loop's fixed point, and NgOptions validates its
parameters.  No GPU needed."""
import numpy as np
import pytest

from ng_reference import cpu_run, ng_step

FIXTURES = [('c1_falc_ca', 46, 29), ('c1v_jitter_ca3', 46, 29), ('c2_falc_cah', 79, 32), ('c2v_jitter_cah_0', 79, 32),
            ('rf_k10m', 5, 5)]


@pytest.mark.parametrize('name,plain,ng', FIXTURES)
def test_iteration_counts_with_default_options(oracle, name, plain, ng):
    a = cpu_run(name)
    b = cpu_run(name, (2, 3, 3))
    print('%s: plain %d, Ng %d, accepted per atom %s' % (name, a.it, b.it, b.accepted.tolist()))
    assert a.it == plain and b.it == ng
    if name == 'rf_k10m':
        assert b.accepted.sum() == 0          # 5 iterations = 2 solves: an extrapolation is never due
        assert np.array_equal(a.oc.n, b.oc.n)


@pytest.mark.parametrize('opts,c1,c2', [((1, 3, 3), 38, 54), ((3, 3, 4), 36, 124), ((2, 5, 5), 25, 31)])
def test_iteration_counts_of_other_settings(oracle, opts, c1, c2):
    assert cpu_run('c1_falc_ca', opts).it == c1
    assert cpu_run('c2_falc_cah', opts).it == c2


def test_order2_period2_does_not_converge_on_c2(oracle):
    """(2, 2, 2) is documented as non-converging on CaII+H/FALC: it is a setting to avoid, not one the options refuse."""
    assert cpu_run('c2_falc_cah', (2, 2, 2), max_iter=400).it == 400


@pytest.mark.parametrize('name', ['c1_falc_ca', 'c2_falc_cah'])
def test_same_fixed_point_at_tight_tolerance(oracle, name):
    a = cpu_run(name, None, 1e-9, 1e-9, 600)
    b = cpu_run(name, (2, 3, 3), 1e-9, 1e-9, 600)
    err = float(np.max(np.abs(b.oc.n / a.oc.n - 1.0)))
    print('%s tight: plain %d, Ng %d iterations, populations differ by %.2e' % (name, a.it, b.it, err))
    assert a.it < 600 and b.it <= 0.5 * a.it
    assert err <= 1e-7


def test_numpy_step_recovers_two_geometric_modes():
    rng = np.random.default_rng(3)
    xs, u, v = 1.0 + rng.random(500), rng.random(500) - 0.5, rng.random(500) - 0.5
    hist = [xs + u * 0.7 ** k + v * 0.4 ** k for k in (3, 2, 1, 0)]     # newest first
    out, ok = ng_step(hist, 2)
    assert ok and np.max(np.abs(out / xs - 1.0)) < 1e-10


@pytest.mark.parametrize('kw', [dict(order=0), dict(order=4), dict(delay=-1), dict(period=0), dict(order=2.0),
                                dict(period=True)])
def test_ng_options_reject_bad_parameters(kw):
    from lightspinner_b200 import NgOptions
    with pytest.raises(ValueError):
        NgOptions(**kw)


def test_ng_options_defaults():
    from lightspinner_b200 import NgOptions
    o = NgOptions()
    assert (o.order, o.delay, o.period) == (2, 3, 3)
    assert [n for n in range(1, 16) if o.due(n)] == [6, 9, 12, 15]
    assert [n for n in range(1, 10) if NgOptions(3, 0, 1).due(n)] == [5, 6, 7, 8, 9]
