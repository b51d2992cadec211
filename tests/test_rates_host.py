"""compute_rates on the CPU: the oracle construction of its definition (tests/rates_reference.py) against two things it
must satisfy.  (1) The J identity: the rates restated with the J of the oracle's own next formal solution.  (2) At the
fixed point of the MALI iteration the PsiStar terms cancel, so the populations solve the plain statistical-equilibrium
equations built from these rates.  No GPU needed."""
import numpy as np
import pytest

from helpers import load_golden
from rates_reference import reference_rates, se_residual, wla

# Residual of the plain equations on c1_falc_ca: 4.5e-4 at the test.py tolerances (46 iterations), 1.3e-8 at
# tolJ = tolPops = 1e-9 (126 iterations).  What is left at the tight point is of the order of the remaining iteration
# change times the PsiStar terms; the bar sits a factor ~4 above that measurement.
SE_BAR = 5e-8


def oracle_state(oracle, p, k):
    oc = oracle.OracleContext(p)
    for it in range(1, k + 1):                     # the loop of test.py:20-29
        oc.formal_sol_gamma_matrices()
        if it > 3:
            oc.stat_equil(use_scipy=False)
    return oc


def converge(oracle, p, tol):
    oc = oracle.OracleContext(p)
    dJ, dP, it = 1.0, 1.0, 0
    while dJ > tol[0] or dP > tol[1]:
        it += 1
        dJ = oc.formal_sol_gamma_matrices()
        if it > 3:
            dP = oc.stat_equil(use_scipy=False)
        assert it < 1000
    return oc, it


def j_identity(oc, J):
    """(Rij, Rji, mask) from the identity R_ij = 4 pi sum_la wla V_ij J, R_ji = 4 pi sum_la wla (U_ji + V_ji J), with
    U, V of angle 0, direction 0; mask[t] says whether it holds for t (continua; lines only where vlos = 0)."""
    k, N = oc._keep, oc.N
    static = not np.any(np.asarray(oc.p['vlos']))
    Rij, Rji = np.zeros((oc.Ntrans, N)), np.zeros((oc.Ntrans, N))
    mask = np.zeros(oc.Ntrans, bool)
    for t in range(oc.Ntrans):
        atom, i, j, isLine, Nblue, Nlam = (int(x) for x in oc.trans[t])
        if isLine and not static:
            continue
        mask[t] = True
        for la in range(Nblue, Nblue + Nlam):
            gij = np.full(N, k['lineconst'][t, 2]) if isLine else k['gijcont'][k['toff'][t] + la - Nblue]
            U, Vij, Vji = oc.uv(t, la, 0, 0, gij)
            w = wla(oc, t, la) * 4 * np.pi
            Rij[t] += w * Vij * J[la]
            Rji[t] += w * (U + Vji * J[la])
    return Rij, Rji, mask


def rel(a, b):
    nz = b != 0
    assert np.array_equal(a == 0, b == 0)
    return float(np.max(np.abs(a[nz] - b[nz]) / np.abs(b[nz]))) if nz.any() else 0.0


@pytest.mark.parametrize('name', ['c1_falc_ca', 'c2v_jitter_cah_0'])
def test_j_identity(oracle, name):
    p, _ = load_golden(name)
    oc = oracle_state(oracle, p, 6)
    n, Jdag = oc.n.copy(), oc.J.copy()
    Rij, Rji = reference_rates(p, n, Jdag)
    assert np.all(Rij >= 0) and np.all(Rji >= 0) and np.all(np.isfinite(Rij)) and np.all(np.isfinite(Rji))
    oc.formal_sol_gamma_matrices()                 # its J is the angle integral of the I the rates integrate
    Iij, Iji, mask = j_identity(oc, oc.J)
    lines = np.asarray(p['trans'])[:, 3] != 0
    e_cont = max(rel(Rij[~lines], Iij[~lines]), rel(Rji[~lines], Iji[~lines]))
    e_line = max(rel(Rij[mask & lines], Iij[mask & lines]), rel(Rji[mask & lines], Iji[mask & lines])) \
        if (mask & lines).any() else float('nan')
    print('%s: J identity after 6 iterations: continua %.3e, lines %s' % (name, e_cont, '%.3e' % e_line
                                                                          if (mask & lines).any() else 'n/a (vlos != 0)'))
    assert e_cont <= 1e-13
    if (mask & lines).any():
        assert e_line <= 1e-13


def test_statistical_equilibrium_at_the_fixed_point(oracle):
    p, _ = load_golden('c1_falc_ca')
    res = {}
    for tol in ((2e-3, 1e-3), (1e-9, 1e-9)):
        oc, it = converge(oracle, p, tol)
        Rij, Rji = reference_rates(p, oc.n, oc.J)
        res[tol] = (se_residual(p, oc.n, Rij, Rji), it)
        print('c1_falc_ca, tolJ %g tolPops %g: %d iterations, plain statistical-equilibrium residual %.3e'
              % (tol[0], tol[1], it, res[tol][0]))
    loose, tight = res[(2e-3, 1e-3)][0], res[(1e-9, 1e-9)][0]
    assert tight < loose * 1e-3
    assert tight <= SE_BAR
