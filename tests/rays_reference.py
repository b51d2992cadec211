"""CPU construction of mali_compute_rays' contract (include/mali_b200.h) on the C oracle.

The emergent intensity at user angles is what the next formal solution returns as I if those angles were the angles of
its quadrature: a copy of the problem with muz = mus, the line profiles formed at those angles by the reference's own
expressions (helpers.recompute_phi, scipy wofz), the given populations n and mean intensity J (the J-dagger of that
formal solution), one OracleContext.formal_sol_gamma_matrices(), and its I."""
import numpy as np

from helpers import recompute_phi


def with_angles(p, mus):
    """The problem with the angle quadrature replaced by `mus`.  The weights are uniform: I does not depend on them
    (they only enter J and Gamma).  phi / wphi are re-formed and phioff rebuilt for the new angle count (each line's
    profile is [Nlambda][nmu][2][Nspace])."""
    mus = np.asarray(mus, dtype=np.float64).reshape(-1)
    q = dict(p)
    q['Nrays'] = int(mus.shape[0])
    q['muz'] = mus.copy()
    q['wmu'] = np.full(mus.shape[0], 1.0 / mus.shape[0])
    q['phi'], q['wphi'] = recompute_phi(q)
    N = int(p['Nspace'])
    tr = np.asarray(p['trans']).reshape(-1, 6)
    offs, o = [], 0
    for t in range(tr.shape[0]):
        if tr[t, 3]:
            offs.append(o)
            o += int(tr[t, 5]) * q['Nrays'] * 2 * N
        else:
            offs.append(0)
    q['phioff'] = np.array(offs, dtype=np.int64)
    return q


def reference_rays(p, n, J, mus):
    """I [Nspect, nmu] at the angles `mus` from populations n [sumNlevel, Nspace] and J [Nspect, Nspace]."""
    from oracle import mali_oracle as O
    oc = O.OracleContext(with_angles(p, mus))
    oc.n[...] = np.asarray(n, dtype=np.float64)
    oc.J[...] = np.asarray(J, dtype=np.float64)
    oc.formal_sol_gamma_matrices()
    return oc.I.copy()
