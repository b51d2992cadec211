"""CPU construction of mali_compute_rates' definition (include/mali_b200.h) on the C oracle.

For every (wavelength, quadrature angle, direction): chi and S from OracleContext.uv in the oracle's summation order
(rh_method.py:601-632, as rays_depth_reference.chi_S, with both directions), I per depth from the oracle's
piecewise_linear_1d, and the Gamma integrands with PsiStar = 0 summed per transition with the oracle's weight
wlamu = wla * hw * 4 * PI (mali_oracle.c).  Rates are [Ntrans, Nspace] for one column."""
import numpy as np


def _uv_all(oc, la, mu, toFrom):
    """[(t, U, Vij, Vji)] of the transitions active at wavelength la, in transition order."""
    k, N = oc._keep, oc.N
    out = []
    for t in range(oc.Ntrans):
        atom, i, j, isLine, Nblue, Nlam = (int(x) for x in oc.trans[t])
        if not Nblue <= la < Nblue + Nlam:
            continue
        gij = np.full(N, k['lineconst'][t, 2]) if isLine else k['gijcont'][k['toff'][t] + la - Nblue]
        out.append((t,) + oc.uv(t, la, mu, toFrom, gij))
    return out


def wla(oc, t, la):
    """The Gamma wavelength weight of transition t at wavelength la [Nspace] (rh_method.py:451-454)."""
    from oracle import mali_oracle as O
    k = oc._keep
    atom, i, j, isLine, Nblue, Nlam = (int(x) for x in oc.trans[t])
    w = k['wlambda'][k['toff'][t] + la - Nblue]
    if isLine:
        return w * k['wphi'][t] / O.HC
    return np.full(oc.N, k['wlacont'][k['toff'][t] + la - Nblue])


def reference_rates(p, n, J):
    """(Rij, Rji) [Ntrans, Nspace] of one column from populations n [sumNlevel, Nspace] and J [Nspect, Nspace] (the
    J-dagger of the sweeps)."""
    from oracle import mali_oracle as O
    oc = O.OracleContext(p)
    oc.n[...] = np.asarray(n, dtype=np.float64)
    oc.J[...] = np.asarray(J, dtype=np.float64)
    k, N = oc._keep, oc.N
    Rij, Rji = np.zeros((oc.Ntrans, N)), np.zeros((oc.Ntrans, N))
    bg = lambda name, la: k[name].reshape(oc.Nspect, N)[la]
    for la in range(oc.Nspect):
        w = {}
        for mu in range(oc.Nrays):
            hw = 0.5 * k['wmu'][mu]
            for toFrom in range(2):
                terms = _uv_all(oc, la, mu, toFrom)
                chiTot, etaTot = np.zeros(N), np.zeros(N)
                for t, U, Vij, Vji in terms:
                    atom, i, j = (int(x) for x in oc.trans[t][:3])
                    lo = oc.lvloff[atom]
                    chiTot += oc.n[lo + i] * Vij - oc.n[lo + j] * Vji
                    etaTot += oc.n[lo + j] * U
                chiTot += bg('bg_chi', la)
                S = (etaTot + bg('bg_eta', la) + bg('bg_sca', la) * oc.J[la]) / chiTot
                I = O.piecewise_linear_1d(k['height'], k['temperature'], k['muz'][mu], toFrom, k['wavelength'][la],
                                          chiTot, S)[0]
                for t, U, Vij, Vji in terms:
                    if t not in w:
                        w[t] = wla(oc, t, la)
                    wlamu = w[t] * hw * 4 * np.pi
                    Rji[t] += (U + Vji * I) * wlamu
                    Rij[t] += (Vij * I) * wlamu
    return Rij, Rji


def rate_matrix(p, Rij, Rji):
    """The plain rate matrix P = C + R [sumNlevel2, Nspace] in Gamma's layout (P[i][j]: the rate from j to i), the
    diagonal formed as gamma_finish_kernel forms it: minus the sum of the column's off-diagonal entries."""
    Nlevel = np.asarray(p['Nlevel'])
    g2off = np.concatenate([[0], np.cumsum(Nlevel.astype(int) ** 2)])
    trans = np.asarray(p['trans']).reshape(-1, 6)
    C = np.asarray(p['C'], dtype=np.float64)
    P = np.array(C, copy=True)
    for t, (atom, i, j, isLine, Nblue, Nlam) in enumerate(trans):
        NL = int(Nlevel[atom])
        P[g2off[atom] + i * NL + j] += Rji[t]
        P[g2off[atom] + j * NL + i] += Rij[t]
    for a, NL in enumerate(Nlevel):
        G = P[g2off[a]:g2off[a + 1]].reshape(NL, NL, -1)
        for i in range(NL):
            G[i, i] = 0.0
        for i in range(NL):
            G[i, i] = -sum(G[l, i] for l in range(NL) if l != i)
    return P


def se_residual(p, n, Rij, Rji):
    """max over atoms and depths of max_i |(P n)_i| / sum_i |P_ii n_i|: how far n is from solving the plain
    statistical-equilibrium equations with the rates Rij, Rji."""
    P = rate_matrix(p, Rij, Rji)
    Nlevel = np.asarray(p['Nlevel'])
    g2off = np.concatenate([[0], np.cumsum(Nlevel.astype(int) ** 2)])
    lvloff = np.concatenate([[0], np.cumsum(Nlevel)])
    n = np.asarray(n, dtype=np.float64)
    worst = 0.0
    for a, NL in enumerate(Nlevel):
        G = P[g2off[a]:g2off[a + 1]].reshape(NL, NL, -1)
        na = n[lvloff[a]:lvloff[a + 1]]
        Pn = np.einsum('ijk,jk->ik', G, na)
        scale = np.sum(np.abs(np.einsum('iik->ik', G) * na), axis=0)
        worst = max(worst, float(np.max(np.max(np.abs(Pn), axis=0) / scale)))
    return worst


def net_rates(p, n, Rij, Rji):
    """n_i Rij - n_j Rji [Ntrans, Nspace]."""
    Nlevel = np.asarray(p['Nlevel'])
    lvloff = np.concatenate([[0], np.cumsum(Nlevel)])
    trans = np.asarray(p['trans']).reshape(-1, 6)
    n = np.asarray(n, dtype=np.float64)
    rowI = lvloff[trans[:, 0]] + trans[:, 1]
    rowJ = lvloff[trans[:, 0]] + trans[:, 2]
    return n[rowI] * Rij - n[rowJ] * Rji
