"""CPU construction of mali_compute_rays_depth's contract (include/mali_b200.h) on the C oracle.

chi and S of the up-going ray at each new angle are rh_method.py:601-632 restated from OracleContext.uv(toFrom=1) on the
problem of rays_reference.with_angles (the line profiles formed at those angles), summed in the oracle's order; I per
depth is the oracle's piecewise_linear_1d on them.  tau, contrib and z_tau1 are the header's formulas, written out
literally with the oracle's w2.  Depth arrays are [Nspace, Nspect, nmu] (depth 0 at the top), as the device returns
one column."""
import numpy as np

from rays_reference import with_angles


def _w2(dtau):
    """The oracle's w2 element by element: (w0, w1) arrays of dtau's shape."""
    from oracle import mali_oracle as O
    d = np.asarray(dtau, dtype=np.float64)
    w = np.array([O.w2(x) for x in d.reshape(-1)]).reshape(d.shape + (2,))
    return w[..., 0], w[..., 1]


def chi_S(oc, la, m):
    """Total opacity and source function [Nspace] of the up-going ray at wavelength la and angle m of `oc` (an
    OracleContext with the current n and J): rh_method.py:601-632 in the oracle's summation order."""
    k, N = oc._keep, oc.N
    chiTot, etaTot = np.zeros(N), np.zeros(N)
    for t in range(oc.Ntrans):
        atom, i, j, isLine, Nblue, Nlam = (int(x) for x in oc.trans[t])
        if not Nblue <= la < Nblue + Nlam:
            continue
        lt = la - Nblue
        gij = np.full(N, k['lineconst'][t, 2]) if isLine else k['gijcont'][k['toff'][t] + lt]
        U, Vij, Vji = oc.uv(t, la, m, 1, gij)
        lo = oc.lvloff[atom]
        ni, nj = oc.n[lo + i], oc.n[lo + j]
        chiTot += ni * Vij - nj * Vji
        etaTot += nj * U
    bg = lambda name: k[name].reshape(oc.Nspect, N)[la]
    chiTot += bg('bg_chi')
    S = (etaTot + bg('bg_eta') + bg('bg_sca') * oc.J[la]) / chiTot
    return chiTot, S


def ray_terms(z, chi, S, I, mus):
    """tau, contrib [N, ...] and z_tau1 [...] from chi, S, I [N, ..., nmu] of up-going rays at the angles `mus` (the
    last axis), by the formulas of include/mali_b200.h: dtau[j] = 0.5*(chi[j]+chi[j+1])*zmu*|z[j]-z[j+1]|, tau summed
    top down, delta[k] = w0*S' + w1*dS (the stale w and S[1] at k = 0), delta[N-1] = I[N-1], T multiplied top down."""
    z = np.asarray(z, dtype=np.float64)
    zmu = 1.0 / np.asarray(mus, dtype=np.float64)
    N = chi.shape[0]
    dtau = [0.5 * (chi[j] + chi[j + 1]) * zmu * np.abs(z[j] - z[j + 1]) for j in range(N - 1)]
    tau = np.zeros_like(chi)
    for k in range(1, N):
        tau[k] = tau[k - 1] + dtau[k - 1]
    delta, a = np.zeros_like(chi), np.zeros_like(chi)
    for k in range(1, N - 1):                          # the step into k
        w0, w1 = _w2(dtau[k])
        dS = (S[k + 1] - S[k]) / dtau[k]
        delta[k] = w0 * S[k] + w1 * dS
        a[k] = 1.0 - w0
    w0, w1 = _w2(dtau[1])                              # k = 0: formal_solver.py:137-139
    dS = (S[1] - S[0]) / dtau[0]
    delta[0] = w0 * S[1] + w1 * dS
    a[0] = 1.0 - w0
    delta[N - 1] = I[N - 1]
    contrib = np.zeros_like(chi)
    T = np.ones_like(chi[0])
    for k in range(N):
        contrib[k] = delta[k] * T
        T = T * a[k]
    return tau, contrib, z_tau1(z, tau)


def z_tau1(z, tau):
    """The height of tau = 1 along each ray of tau [N, ...]: the first k* with tau[k*] >= 1, linear in tau between
    k*-1 and k*; NaN where tau stays below 1."""
    z = np.asarray(z, dtype=np.float64)
    hit = tau >= 1.0
    reached = hit.any(axis=0)
    ks = np.where(reached, np.argmax(hit, axis=0), 1)
    t1 = np.take_along_axis(tau, ks[None], 0)[0]
    t0 = np.take_along_axis(tau, ks[None] - 1, 0)[0]
    z1, z0 = z[ks], z[ks - 1]
    with np.errstate(divide='ignore', invalid='ignore'):
        out = z0 + (z1 - z0) * ((1.0 - t0) / (t1 - t0))
    return np.where(reached, out, np.nan)


def reference_rays_depth(p, n, J, mus):
    """dict of I, chi, S, tau, contrib [Nspace, Nspect, nmu], z_tau1 [Nspect, nmu] and height [Nspace] at the angles
    `mus` from populations n [sumNlevel, Nspace] and J [Nspect, Nspace] (the J-dagger of the sweep)."""
    from oracle import mali_oracle as O
    mus = np.asarray(mus, dtype=np.float64).reshape(-1)
    oc = O.OracleContext(with_angles(p, mus))
    oc.n[...] = np.asarray(n, dtype=np.float64)
    oc.J[...] = np.asarray(J, dtype=np.float64)
    N, Ns, nmu = oc.N, oc.Nspect, mus.shape[0]
    k = oc._keep
    chi, S, I = (np.zeros((N, Ns, nmu)) for _ in range(3))
    for la in range(Ns):
        for m in range(nmu):
            c, s = chi_S(oc, la, m)
            chi[:, la, m], S[:, la, m] = c, s
            I[:, la, m] = O.piecewise_linear_1d(k['height'], k['temperature'], mus[m], 1, k['wavelength'][la], c, s)[0]
    tau, contrib, zt = ray_terms(k['height'], chi, S, I, mus)
    return dict(I=I, chi=chi, S=S, tau=tau, contrib=contrib, z_tau1=zt, height=k['height'].copy())
