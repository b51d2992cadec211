"""The derived models of tests/model_shapes.py on the CPU: the builders' invariants, the tile structures the
specialised path will be asked for, and each model's population floor (how far two correct fp64 solvers of the same
statistical-equilibrium systems land apart), from which the GPU population bar of tests/test_gpu_model_shapes.py
is derived."""
import numpy as np
import pytest

import model_shapes as ms

# (largest slots per tile, tiles with > 8 slots, tiles with <= 8 slots) on the 5-ray grid
SLOTS = {'c1x2': (10, 2, 46), 'c2x2': (16, 36, 94), 'c1x5': (25, 24, 24), 'c2x5': (40, 127, 3),
         'merged12': (10, 2, 46), 'merged16': (10, 2, 46), 'small': (5, 0, 48)}


def tile_slots(q):
    tr = np.asarray(q['trans']).reshape(-1, 6)
    Lw, S = 32 // int(q['Nrays']), int(q['Nspect'])
    return np.array([int(((tr[:, 4] < min(S, la0 + Lw)) & (tr[:, 4] + tr[:, 5] > la0)).sum())
                     for la0 in range(0, S, Lw)])


def population_floor(oracle, q, niter=8):
    """Largest relative difference between the oracle's own LU and scipy.linalg.solve on identical Gamma over
    iterations 4..niter (the run continues from scipy's populations, as the reference's would)."""
    oc = oracle.OracleContext(q)
    floor = 0.0
    for it in range(1, niter + 1):
        oc.formal_sol_gamma_matrices()
        if it > 3:
            floor = max(floor, ms.stat_equil_both(oc))
    return floor


@pytest.mark.parametrize('name', ms.MODELS)
def test_builder_invariants(oracle, name):
    from lightspinner_b200.tables import ModelTables
    q = ms.build(name)
    N, R = int(q['Nspace']), int(q['Nrays'])
    mt = ModelTables(q)
    NL = np.asarray(q['Nlevel'], dtype=int)
    assert mt.Natom == len(NL) and q['nStar'].shape == q['n'].shape == (NL.sum(), N)
    assert q['C'].shape == ((NL ** 2).sum(), N) and q['nTotal'].shape == q['vBroad'].shape == (len(NL), N)
    assert np.all(q['n'] > 0) and np.all(q['nStar'] > 0) and np.all(q['C'] >= 0)
    # every line's profile block lies inside phi, the blocks tile phi without gaps or overlaps
    tr = q['trans']
    ends = sorted((int(q['phioff'][t]), int(q['phioff'][t]) + int(tr[t, 5]) * R * 2 * N)
                  for t in range(tr.shape[0]) if tr[t, 3])
    assert ends[0][0] == 0 and ends[-1][1] == q['phi'].size
    assert all(a[1] == b[0] for a, b in zip(ends, ends[1:]))
    # Gamma of one formal solution: columns sum to zero (rh_method.py:698-703); every system solvable both ways
    oc = oracle.OracleContext(q)
    oc.formal_sol_gamma_matrices()
    cond = 0.0
    for a in range(len(NL)):
        G = oc.atom_Gamma(a)
        assert np.max(np.abs(G.sum(axis=0))) <= 1e-12 * max(np.max(np.abs(G)), 1e-300), (name, a)
        n = oc.atom_n(a)
        for k in range(N):
            Gp = G[:, :, k].copy()
            Gp[np.argmax(n[:, k]), :] = 1.0
            cond = max(cond, np.linalg.cond(Gp))
    assert np.isfinite(cond)
    n0 = oc.n.copy()
    oc.stat_equil(use_scipy=False)          # raises LinAlgError on a singular system
    n_lu = oc.n.copy()
    oc.n[:] = n0
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('error')      # scipy's ill-conditioning warning fails the test
        oc.stat_equil(use_scipy=True)
    assert np.all(np.isfinite(n_lu)) and np.all(n_lu > 0) and np.all(oc.n > 0)
    print('%s: Natom %d, Nlevel %s, max cond(Gamma\') %.1e' % (name, len(NL), NL.tolist(), cond))


@pytest.mark.parametrize('name', ms.MODELS)
def test_tile_structures_are_the_specialisable_tiles(name):
    """specialize.tile_structures lists exactly the tiles with <= 8 slots, and none when the model has > 4 atoms."""
    from lightspinner_b200 import specialize
    q = ms.build(name)
    cnt = tile_slots(q)
    assert (cnt.max(), int((cnt > 8).sum()), int((cnt <= 8).sum())) == SLOTS[name]
    keys = specialize.tile_structures(q)
    natom = len(q['Nlevel'])
    assert len(keys) == (int((cnt <= 8).sum()) if natom <= 4 else 0)
    nslot = [int(k[1:].split(',')[1]) for k in keys]
    assert nslot == [int(c) for c in cnt if c <= 8 and natom <= 4]


def test_merged_atoms_couple_their_blocks():
    """The merged atoms: one atom, the collisional coupling obeys detailed balance on nStar."""
    for name, NL in (('merged12', 12), ('merged16', 16)):
        q = ms.build(name)
        assert q['Nlevel'].tolist() == [NL]
        N = int(q['Nspace'])
        C = q['C'].reshape(NL, NL, N)
        nS = q['nStar']
        for l in range(4):
            for lb in range(l + 6, NL, 6):
                assert np.all(C[lb, l] > 0)
                assert np.allclose(nS[l] * C[lb, l], nS[lb] * C[l, lb], rtol=1e-14, atol=0)


@pytest.mark.parametrize('name', ms.MODELS)
def test_population_floor(oracle, name):
    """The floor two correct solvers share; the GPU bar on n is max(1e-9, 10 x floor)."""
    floor = population_floor(oracle, ms.build(name))
    print('%s: population floor %.2e  (GPU n bar %.1e)' % (name, floor, max(1e-9, 10 * floor)))
    assert floor < 1e-8
