"""Models of shapes no committed fixture has, derived from the fixtures by changing only the atomic structure.

Every fixture is CaII (1 atom, 6 levels) or CaII+H (2 atoms of 6 levels), and on the 5-ray grid none of their
wavelength tiles holds more than 8 transitions.  The builders here keep a fixture's atmosphere, background,
wavelength grid and rays, and re-arrange its atoms:

    c1x2      CaII + a copy of CaII with n, nStar, nTotal x 0.1               mixed specialised / generic tiles
    c2x2      CaII+H + a x0.1 copy of both: 4 atoms                          the Natom <= 4 edge of the specialised path
    c1x5      5 copies of CaII, scales 1, .1, .05, .02, .01                  5 atoms: every tile generic
    c2x5      5 copies of CaII+H: 10 atoms                                    up to 40 transitions per tile
    merged12  CaII and its x0.1 copy stacked into ONE 12-level atom           the 16-level statistical-equilibrium solve
    merged16  merged12 plus a third block of CaII's levels 0-3 (x0.05)        Nlevel = 16, the largest accepted
    small     CaII + a 2-level atom (one CaII line) + a 1-level atom          the 2-level solve, the NL = 1 path, an
                                                                              atom no wavelength tile touches

The blocks of a merged atom are coupled by collisions between level l of the first block and the same level of the
others: the rate l -> l' is 1e-2 of level l's collisional out-rate, the reverse rate follows detailed balance on nStar.

The results are problem dicts in the layout tests/helpers.load_golden returns, so MaliEngine, oracle.OracleContext,
tables.ModelTables and specialize.tile_structures take them unchanged.  They are not outputs of the reference: the
checker for them is the C oracle, which is general in the atom and level counts and pinned to the reference on the
fixtures (tests/test_oracle_golden.py)."""
import numpy as np

from helpers import load_golden

COUPLING = 1e-2


def atom_blocks(p):
    """The atoms of problem p, each as a dict of its own arrays (levels local to the atom)."""
    N, R = int(p['Nspace']), int(p['Nrays'])
    Nlevel = np.asarray(p['Nlevel'], dtype=int)
    lvloff = np.concatenate([[0], np.cumsum(Nlevel)])
    g2off = np.concatenate([[0], np.cumsum(Nlevel ** 2)])
    tr = np.asarray(p['trans']).reshape(-1, 6)
    toff = np.concatenate([[0], np.cumsum(tr[:, 5])]).astype(int)
    names = [str(s).strip() for s in p['atom_names']]
    blocks = []
    for a, NL in enumerate(Nlevel):
        trans = []
        for t in np.nonzero(tr[:, 0] == a)[0]:
            isLine, Nlam = int(tr[t, 3]), int(tr[t, 5])
            po = int(p['phioff'][t])
            trans.append(dict(i=int(tr[t, 1]), j=int(tr[t, 2]), isLine=isLine, Nblue=int(tr[t, 4]), Nlam=Nlam,
                              linepar=np.asarray(p['linepar']).reshape(-1, 4)[t],
                              alpha=np.asarray(p['alpha'])[toff[t]:toff[t + 1]],
                              aDamp=np.asarray(p['aDamp'])[t], wphi=np.asarray(p['wphi'])[t],
                              phi=np.asarray(p['phi'])[po:po + Nlam * R * 2 * N] if isLine else None))
        sl = slice(lvloff[a], lvloff[a + 1])
        blocks.append(dict(name=names[a], NL=int(NL), nStar=np.asarray(p['nStar'])[sl], n=np.asarray(p['n'])[sl],
                           nTotal=np.asarray(p['nTotal'])[a], vBroad=np.asarray(p['vBroad'])[a],
                           C=np.asarray(p['C'])[g2off[a]:g2off[a + 1]].reshape(NL, NL, N), trans=trans))
    return blocks


def scaled(b, s, name=None):
    """A copy of atom block b with its populations and abundance scaled by s (rates and profiles unchanged)."""
    q = dict(b)
    q['nStar'], q['n'], q['nTotal'] = b['nStar'] * s, b['n'] * s, b['nTotal'] * s
    q['name'] = name or b['name']
    return q


def sub_atom(b, levels, name):
    """The atom made of the given levels of block b and the transitions among them (populations and rates kept)."""
    levels = list(levels)
    idx = {lv: q for q, lv in enumerate(levels)}
    trans = [dict(t, i=idx[t['i']], j=idx[t['j']]) for t in b['trans'] if t['i'] in idx and t['j'] in idx]
    n = b['n'][levels]
    return dict(name=name, NL=len(levels), nStar=b['nStar'][levels], n=n, nTotal=n.sum(axis=0), vBroad=b['vBroad'],
                C=b['C'][np.ix_(levels, levels)], trans=trans)


def one_level_atom(N, nTotal, vBroad, name):
    nTotal = np.asarray(nTotal, dtype=np.float64)
    return dict(name=name, NL=1, nStar=nTotal[None, :].copy(), n=nTotal[None, :].copy(), nTotal=nTotal,
                vBroad=vBroad, C=np.zeros((1, 1, N)), trans=[])


def merge(blocks, name):
    """One atom holding the levels of every block (block 0 first).  Block b > 0 is coupled to block 0 by collisions
    between its level l and level l of block 0 (see the module docstring)."""
    N = blocks[0]['C'].shape[-1]
    NL = sum(b['NL'] for b in blocks)
    C = np.zeros((NL, NL, N))
    off, trans = [], []
    o = 0
    for b in blocks:
        C[o:o + b['NL'], o:o + b['NL']] = b['C']
        trans += [dict(t, i=t['i'] + o, j=t['j'] + o) for t in b['trans']]
        off.append(o)
        o += b['NL']
    nStar = np.concatenate([b['nStar'] for b in blocks])
    C0 = blocks[0]['C']
    for b, ob in zip(blocks[1:], off[1:]):
        for l in range(b['NL']):
            out = C0[:, l].sum(axis=0) - C0[l, l]           # C[i, j]: rate from j to i
            up = COUPLING * out
            C[ob + l, l] = up                               # l -> its image in block b
            C[l, ob + l] = up * nStar[l] / nStar[ob + l]    # detailed balance on nStar
    return dict(name=name, NL=NL, nStar=nStar, n=np.concatenate([b['n'] for b in blocks]),
                nTotal=sum(b['nTotal'] for b in blocks), vBroad=blocks[0]['vBroad'], C=C, trans=trans)


def assemble(p, blocks):
    """Problem dict with p's atmosphere, background, wavelength grid and rays, and the atoms `blocks`."""
    N, R = int(p['Nspace']), int(p['Nrays'])
    q = {k: p[k] for k in ('Nspace', 'Nrays', 'Nspect', 'wavelength', 'muz', 'wmu', 'height', 'temperature', 'vlos',
                           'vturb', 'hGround', 'bg_chi', 'bg_eta', 'bg_sca') if k in p}
    q['atom_names'] = np.array([b['name'] for b in blocks])
    q['Nlevel'] = np.array([b['NL'] for b in blocks], dtype=np.int32)
    trans, linepar, alpha, aDamp, wphi, phis, phioff = [], [], [], [], [], [], []
    po = 0
    for a, b in enumerate(blocks):
        for t in b['trans']:
            trans.append([a, t['i'], t['j'], t['isLine'], t['Nblue'], t['Nlam']])
            linepar.append(t['linepar'])
            alpha.append(t['alpha'])
            aDamp.append(t['aDamp'])
            wphi.append(t['wphi'])
            if t['isLine']:
                phis.append(t['phi'])
                phioff.append(po)
                po += t['phi'].size
            else:
                phioff.append(0)
    q['trans'] = np.array(trans, dtype=np.int32).reshape(-1, 6)
    q['linepar'] = np.array(linepar, dtype=np.float64).reshape(-1, 4)
    q['alpha'] = np.concatenate(alpha) if alpha else np.zeros(0)
    q['aDamp'] = np.array(aDamp, dtype=np.float64).reshape(-1, N)
    q['wphi'] = np.array(wphi, dtype=np.float64).reshape(-1, N)
    q['phi'] = np.concatenate(phis) if phis else np.zeros(0)
    q['phioff'] = np.array(phioff, dtype=np.int64)
    q['nStar'] = np.ascontiguousarray(np.concatenate([b['nStar'] for b in blocks]))
    q['n'] = np.ascontiguousarray(np.concatenate([b['n'] for b in blocks]))
    q['nTotal'] = np.ascontiguousarray(np.stack([b['nTotal'] for b in blocks]))
    q['vBroad'] = np.ascontiguousarray(np.stack([b['vBroad'] for b in blocks]))
    q['C'] = np.ascontiguousarray(np.concatenate([b['C'].reshape(-1, N) for b in blocks]))
    return q


def replicated(p, scales):
    """All of p's atoms once per scale (copy k after copy k-1), populations and abundances x scale."""
    base = atom_blocks(p)
    return assemble(p, [scaled(b, s, b['name'] + ("'" * k)) for k, s in enumerate(scales) for b in base])


def build(name):
    """The named model (see the module docstring) as a problem dict."""
    if name in ('c1x2', 'c1x5', 'merged12', 'merged16', 'small'):
        p, _ = load_golden('c1_falc_ca')
    else:
        p, _ = load_golden('c2_falc_cah')
    if name in ('c1x2', 'c2x2'):
        return replicated(p, (1.0, 0.1))
    if name in ('c1x5', 'c2x5'):
        return replicated(p, (1.0, 0.1, 0.05, 0.02, 0.01))
    ca = atom_blocks(p)[0]
    if name == 'merged12':
        return assemble(p, [merge([ca, scaled(ca, 0.1)], 'CA')])
    if name == 'merged16':
        return assemble(p, [merge([ca, scaled(ca, 0.1), scaled(sub_atom(ca, range(4), 'CA'), 0.05)], 'CA')])
    if name == 'small':
        two = scaled(sub_atom(ca, [ca['trans'][0]['i'], ca['trans'][0]['j']], 'CA2'), 0.1)
        one = one_level_atom(int(p['Nspace']), 0.01 * ca['nTotal'], ca['vBroad'], 'CA1')
        return assemble(p, [ca, two, one])
    raise KeyError(name)


MODELS = ['c1x2', 'c2x2', 'c1x5', 'c2x5', 'merged12', 'merged16', 'small']


def stat_equil_both(oc):
    """oc.stat_equil with scipy's solve (the reference's call), after solving the same systems with the oracle's own
    LU; returns the largest relative difference of the two -- the population floor of this step."""
    from helpers import relerr
    n0 = oc.n.copy()
    oc.stat_equil(use_scipy=False)
    n_lu = oc.n.copy()
    oc.n[:] = n0
    oc.stat_equil(use_scipy=True)
    return relerr(n_lu, oc.n)
