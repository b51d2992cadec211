"""Drop-in for the MALI hot path of Lightspinner's rh_method.py, running on a B200 through libmali_b200.so.

    from lightspinner_b200 import Context          # instead of: from rh_method import Context
    ctx = Context(atmos, spect, eqPops, background)   # same objects the reference builds (test.py:8-18)
    dJ = ctx.formal_sol_gamma_matrices()              # rh_method.py:565-708
    dPops = ctx.stat_equil()                          # rh_method.py:710-745
    ctx.I, ctx.J, ctx.activeAtoms[0].n, .Gamma        # same names, shapes and aliasing as the reference
    I = ctx.compute_rays([1.0, 0.5])                  # [Nspect, nmu]: emergent intensity at user angles (Lightweaver)

Only the hot path moves to the GPU.  Everything in this file is the host-side mirror of the reference's per-Context
SET-UP (ComputationalTransition / ComputationalAtom construction, rh_method.py:93-131,366-423,474-487): it asks the
model objects for what only they know (`line.damping`, `atom.v_broad`, `collision.compute_rates`), flattens the
result (lightspinner_b200/tables.py) and uploads it once; the Voigt line profiles (rh_method.py:198-243) are formed on
the GPU from the damping parameters (mali_compute_phi) and the wavelength weights by tables.ModelTables.  The iteration itself never touches the host except for
the two scalars the reference's loop reads (dJ, dPops) and the population write-back that keeps
`eqPops[name].pops is atom.n` true (SURVEY.md 8b).
"""
from dataclasses import dataclass

import numpy as np

from . import tables
from .engine import MaliEngine, piecewise_linear_1d_batch

@dataclass
class UV:
    """Container for the [RH92]/[U01] Uji, Vij and Vji terms (rh_method.py:17-23)."""
    Uji: np.ndarray
    Vij: np.ndarray
    Vji: np.ndarray


def _is_line(trans):
    # reference: isinstance(trans, AtomicLine); lines carry Einstein coefficients, continua a cross-section
    return hasattr(trans, 'Aji') and hasattr(trans, 'lambda0')


class ComputationalTransition:
    """Host-side handle of one radiative transition (rh_method.ComputationalTransition's role): the model constants
    the flattening needs plus views of what lives on the device.  The line profiles are formed on the GPU
    (mali_compute_phi); `phi` / `wphi` read them back on first use, `uv` evaluates on the GPU tables."""

    def __init__(self, trans, compAtom, atmos, spect):
        self.transModel = trans
        self.atom = compAtom
        self.wavelength = trans.wavelength
        self.isLine = _is_line(trans)
        if self.isLine:
            self.Aji, self.Bji, self.Bij, self.lambda0 = trans.Aji, trans.Bji, trans.Bij, trans.lambda0
            # the one per-depth quantity of a line the device needs from the model objects (atomic_model.py:491-502)
            self.aDamp = trans.damping(atmos, compAtom.vBroad, compAtom.hPops.n[0])[0]
        else:
            self.alpha = trans.alpha
            self.aDamp = None
        self.i = trans.i
        self.j = trans.j
        self.Nblue = int(np.searchsorted(spect.wavelength, self.wavelength[0]))     # rh_method.py:122
        Nlam = int(self.wavelength.shape[0])
        self.active = np.zeros(spect.wavelength.shape[0], bool)                     # rh_method.py:125-127
        for la, s in enumerate(spect.activeSet):
            if trans in s:
                self.active[la] = True
        self.gij = None
        self.Rij = np.zeros(atmos.Nspace)    # dead outputs of the reference (never zeroed, never read): not maintained
        self.Rji = np.zeros(atmos.Nspace)
        self.index = None                    # position in the flattened transition table
        self._profile = None
        del Nlam

    def lt(self, la):
        return la - self.Nblue

    def wlambda(self, la=None):
        """Wavelength quadrature weights (rh_method.py:157-196), from the model tables the device uses."""
        mt = self.atom.ctx._engine.mt
        w = mt.wlambda[mt.toff[self.index]:mt.toff[self.index + 1]]
        return np.array(w) if la is None else float(w[la])

    def _line_profile(self):
        if self._profile is None:
            self._profile = self.atom.ctx._engine.line_profile(self.atom.ctx._col, self.index)
        return self._profile

    @property
    def phi(self):
        """[Nlambda, Nrays, 2, Nspace] (rh_method.py:224), read back from the device tables on first use."""
        return self._line_profile()[0] if self.isLine else None

    @property
    def wphi(self):
        return self._line_profile()[1] if self.isLine else None

    def uv(self, la, mu, toFrom):
        """rh_method.py:245-288, evaluated by the GPU from the packed tables (mali_uv)."""
        U, Vij, Vji = self.atom.ctx._engine.uv(self.atom.ctx._col, self.index, int(la), int(mu), bool(toFrom))
        return UV(Uji=U, Vij=Vij, Vji=Vji)


class ComputationalAtom:
    """Host mirror of rh_method.ComputationalAtom: state and set-up (rh_method.py:366-423, 474-487)."""

    def __init__(self, atom, atmos, spect, eqPops, ctx):
        self.ctx = ctx
        self.atomicModel = atom
        self.atomicTable = getattr(eqPops, 'atomicTable', None)
        self.spect = spect
        self.atmos = atmos
        self.vBroad = atom.v_broad(atmos)
        self.pops = eqPops[atom.name]
        self.hPops = eqPops['H']
        self.nTotal = self.pops.nTotal
        self.trans = []
        for l in atom.lines:
            if l in spect.transitions:
                self.trans.append(ComputationalTransition(l, self, atmos, spect))
        for c in atom.continua:
            if c in spect.transitions:
                self.trans.append(ComputationalTransition(c, self, atmos, spect))
        Nlevel = len(atom.levels)
        self.C = np.zeros((Nlevel, Nlevel, atmos.Nspace))
        self.nStar = self.pops.nStar
        if self.pops.pops is not None:          # rh_method.py:411-416: alias, not copy
            self.n = self.pops.pops
        else:
            self.n = np.copy(self.nStar)
            self.pops.pops = self.n
        self.Nlevel = Nlevel
        self.Ntrans = len(self.trans)
        self.index = None

    def compute_collisions(self):
        """rh_method.py:474-487 (iteration-invariant: evaluated once per Context, uploaded with the column)."""
        self.C = np.zeros((self.Nlevel, self.Nlevel, self.atmos.Nspace))
        for col in self.atomicModel.collisions:
            col.compute_rates(self.atmos, self.nStar, self.C)
        self.C[self.C < 0.0] = 0.0

    @property
    def Gamma(self):
        return self.ctx._atom_Gamma(self.index)


class Context:
    """Drop-in for rh_method.Context (rh_method.py:490-745) -- one column on one GPU.

    Batches of columns (response functions, 1.5D runs) go through BatchContext (below) / MaliEngine, which run the
    same kernels over many columns per launch.
    """

    def __init__(self, atmos, spect, eqPops, background, device=None, ng=None, _host_only=False):
        """The Voigt line profiles (ComputationalTransition.compute_phi, rh_method.py:198-243) are formed on the GPU
        from the damping parameters -- same values to ~1e-13 (the accuracy of the scipy wofz the reference calls);
        `trans.phi` / `trans.wphi` are read back from the device if somebody asks for them.
        ng: an NgOptions to accelerate the population iteration of stat_equil() (off by default; the reference has no
        such option, so with it on the iteration count differs from the reference's)."""
        self.atmos = atmos
        self.atmos.nondimensionalise()                                    # rh_method.py:553
        self.spect = spect
        self.background = background
        self.eqPops = eqPops
        self.activeAtoms = []
        for a in spect.radSet.activeAtoms:                                # rh_method.py:558-560
            self.activeAtoms.append(ComputationalAtom(a, atmos, spect, eqPops, self))
        self._problem = flatten_context(self)
        self._cache = {}
        self._engine = None
        self._col = 0       # column of the engine's batch this Context owns (BatchContext hands out others)
        if _host_only:      # unit tests of the host-side flattening only; every compute method then fails
            return
        self._engine = MaliEngine(self._problem, 1, device=device, ng=ng)
        self._engine.upload_device_phi([self._problem])

    # -- lazily fetched results (numpy, C order, the reference's shapes)
    def _get(self, key, fn):
        if key not in self._cache:
            self._cache[key] = fn()
        return self._cache[key]

    @property
    def J(self):
        return self._get('J', lambda: self._engine.J(self._col))

    @property
    def I(self):
        return self._get('I', lambda: self._engine.I(self._col))

    def _atom_Gamma(self, a):
        return self._get(('G', a), lambda: self._engine.atom_Gamma(self._col, a))

    def _push_pops(self):
        # the reference reads atom.n afresh on every call: honour edits made through the eqPops alias
        self._engine.set_n(self._col, np.concatenate([a.n for a in self.activeAtoms], axis=0))

    def formal_sol_gamma_matrices(self):
        """rh_method.py:565-708.  Returns dJ = max |1 - JDag/J| as a float."""
        self._push_pops()
        self._cache = {}
        return float(self._engine.formal_sol_gamma_matrices(self._col, 1)[0])

    def stat_equil(self):
        """rh_method.py:710-745.  Updates every atom.n IN PLACE; raises numpy.linalg.LinAlgError if singular."""
        dPops = float(self._engine.stat_equil(self._col, 1)[0])
        self._pull_pops()
        return dPops

    def compute_rays(self, mus):
        """Emergent intensity [Nspect, nmu] at the angles `mus` (0 < mu <= 1; a scalar gives nmu = 1) from the current
        populations (edits through the eqPops alias included) and the current J -- Lightweaver's Context.compute_rays.
        It is the I the next formal_sol_gamma_matrices() would return if `mus` were the angles of the quadrature
        (the same line profiles, formed on the GPU at these angles); it changes nothing the iteration uses."""
        self._push_pops()
        return self._engine.compute_rays(mus, self._col, 1)[0]

    def ng_reset(self):
        """Restart the Ng history (Context(ng=...)): call it after editing populations between iterations."""
        self._engine.ng_reset(self._col, 1)

    def _pull_pops(self):
        n = self._engine.n(self._col)
        mt = self._engine.mt
        for ia, atom in enumerate(self.activeAtoms):
            atom.n[...] = n[mt.lvloff[ia]:mt.lvloff[ia + 1]]

    def close(self):
        if self._engine is not None and self._col == 0 and not getattr(self, '_borrowed', False):
            self._engine.close()


class BatchContext:
    """Many columns that share one radiative model (same atoms, wavelength grid and angle quadrature) solved in one
    batch -- the response-function / 1.5D use of the reference, which builds one Context per column and iterates
    them one after the other (response_fn.py:23-39).

        batch = BatchContext([(atmos_k, spect, eqPops_k, background_k) for k in columns])
        its = batch.iterate()                       # test.py:20-29 for every column, on the device
        I = batch[k].I ;  n = eqPops_k['Ca'].n      # per-column results through the usual Context attributes

    `batch[k]` is a Context (host mirrors, results, the eqPops alias) bound to column k of the batch; the per-call
    methods of the reference exist in batched form too: formal_sol_gamma_matrices() and stat_equil() return one
    value per column."""

    def __init__(self, columns, device=None, ng=None):
        """ng: an NgOptions to accelerate the population iteration (off by default, see Context)."""
        if not columns:
            raise ValueError('BatchContext needs at least one column')
        self.contexts = [Context(*c, _host_only=True) for c in columns]
        problems = [c._problem for c in self.contexts]
        p0 = problems[0]
        for q in problems[1:]:
            for key in ('Nspace', 'Nrays', 'Nspect'):
                if int(q[key]) != int(p0[key]):
                    raise ValueError('columns of a batch must share %s' % key)
            for key in ('trans', 'wavelength', 'muz', 'wmu', 'Nlevel', 'linepar', 'alpha'):
                if not np.array_equal(np.asarray(q[key]), np.asarray(p0[key])):
                    raise ValueError('columns of a batch must share the radiative model (%s differs)' % key)
        self._engine = MaliEngine(p0, len(problems), device=device, ng=ng)
        self._engine.upload_device_phi(problems)
        for k, c in enumerate(self.contexts):
            c._engine, c._col, c._borrowed = self._engine, k, True

    def __len__(self):
        return len(self.contexts)

    def __getitem__(self, k):
        return self.contexts[k]

    def _invalidate(self):
        for c in self.contexts:
            c._cache = {}

    def formal_sol_gamma_matrices(self):
        """rh_method.py:565-708 for every column: returns dJ[ncol]."""
        for c in self.contexts:
            c._push_pops()
        self._invalidate()
        return np.array(self._engine.formal_sol_gamma_matrices())

    def stat_equil(self):
        """rh_method.py:710-745 for every column: returns dPops[ncol]; every atom.n is updated in place."""
        dPops = np.array(self._engine.stat_equil())
        for c in self.contexts:
            c._pull_pops()
        return dPops

    def compute_rays(self, mus):
        """Context.compute_rays for every column: [ncol, Nspect, nmu]."""
        for c in self.contexts:
            c._push_pops()
        return self._engine.compute_rays(mus)

    def iterate(self, max_iter=500, tolJ=2e-3, tolPops=1e-3):
        """The loop of test.py:20-29 for every column, kept on the device (mali_iterate): returns the iteration
        count of each column (a column stops as soon as it meets the tolerances)."""
        import torch
        for c in self.contexts:
            c._push_pops()
        self._invalidate()
        self._engine.reset_iteration_state()
        done = 0
        while done < max_iter:
            nit = min(16, max_iter - done)
            self._engine.iterate_async(nit, tolJ, tolPops)
            done += nit
            if bool((self._engine.t_done != 0).all().item()):
                break
        torch.cuda.synchronize(self._engine.device)
        for c in self.contexts:
            c._pull_pops()
        self._engine.raise_on_faults()      # LinAlgError / FloatingPointError, as the reference's loop would raise
        return self._engine.t_iter.cpu().numpy().copy()

    def close(self):
        self._engine.close()


def flatten_context(ctx):
    """Reference-layout problem dict (lightspinner_b200/tables.py) from the host mirrors of a Context: everything but
    the line profiles, for which it carries what compute_phi consumes (aDamp, vBroad, vlos)."""
    atmos, spect, bg = ctx.atmos, ctx.spect, ctx.background
    N = atmos.Nspace
    Nlevel, trans, linepar, alpha = [], [], [], []
    nStar, nTotal, Cs, ns = [], [], [], []
    aDamp, vBroad = [], []
    it = 0
    for ia, atom in enumerate(ctx.activeAtoms):
        vBroad.append(np.asarray(atom.vBroad, dtype=np.float64))
        atom.index = ia
        atom.compute_collisions()
        Nlevel.append(atom.Nlevel)
        nStar.append(np.asarray(atom.nStar, dtype=np.float64))
        nTotal.append(np.asarray(atom.nTotal, dtype=np.float64))
        Cs.append(atom.C.reshape(atom.Nlevel * atom.Nlevel, N))
        ns.append(np.asarray(atom.n, dtype=np.float64))
        for t in atom.trans:
            t.index = it
            it += 1
            Nlam = int(t.wavelength.shape[0])
            if not np.array_equal(t.wavelength, spect.wavelength[t.Nblue:t.Nblue + Nlam]):
                raise ValueError('transition wavelength grid is not a slice of the global grid')
            act = np.zeros(spect.wavelength.shape[0], bool)
            act[t.Nblue:t.Nblue + Nlam] = True
            if not np.array_equal(act, t.active):
                raise ValueError('transition is not active on a contiguous wavelength range')
            trans.append([ia, t.i, t.j, int(t.isLine), t.Nblue, Nlam])
            if t.isLine:
                linepar.append([t.Aji, t.Bji, t.Bij, t.lambda0])
                alpha.append(np.zeros(Nlam))
                aDamp.append(np.asarray(t.aDamp, dtype=np.float64))
            else:
                linepar.append([0.0, 0.0, 0.0, 0.0])
                alpha.append(np.asarray(t.alpha, dtype=np.float64))
                aDamp.append(np.zeros(N))
    return dict(
        Nspace=N, Nrays=atmos.Nrays, Nspect=int(spect.wavelength.shape[0]),
        wavelength=np.asarray(spect.wavelength, dtype=np.float64), muz=np.asarray(atmos.muz, dtype=np.float64),
        wmu=np.asarray(atmos.wmu, dtype=np.float64), Nlevel=np.array(Nlevel, dtype=np.int32),
        trans=np.array(trans, dtype=np.int32).reshape(-1, 6), linepar=np.array(linepar).reshape(-1, 4),
        alpha=np.concatenate(alpha) if alpha else np.zeros(0),
        height=np.asarray(atmos.height, dtype=np.float64), temperature=np.asarray(atmos.temperature, dtype=np.float64),
        bg_chi=np.asarray(bg.chi), bg_eta=np.asarray(bg.eta), bg_sca=np.asarray(bg.sca),
        nStar=np.concatenate(nStar, axis=0), nTotal=np.stack(nTotal), C=np.concatenate(Cs, axis=0),
        n=np.concatenate(ns, axis=0),
        aDamp=np.stack(aDamp) if aDamp else np.zeros((0, N)), vBroad=np.stack(vBroad),
        vlos=np.asarray(atmos.vlos, dtype=np.float64))


@dataclass
class IPsi:
    """formal_solver.py:6-12"""
    I: np.ndarray
    PsiStar: np.ndarray


def piecewise_linear_1d(atmos, mu, toFrom, wav, chi, S):
    """formal_solver.piecewise_linear_1d (formal_solver.py:144-212) on the GPU: same signature, same result bits."""
    bbc = tables.planck_bc(np.array([wav], dtype=np.float64), np.asarray(atmos.temperature, dtype=np.float64))
    I, Psi = piecewise_linear_1d_batch(np.asarray(atmos.height, dtype=np.float64), [atmos.muz[mu]], [int(bool(toFrom))],
                                       [bbc[0, 0]], [bbc[0, 1]], np.asarray(chi, dtype=np.float64)[None, :],
                                       np.asarray(S, dtype=np.float64)[None, :])
    return IPsi(I[0], Psi[0])
