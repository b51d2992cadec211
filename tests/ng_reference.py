"""CPU restatement of the Ng acceleration (include/mali_b200.h, mali_iterate_ng) on top of the C oracle's MALI loop.

ng_step is the definition, written out in numpy: per column and active atom, x0 the newest solved population vector
(flattened over level, depth), x1, x2, ... the older ones, d_i = x_i - x_{i+1}, w = 1 / x0^2,
    A_ij = sum w (d0 - d_{i+1})(d0 - d_{j+1}),  b_i = sum w d0 (d0 - d_{i+1}),  A c = b,
    x* = (1 - sum c) x0 + sum_i c_i x_{i+1},
accepted only if A is non-singular and x* is finite and > 0 everywhere.  NgLoop drives the oracle through the loop of
test.py:20-29 with that step after every statistical equilibrium that is due."""
import numpy as np

from helpers import load_golden


def ng_step(hist, order):
    """hist: [order + 2] flat vectors, NEWEST FIRST -> (x*, True), or (None, False) when rejected."""
    x = [np.asarray(h, dtype=np.float64) for h in hist[:order + 2]]
    x0 = x[0]
    w = 1.0 / (x0 * x0)
    d = [x[i] - x[i + 1] for i in range(order + 1)]
    A = np.zeros((order, order))
    b = np.zeros(order)
    for i in range(order):
        ei = d[0] - d[i + 1]
        b[i] = np.sum(w * d[0] * ei)
        for j in range(order):
            A[i, j] = np.sum(w * ei * (d[0] - d[j + 1]))
    try:
        c = np.linalg.solve(A, b)
    except np.linalg.LinAlgError:
        return None, False
    out = (1.0 - c.sum()) * x0
    for i in range(order):
        out = out + c[i] * x[i + 1]
    if not (np.all(np.isfinite(out)) and np.all(out > 0)):
        return None, False
    return out, True


def due(nse, order, delay, period):
    return nse > delay and nse >= order + 2 and (nse - delay) % period == 0


class NgLoop:
    """The oracle's MALI loop for one column (its own LU for the statistical equilibrium) with optional Ng steps.

    loop.step() runs one iteration and returns (dJ, dPops); run() iterates to the tolerances.  Attributes: it (iterations
    done), nse, accepted [Natom], solved (every solved vector per atom, oldest first, when record=True)."""

    def __init__(self, problem, ng=None, record=False):
        from oracle import mali_oracle as O
        self.oc = O.OracleContext(problem)
        self.ng = ng                      # (order, delay, period) or None
        self.record = record
        self.it = 0
        self.nse = 0
        self.accepted = np.zeros(self.oc.Natom, dtype=int)
        self.accepted_at = []             # nse of every solve that was followed by at least one accepted step
        R = (ng[0] + 2) if ng else 0
        self.hist = [[] for _ in range(self.oc.Natom)]
        self.R = R
        self.solved = [[] for _ in range(self.oc.Natom)]

    def stat_equil(self):
        oc = self.oc
        n0 = oc.n.copy()
        dP = oc.stat_equil(use_scipy=False)
        self.nse += 1
        for a in range(oc.Natom):
            v = oc.atom_n(a).ravel().copy()
            if self.record:
                self.solved[a].append(v)
            if self.ng:
                self.hist[a] = ([v] + self.hist[a])[:self.R]
        if self.ng and due(self.nse, *self.ng):
            any_acc = False
            for a in range(oc.Natom):
                out, ok = ng_step(self.hist[a], self.ng[0])
                if ok:
                    oc.atom_n(a)[...] = out.reshape(oc.atom_n(a).shape)
                    self.hist[a][0] = out.copy()
                    self.accepted[a] += 1
                    any_acc = True
            if any_acc:
                self.accepted_at.append(self.nse)
            dP = float(np.max(np.abs(1.0 - n0 / oc.n)))
        return dP

    def step(self):
        self.it += 1
        dJ = self.oc.formal_sol_gamma_matrices()
        dP = self.stat_equil() if self.it > 3 else 1.0
        return dJ, dP

    def run(self, tolJ=2e-3, tolPops=1e-3, max_iter=400):
        dJ, dP = 1.0, 1.0
        while (dJ > tolJ or dP > tolPops) and self.it < max_iter:
            dJ, dP = self.step()
        return self.it


def cpu_run(name, ng=None, tolJ=2e-3, tolPops=1e-3, max_iter=400):
    p, _ = load_golden(name)
    loop = NgLoop(p, ng)
    loop.run(tolJ, tolPops, max_iter)
    return loop
