"""Ng acceleration on the GPU (mali_iterate_ng, mali_stat_equil_ng, mali_ng_hook) against the CPU restatement of
tests/ng_reference.py (numpy Ng step on the C oracle's loop).  Every achieved error is printed."""
import numpy as np
import pytest

from helpers import load_golden, relerr
from ng_reference import NgLoop, ng_step

pytestmark = pytest.mark.gpu

DEFAULT = (2, 3, 3)
# final n, J, I of the free-running GPU loop vs the CPU loop after the same iteration count: 10x the worst measured on a
# B200 (3.6e-11, I of c2v_jitter_cah_0 in the contracted mode; the other cases 5e-12..3e-11)
TOL_FINAL = 4e-10


@pytest.fixture(scope='module')
def eng_mod():
    import torch
    assert torch.cuda.is_available()
    from lightspinner_b200 import engine
    return engine


def ng_opts(order=2, delay=3, period=3):
    from lightspinner_b200 import NgOptions
    return NgOptions(order, delay, period)


def run_device(eng_mod, probs, ng, max_iter=400, tolJ=2e-3, tolPops=1e-3, arith=None, ranges=None, graph=True):
    eng = eng_mod.MaliEngine(probs[0], len(probs), arith=arith, ng=ng)
    eng.upload(probs)
    eng.reset_iteration_state()
    if not graph:
        eng.profile_begin(4 * max_iter)      # profiling disables the captured graph: plain launches
    for c0, nc in (ranges or [(0, len(probs))]):
        eng.iterate_async(max_iter, tolJ, tolPops, col0=c0, ncol=nc)
    if not graph:
        eng.profile_end()
    import torch
    torch.cuda.synchronize()
    return eng


# ---------------------------------------------------------------------------------------------------- 1. the hook
def recorded_histories():
    out = []
    for name in ('c1_falc_ca', 'c2_falc_cah'):
        p, _ = load_golden(name)
        loop = NgLoop(p, None, record=True)
        while loop.nse < 12:
            loop.step()
        for a in range(loop.oc.Natom):
            for nse in (6, 9, 12):
                out.append((name, a, nse, loop.solved[a][:nse][::-1]))    # newest first
    return out


def test_hook_matches_numpy_on_recorded_histories(eng_mod, oracle):
    """The kernels' Ng step vs the numpy definition on the oracle loop's solved vectors.  The bar is 1e-12 relative,
    or -- where the small system is ill-conditioned -- 10 x cond(A) eps |c| |x1 - x0| / |x*|: the coefficients of the
    two codes then agree only to cond(A) eps, and an error dc moves x* by dc (x_i - x0)."""
    for name, a, nse, solved in recorded_histories():
        for order in (1, 2, 3):
            hist = np.array(solved[:order + 2])
            ref, ok = ng_step(hist, order)
            got, acc = eng_mod.ng_hook(hist, order)
            assert acc == ok, (name, a, nse, order)
            if not ok:
                assert np.array_equal(got, hist[0])
                print('%s atom %d nse %2d order %d: rejected by both' % (name, a, nse, order))
                continue
            x0 = hist[0]
            d = [hist[i] - hist[i + 1] for i in range(order + 1)]
            w = 1.0 / (x0 * x0)
            E = np.array([d[0] - d[i + 1] for i in range(order)])
            A = (E * w) @ E.T
            c = np.linalg.solve(A, (E * w) @ d[0])
            spread = max(float(np.max(np.abs(hist[i] - x0) / ref)) for i in range(1, order + 1))
            bound = 10.0 * np.linalg.cond(A) * np.finfo(float).eps * float(np.max(np.abs(c))) * spread
            err = relerr(got, ref)
            print('%s atom %d nse %2d order %d: rel err %.2e  (cond(A) %.1e, bar %.1e)'
                  % (name, a, nse, order, err, np.linalg.cond(A), max(1e-12, bound)))
            assert err <= max(1e-12, bound)


def test_hook_recovers_two_geometric_modes(eng_mod):
    rng = np.random.default_rng(11)
    xs = 1.0 + rng.random(3000)
    u, v = rng.random(3000) - 0.5, rng.random(3000) - 0.5
    hist = np.array([xs + u * 0.7 ** k + v * 0.4 ** k for k in (3, 2, 1, 0)])
    got, acc = eng_mod.ng_hook(hist, 2)
    err = relerr(got, xs)
    print('order 2 on two geometric modes: x* recovered to %.2e' % err)
    assert acc and err <= 1e-10


def test_hook_rejects_and_leaves_the_input(eng_mod):
    rng = np.random.default_rng(5)
    xs = 1.0 + rng.random(700)
    xs[17] = -0.05                                          # the exact limit has a negative entry ...
    u, v = 0.5 + rng.random(700), 0.5 + rng.random(700)
    neg = np.array([xs + u * 0.7 ** k + v * 0.4 ** k for k in (3, 2, 1, 0)])
    assert (neg > 0).all()                                  # ... the iterates do not
    nan = neg.copy()
    nan[0, 3] = np.nan
    same = np.repeat(neg[:1], 4, axis=0)                    # identical iterates: A == 0
    for label, hist in (('negative x*', neg), ('NaN input', nan), ('identical iterates', same)):
        got, acc = eng_mod.ng_hook(hist, 2)
        print('%s: accepted %s' % (label, acc))
        assert not acc
        assert np.array_equal(got, hist[0], equal_nan=True)


# ---------------------------------------------------------------------------------------------------- 2. vs the CPU loop
@pytest.mark.parametrize('arith', ['exact', 'contracted'])
@pytest.mark.parametrize('name,count', [('c1_falc_ca', 29), ('c2_falc_cah', 32), ('c2v_jitter_cah_0', 32)])
def test_device_loop_matches_cpu_ng_loop(eng_mod, oracle, name, count, arith):
    p, _ = load_golden(name)
    loop = NgLoop(p, DEFAULT)
    loop.run()
    eng = run_device(eng_mod, [p], ng_opts(), arith=arith)
    it = int(eng.t_iter.cpu()[0])
    acc = eng.ng_accepted()[0]
    e = dict(n=relerr(eng.n(0), loop.oc.n), J=relerr(eng.J(0), loop.oc.J), I=relerr(eng.I(0), loop.oc.I))
    print('%s %s: iterations GPU %d CPU %d, accepted GPU %s CPU %s, rel err n %.2e J %.2e I %.2e'
          % (name, arith, it, loop.it, acc.tolist(), loop.accepted.tolist(), e['n'], e['J'], e['I']))
    assert it == loop.it == count
    assert int(eng.t_done.cpu()[0]) == 1
    assert acc.tolist() == loop.accepted.tolist()
    assert max(e.values()) <= TOL_FINAL
    eng.close()


def test_tight_tolerance_same_fixed_point_in_half_the_iterations(eng_mod):
    p, _ = load_golden('c2_falc_cah')
    plain = run_device(eng_mod, [p], None, max_iter=600, tolJ=1e-9, tolPops=1e-9)
    ng = run_device(eng_mod, [p], ng_opts(), max_iter=600, tolJ=1e-9, tolPops=1e-9)
    ip, ig = int(plain.t_iter.cpu()[0]), int(ng.t_iter.cpu()[0])
    err = relerr(ng.n(0), plain.n(0))
    print('C2 at tol 1e-9: plain %d, Ng %d iterations; populations differ by %.2e' % (ip, ig, err))
    assert int(plain.t_done.cpu()[0]) == 1 and int(ng.t_done.cpu()[0]) == 1
    assert ig <= 0.5 * ip
    assert err <= 1e-7
    plain.close()
    ng.close()


# ---------------------------------------------------------------------------------------------------- 4. off means off
def test_never_due_is_bit_identical_to_plain(eng_mod):
    names = ['c1_falc_ca', 'rf_k40p', 'rf_k10m']
    probs = [load_golden(n)[0] for n in names]
    a = run_device(eng_mod, probs, None, max_iter=60)
    b = run_device(eng_mod, probs, ng_opts(delay=60), max_iter=60)
    for c in range(3):
        for f in ('n', 'J', 'I'):
            assert np.array_equal(getattr(a, f)(c), getattr(b, f)(c)), (names[c], f)
    for t in ('t_iter', 't_done', 't_dJ', 't_dPops', 't_status'):
        assert np.array_equal(getattr(a, t).cpu().numpy(), getattr(b, t).cpu().numpy()), t
    assert b.ng_accepted().sum() == 0 and b.t_ng_nse.cpu().numpy().tolist() == [int(i) - 3 for i in b.t_iter.cpu()]
    a.close()
    b.close()


# ---------------------------------------------------------------------------------------------------- 5. determinism
def batch7():
    """Seven columns of one radiative model (CaII/FALC, 5 rays): the three fixtures of that model and four jittered
    copies of the first (synth.jitter_problem).  c1v_jitter_ca3 has another ray quadrature, so it is not one of them."""
    from lightspinner_b200 import synth
    probs = [load_golden(n)[0] for n in ('c1_falc_ca', 'rf_k40p', 'rf_k10m')]
    return probs + [synth.jitter_problem(probs[0], c) for c in range(1, 5)]


def test_batch_split_single_and_graph_are_bit_identical(eng_mod):
    probs = batch7()
    whole = run_device(eng_mod, probs, ng_opts(), max_iter=100)
    assert whole.graph_iterations() == 100
    split = run_device(eng_mod, probs, ng_opts(), max_iter=100, ranges=[(0, 3), (3, 4)])
    plain_launch = run_device(eng_mod, probs, ng_opts(), max_iter=100, graph=False)
    assert plain_launch.graph_iterations() == 0
    print('7-column batch: iterations %s, accepted %s' % (whole.t_iter.cpu().numpy().tolist(),
                                                          whole.ng_accepted()[:, 0].tolist()))
    assert whole.ng_accepted().sum() > 0
    for other in (split, plain_launch):
        assert np.array_equal(whole.t_iter.cpu().numpy(), other.t_iter.cpu().numpy())
        assert np.array_equal(whole.ng_accepted(), other.ng_accepted())
        for c in range(7):
            assert np.array_equal(whole.n(c), other.n(c)) and np.array_equal(whole.I(c), other.I(c)), c
    for c, p in enumerate(probs):
        single = run_device(eng_mod, [p], ng_opts(), max_iter=100)
        assert int(single.t_iter.cpu()[0]) == int(whole.t_iter.cpu()[c])
        assert np.array_equal(single.n(0), whole.n(c)) and np.array_equal(single.J(0), whole.J(c)), c
        single.close()
    for e in (whole, split, plain_launch):
        e.close()


def test_per_call_context_equals_batch_context(eng_mod):
    """The loop of test.py:20-29 on Context(ng=...) gives the same populations, bit for bit, and the same count as
    BatchContext(ng=...).iterate()."""
    from helpers import fake_reference_objects
    from lightspinner_b200 import BatchContext, Context
    p, _ = load_golden('c2_falc_cah')
    ctx = Context(*fake_reference_objects(p), ng=ng_opts())
    dJ, dPops, i = 1.0, 1.0, 0
    while dJ > 2e-3 or dPops > 1e-3:
        i += 1
        dJ = ctx.formal_sol_gamma_matrices()
        if i > 3:
            dPops = ctx.stat_equil()
    n_ctx = np.concatenate([a.n for a in ctx.activeAtoms])
    objs = fake_reference_objects(p)
    batch = BatchContext([objs], ng=ng_opts())
    its = batch.iterate()
    n_batch = np.concatenate([a.n for a in batch[0].activeAtoms])
    print('Context loop %d iterations, BatchContext %d' % (i, its[0]))
    assert i == int(its[0]) == 32
    assert np.array_equal(n_ctx, n_batch)
    ctx.close()
    batch.close()


# ---------------------------------------------------------------------------------------------------- 6. conservation
def test_accepted_steps_conserve_particles(eng_mod):
    p, _ = load_golden('c2_falc_cah')
    eng = eng_mod.MaliEngine(p, 1, ng=ng_opts())
    eng.upload([p])
    nTot = np.asarray(p['nTotal'])
    lvl = np.concatenate([[0], np.cumsum(p['Nlevel'])])
    worst, steps = 0.0, 0
    for i in range(1, 33):
        eng.formal_sol_gamma_matrices()
        if i > 3:
            before = eng.ng_accepted().sum()
            eng.stat_equil()
            if eng.ng_accepted().sum() > before:
                steps += 1
                n = eng.n(0)
                for a in range(len(lvl) - 1):
                    worst = max(worst, float(np.max(np.abs(n[lvl[a]:lvl[a + 1]].sum(axis=0) / nTot[a] - 1.0))))
    print('%d accepted steps, worst relative violation of sum_l n_l = nTotal: %.2e' % (steps, worst))
    assert steps == 8 and worst <= 1e-12
    eng.close()


# ---------------------------------------------------------------------------------------------------- 7. shapes
def lockstep_ng(eng, p, niter, ng):
    """Both sides start every iteration from the CPU side's populations; each keeps its own Ng history."""
    loop = NgLoop(p, ng)
    worst, acc = 0.0, []
    for it in range(1, niter + 1):
        eng.set_n(0, loop.oc.n)
        eng.formal_sol_gamma_matrices()
        loop.it += 1
        loop.oc.formal_sol_gamma_matrices()
        if it > 3:
            a0 = eng.ng_accepted()[0].copy()
            dP = float(eng.stat_equil()[0])
            l0 = loop.accepted.copy()
            dPo = loop.stat_equil()
            assert np.array_equal(eng.ng_accepted()[0] - a0, loop.accepted - l0), it
            assert abs(dP - dPo) <= 1e-8 + 1e-6 * dPo, (it, dP, dPo)
            worst = max(worst, relerr(eng.n(0), loop.oc.n))
    return worst, loop


def test_stress_512_depths_10_rays(eng_mod, oracle):
    p, _ = load_golden('stress_r10_d512')
    eng = eng_mod.MaliEngine(p, 1, ng=ng_opts(delay=0))
    eng.upload([p])
    worst, loop = lockstep_ng(eng, p, 12, (2, 0, 3))
    print('stress_r10_d512, 12 lock-step iterations, delay 0: accepted %s, worst rel err n %.2e'
          % (loop.accepted.tolist(), worst))
    # extrapolations are due after solves 6 and 9; this far from convergence x* has negative entries at 3 of the
    # 512 x 6 points (c ~ (-7.7, 1.9) and (-29, 10)), so both codes reject both steps and keep the solved populations
    assert loop.nse == 9 and loop.accepted.sum() == 0 and worst <= 1e-8
    eng.close()


@pytest.mark.parametrize('name', ['merged12', 'merged16'])
def test_many_level_atoms(eng_mod, oracle, name):
    import warnings
    import model_shapes as ms
    q = ms.build(name)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)     # the generic-kernel notice
        eng = eng_mod.MaliEngine(q, 1, ng=ng_opts(delay=0))
    eng.upload([q])
    worst, loop = lockstep_ng(eng, q, 10, (2, 0, 3))
    print('%s (Nlevel %s), 10 lock-step iterations: accepted %s, worst rel err n %.2e'
          % (name, list(q['Nlevel']), loop.accepted.tolist(), worst))
    assert loop.accepted.sum() > 0 and worst <= 1e-8
    eng.close()


# ---------------------------------------------------------------------------------------------------- 8. faults
def test_singular_system_still_raises_through_the_ng_loop(eng_mod):
    from helpers import only_transitions
    p, _ = load_golden('c1_falc_ca')
    q = dict(p)
    q['C'] = np.zeros_like(np.asarray(p['C']))
    q = only_transitions(q, [])
    eng = run_device(eng_mod, [q], ng_opts(delay=0, period=1), max_iter=8)
    assert int(eng.t_done.cpu()[0]) == 2 and int(eng.t_iter.cpu()[0]) == 4
    with pytest.raises(np.linalg.LinAlgError):
        eng.raise_on_faults()
    eng.close()


def test_done_column_history_stops_changing(eng_mod):
    p, _ = load_golden('c1_falc_ca')
    eng = run_device(eng_mod, [p], ng_opts(), max_iter=40)
    assert int(eng.t_done.cpu()[0]) == 1
    nse, hist = eng.t_ng_nse.clone(), eng.t_ng_hist.clone()
    eng.iterate_async(10)
    import torch
    torch.cuda.synchronize()
    assert int(eng.t_iter.cpu()[0]) == 29
    assert torch.equal(nse, eng.t_ng_nse) and torch.equal(hist, eng.t_ng_hist)
    eng.close()
