"""Time of MaliEngine.compute_response beside the hand-built upload_thermo path on the same columns.

    python tools/rf_time.py [--reps 5] [--out profiles/rf_b200.json]

Workloads: (1) response_fn.py's own: CaII / FALC, temperature +- 25 K at all 82 depths (164 columns); (2) one config-4
column (CaII+H, synth.jitter_atmosphere column 0) with temperature (+- 25 K), vturb (+- 500 m/s) and vlos (+- 1 km/s) at
all 82 depths (3 x 164 columns).  The workspace holds every column of a workload (166 columns), so each runs as one
chunk.  The damping of the shifted atmospheres is the base's (a stand-in: it is a host input).

compute_response is timed as a whole (host clock around the call, which ends in a device synchronise) and by stage,
with the engine's own stages (_solve_range, _perturb_chunk, _response_intensity) each bracketed by CUDA events and a
synchronise: base set-up and solve, clone + perturb, perturbed solve, intensity.  The hand-built path is split into
building the host problem dicts, host packing (pack_column, which upload_thermo runs per column), upload_thermo as a
whole (packing, copies and device set-up) and the solve.  Best of --reps after a warm-up run; the GPU's name and power
limit are recorded in the same run, and the two paths' intensities and iteration counts are compared bit for bit.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from ng_converge import gpu_identity  # noqa: E402

STEPS = {'temperature': 25.0, 'vturb': 500.0, 'vlos': 1000.0}


def workloads():
    from helpers import load_golden, load_setup_inputs
    from lightspinner_b200 import synth
    from lightspinner_b200.atoms import AtomTables
    from lightspinner_b200.eos import EosTables
    z = np.load(os.path.join(ROOT, 'tests', 'golden', 'eos.npz'))
    eos = EosTables.from_arrays(z)
    p1, _ = load_golden('c1_falc_ca')
    a1, _ = load_setup_inputs('c1_falc_ca')
    b1 = dict(temperature=z['falc_T'], ne=z['falc_ne'], nHTot=z['falc_nHTot'], cmass=z['falc_cmass'], vturb=p1['vturb'],
              vlos=p1['vlos'], aDamp=p1['aDamp'], nTotal=(a1['CA']['abundance'] * z['falc_nHTot'])[None, :])
    p2, _ = load_golden('c2_falc_cah')
    a2, _ = load_setup_inputs('c2_falc_cah')
    names = [str(x).strip().upper() for x in p2['atom_names']]
    T, ne, vl = synth.jitter_atmosphere(0, z['falc_T'], z['falc_ne'])
    b2 = dict(temperature=T, ne=ne, vlos=vl, nHTot=z['falc_nHTot'], cmass=z['falc_cmass'], vturb=p2['vturb'],
              aDamp=p2['aDamp'], nTotal=np.stack([a2[nm]['abundance'] * z['falc_nHTot'] for nm in names]))
    return [('falc_caII_temperature', p1, b1, eos, AtomTables.from_arrays([dict(a1['CA'])]), ['temperature']),
            ('config4_caII_h_column0', p2, b2, eos, AtomTables.from_arrays([dict(a2[nm]) for nm in names]),
             ['temperature', 'vturb', 'vlos'])]


def staged(eng, b, param, step, depths):
    """compute_response's steps one by one, each timed by CUDA events (ms); returns (times, I [ndepth, 2, ...], its)."""
    import torch
    N = eng.mt.Nspace
    adm = adp = None if param == 'vlos' else np.asarray(b['aDamp'])
    t = {}

    def ev(name, fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0 = time.perf_counter()
        e0.record()
        out = fn()
        e1.record()
        e1.synchronize()
        t[name] = dict(event_ms=e0.elapsed_time(e1), wall_ms=1e3 * (time.perf_counter() - h0))
        return out

    cols = [(int(k), s) for k in depths for s in (-1, 1)]

    def base():
        eng.upload_thermo([b], 0)
        work = eng._last_work
        eng.upload_thermo([b], 1)
        eng._solve_range(1, 1, 500, 2e-3, 1e-3)
        return work

    work = ev('base_setup_and_solve', base)
    pops0 = eng.t_pops[eng.lay.pops:2 * eng.lay.pops]
    ev('clone_and_perturb', lambda: eng._perturb_chunk(b, param, step, cols, adm, adp, 0, work, pops0, 2))
    ev('perturbed_solve', lambda: eng._solve_range(2, len(cols), 500, 2e-3, 1e-3))
    I = ev('intensity', lambda: eng._response_intensity(None, 2, len(cols)))
    its = eng.t_iter[2:2 + len(cols)].cpu().numpy()
    assert N == len(depths)
    return t, I.reshape(len(depths), 2, *I.shape[1:]), its.reshape(len(depths), 2)


def hand_built(eng, b, param, step, depths, n):
    """The path bench.py's rf_thermo section takes: host problem dicts -> upload_thermo (warm start) -> the device loop."""
    import torch
    from lightspinner_b200.response import perturbed_problem
    from lightspinner_b200.tables import pack_column
    t = {}
    h0 = time.perf_counter()
    probs = []
    for k in depths:
        for s in (-1, 1):
            q = perturbed_problem(b, param, step, int(k), s, b['aDamp'], b['aDamp'])
            q['n'] = n
            probs.append(q)
    t['build_problem_dicts_ms'] = 1e3 * (time.perf_counter() - h0)
    out = np.empty(int(eng.lay.hp_bg_chi))
    h0 = time.perf_counter()
    for q in probs:
        pack_column(eng.mt, eng.lay, q, out=out, with_background=False)
    t['host_packing_ms'] = 1e3 * (time.perf_counter() - h0)
    torch.cuda.synchronize()
    h0 = time.perf_counter()
    eng.upload_thermo(probs, 2, start_from_lte=False)
    torch.cuda.synchronize()
    t['upload_thermo_ms'] = 1e3 * (time.perf_counter() - h0)
    t['upload_thermo_without_host_packing_ms'] = t['upload_thermo_ms'] - t['host_packing_ms']
    h0 = time.perf_counter()
    eng._solve_range(2, len(probs), 500, 2e-3, 1e-3)
    torch.cuda.synchronize()
    t['solve_ms'] = 1e3 * (time.perf_counter() - h0)
    I = eng._response_intensity(None, 2, len(probs))
    its = eng.t_iter[2:2 + len(probs)].cpu().numpy()
    return t, I.reshape(len(depths), 2, *I.shape[1:]), its.reshape(len(depths), 2)


def best(runs):
    """Per key, the minimum over runs (dicts of numbers or of dicts of numbers)."""
    out = {}
    for k in runs[0]:
        v = runs[0][k]
        out[k] = best([r[k] for r in runs]) if isinstance(v, dict) else min(r[k] for r in runs)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from lightspinner_b200.engine import MaliEngine
    result = {'device': gpu_identity(), 'reps': args.reps,
              'method': 'best of --reps after one warm-up run; stages bracketed by CUDA events with a synchronise '
                        'before each; whole calls by the host clock ending in a device synchronise'}
    print(json.dumps(result['device']), flush=True)
    for name, p, b, eos, atoms, params in workloads():
        N = int(p['Nspace'])
        depths = np.arange(N)
        ncol = 2 + 2 * N
        eng = MaliEngine(p, ncol, max_upload_chunk=ncol)
        eng.set_eos(eos)
        eng.set_atoms(atoms)
        res = {'columns_per_param': 2 * N, 'workspace_columns': ncol, 'params': {}}
        for param in params:
            step = STEPS[param]
            ad = None if param == 'vlos' else np.asarray(b['aDamp'])
            whole, stages, hand = [], [], []
            for rep in range(args.reps + 1):
                torch.cuda.synchronize()
                h0 = time.perf_counter()
                rf = eng.compute_response(b, param, step, aDamp_minus=ad, aDamp_plus=ad)
                torch.cuda.synchronize()
                w = 1e3 * (time.perf_counter() - h0)
                st, I_st, its_st = staged(eng, b, param, step, depths)
                n = eng.n(1)
                hb, I_hb, its_hb = hand_built(eng, b, param, step, depths, n)
                if rep > 0:
                    whole.append({'compute_response_ms': w})
                    stages.append(st)
                    hand.append(hb)
            same = (np.array_equal(rf.I_minus, I_hb[:, 0]) and np.array_equal(rf.I_plus, I_hb[:, 1])
                    and np.array_equal(rf.iterations, its_hb) and np.array_equal(I_st, I_hb)
                    and np.array_equal(its_st, its_hb))
            r = {'step': step, 'compute_response': best(whole), 'compute_response_stages': best(stages),
                 'hand_built': best(hand), 'bit_identical': bool(same),
                 'iterations': {'base': int(rf.base_iterations), 'min': int(rf.iterations.min()),
                                'max': int(rf.iterations.max()), 'mean': float(rf.iterations.mean())},
                 'all_converged': bool(rf.converged.all())}
            hb = r['hand_built']
            r['hand_built_total_ms'] = hb['build_problem_dicts_ms'] + hb['upload_thermo_ms'] + hb['solve_ms']
            print(name, param, json.dumps(r), flush=True)
            res['params'][param] = r
        result[name] = res
        eng.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
