"""Seconds to converge and iteration counts with and without Ng acceleration (lightspinner_b200.NgOptions), on one GPU.

    python tools/ng_converge.py [--ncol4 1024] [--out ng_converge.json]

Cases: one CaII/FALC column (C1), one CaII+H/FALC column (C2), the 164-column response-function batch (FALC with
T[k] +- 25 K, warm-started from the converged C1 populations; Ng is never due within its 5 iterations) and the
config-4 batch (CaII+H, every column jittered by synth.jitter_atmosphere and set up on the device from the
thermodynamic state by upload_thermo -- the recipe of bench.py's config4_from_thermodynamic_state).  For every case
and mode: one warm-up solve, then the best of 3 (set-up excluded: the columns are re-uploaded before each solve), the
per-column iteration histogram and the number of columns that hit the iteration cap.  Also the time per iteration
with and without Ng on the config-4 batch (fixed iteration count, Ng extrapolations due as in a converging run).
The GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

MAX_ITER = 400


def gpu_identity():
    import torch
    info = {'gpu': torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        info['nvidia_smi'] = out
    except Exception as ex:   # the numbers are still reported; the power limit is then unknown
        info['nvidia_smi'] = 'unavailable: %r' % (ex,)
    return info


def solve(eng, setup, fixed=None):
    """(seconds, iterations per column) of one solve; set-up (re-upload) not timed."""
    import torch
    setup()
    eng.reset_iteration_state()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if fixed is not None:
        eng.iterate_async(fixed, -1.0, -1.0)
    else:
        done = 0
        while done < MAX_ITER:
            eng.iterate_async(16)
            done += 16
            if bool((eng.t_done != 0).all().item()):
                break
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    eng.raise_on_faults()
    return dt, eng.t_iter.cpu().numpy().copy()


def measure(make, label, fixed=None):
    from lightspinner_b200 import NgOptions
    out = {}
    for mode, ng in (('plain', None), ('ng', NgOptions())):
        eng, setup = make(ng)
        solve(eng, setup, fixed)                     # warm-up: graph capture, module loading
        runs = [solve(eng, setup, fixed) for _ in range(3)]
        its = runs[0][1]
        hist = {int(k): int(v) for k, v in zip(*np.unique(its, return_counts=True))}
        r = {'seconds_best_of_3': min(t for t, _ in runs), 'seconds_all': [t for t, _ in runs],
             'iteration_histogram': hist, 'columns_at_cap': int((its >= MAX_ITER).sum())}
        if fixed is not None:
            r = {'iterations': fixed, 'ms_per_iteration': 1e3 * r['seconds_best_of_3'] / fixed,
                 'seconds_all': r['seconds_all']}
        if ng is not None:
            r['ng_accepted_total'] = int(eng.ng_accepted().sum())
        out[mode] = r
        eng.close()
    if fixed is None:
        out['speedup'] = out['plain']['seconds_best_of_3'] / out['ng']['seconds_best_of_3']
    print(label, json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--ncol4', type=int, default=1024)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from helpers import load_golden, load_setup_inputs
    from lightspinner_b200 import synth
    from lightspinner_b200.atoms import AtomTables
    from lightspinner_b200.engine import MaliEngine
    from lightspinner_b200.eos import EosTables
    result = {'device': gpu_identity()}
    print(json.dumps(result['device']), flush=True)

    def single(name):
        p, _ = load_golden(name)

        def make(ng):
            eng = MaliEngine(p, 1, ng=ng)
            return eng, lambda: eng.upload([p])
        return make

    result['c1_falc_ca'] = measure(single('c1_falc_ca'), 'C1')
    result['c2_falc_cah'] = measure(single('c2_falc_cah'), 'C2')

    zeos = np.load(os.path.join(ROOT, 'tests', 'golden', 'eos.npz'))
    c1p, c1r = load_golden('c1_falc_ca')
    rfg = {40: load_golden('rf_k40p'), -10: load_golden('rf_k10m')}
    atoms1, _ = load_setup_inputs('c1_falc_ca')
    base1 = {k: c1p[k] for k in ('Nspace', 'Nrays', 'Nspect', 'wavelength', 'muz', 'wmu', 'Nlevel', 'trans', 'linepar',
                                 'alpha', 'vturb', 'vlos', 'atom_names')}
    rf_probs = []
    for k in range(int(c1p['Nspace'])):
        for sgn in (+1, -1):
            q = dict(base1)
            T = np.array(zeos['falc_T'])
            T[k] += 25.0 * sgn
            q['temperature'], q['ne'], q['nHTot'], q['cmass'] = T, zeos['falc_ne'], zeos['falc_nHTot'], zeos['falc_cmass']
            q['nTotal'] = (atoms1['CA']['abundance'] * q['nHTot'])[None, :]
            q['aDamp'] = rfg[k * sgn][0]['aDamp'] if k * sgn in rfg else c1p['aDamp']
            q['n'] = c1r['final_n']
            rf_probs.append(q)

    def make_rf(ng):
        eng = MaliEngine(c1p, len(rf_probs), max_upload_chunk=len(rf_probs), ng=ng)
        eng.set_eos(EosTables.from_arrays(zeos))
        eng.set_atoms(AtomTables.from_arrays([dict(atoms1['CA'])]))
        return eng, lambda: eng.upload_thermo(rf_probs, start_from_lte=False)
    result['response_function_164'] = measure(make_rf, 'RF164')

    base, _ = load_golden('c2_falc_cah')
    atoms4, _ = load_setup_inputs('c2_falc_cah')
    fx = {c: load_golden('c2v_jitter_cah_%d' % c) for c in (0, 1)}
    names4 = [str(x).strip().upper() for x in base['atom_names']]
    ab4 = [atoms4[nm]['abundance'] for nm in names4]
    c4_probs = []
    for c in range(args.ncol4):
        T4, ne4, vl4 = synth.jitter_atmosphere(c, zeos['falc_T'], zeos['falc_ne'])
        c4_probs.append(dict(temperature=T4, ne=ne4, vlos=vl4, nHTot=zeos['falc_nHTot'], cmass=zeos['falc_cmass'],
                             vturb=base['vturb'], nTotal=np.stack([a * zeos['falc_nHTot'] for a in ab4]),
                             aDamp=fx[c][0]['aDamp'] if c in fx else base['aDamp']))

    def make_c4(ng):
        eng = MaliEngine(base, len(c4_probs), max_upload_chunk=256, ng=ng)
        eng.set_eos(EosTables.from_arrays(zeos))
        eng.set_atoms(AtomTables.from_arrays([dict(atoms4[nm]) for nm in names4]))
        return eng, lambda: eng.upload_thermo(c4_probs)
    result['config4_%d' % args.ncol4] = measure(make_c4, 'C4x%d' % args.ncol4)
    result['config4_%d_per_iteration' % args.ncol4] = measure(make_c4, 'C4x%d per iteration' % args.ncol4, fixed=30)
    torch.cuda.synchronize()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(result, f, indent=1)


if __name__ == '__main__':
    main()
