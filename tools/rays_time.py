"""Device time of compute_rays (mali_compute_rays) beside one formal solution (mali_formal_sol_gamma) on the same batch.

    python tools/rays_time.py [--ncol 1024] [--out profiles/rays_b200.json]

The batch is BASELINE config 4 (CaII+H, every column jittered by synth.jitter_atmosphere and set up on the device from
the thermodynamic state by upload_thermo -- the recipe of tools/ng_converge.py), advanced by 6 iterations so that J and
the populations are those of a running iteration.  Every number is the best of 5 CUDA-event timings of one call after a
warm-up call; the formal solution is timed in both arithmetic modes.  The GPU's name, power limit and clocks are
recorded with the numbers.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from ng_converge import gpu_identity  # noqa: E402


def event_ms(fn, reps=5):
    import torch
    fn()                                   # warm-up
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1))
    return min(out), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--ncol', type=int, default=1024)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from test_gpu_rays import thermo_problems
    from lightspinner_b200.engine import MaliEngine
    result = {'device': gpu_identity(), 'ncol': args.ncol, 'workload': 'config 4 (CaII+H, 82 depths, 5 rays, 777 '
              'wavelengths), upload_thermo, 6 iterations; best of 5 CUDA-event timings after a warm-up'}
    print(json.dumps(result['device']), flush=True)
    base, probs, eos, atoms = thermo_problems(args.ncol)
    eng = MaliEngine(base, args.ncol, max_upload_chunk=256)
    eng.set_eos(eos)
    eng.set_atoms(atoms)
    eng.upload_thermo(probs)
    for it in range(1, 7):
        eng.formal_sol_gamma_matrices()
        if it > 3:
            eng.stat_equil()
    rng = np.random.default_rng(0)
    rays = {}
    for nmu in (1, 5, 10, 64):
        mus = np.sort(1.0 - rng.random(nmu))[::-1].copy()
        out = torch.empty(args.ncol, int(base['Nspect']), nmu, dtype=torch.float64, device=eng.device)
        best, allv = event_ms(lambda: eng.compute_rays_async(mus, out=out))
        rays[nmu] = {'ms': best, 'ms_all': allv, 'ms_per_ray_per_column_ns': 1e6 * best / nmu / args.ncol}
        print('compute_rays nmu=%2d: %.3f ms' % (nmu, best), flush=True)
    fs = {}
    for mode in ('exact', 'contracted'):
        eng.set_arith(mode)
        best, allv = event_ms(lambda: eng.formal_sol_gamma_async())
        fs[mode] = {'ms': best, 'ms_all': allv}
        print('formal solution (%s): %.3f ms' % (mode, best), flush=True)
    result['compute_rays'] = rays
    result['formal_sol_gamma'] = fs
    result['ratio_rays_nmu5_to_fs'] = {m: rays[5]['ms'] / fs[m]['ms'] for m in fs}
    print(json.dumps(result['ratio_rays_nmu5_to_fs']), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(result, f, indent=1)
    eng.close()


if __name__ == '__main__':
    main()
