"""Device time of compute_rays_depth (mali_compute_rays_depth) beside compute_rays (mali_compute_rays) on the same batch.

    python tools/rays_depth_time.py [--ncol 1024] [--out profiles/rays_depth_b200.json]

The batch is the one of tools/rays_time.py: BASELINE config 4 (CaII+H, every column jittered by synth.jitter_atmosphere
and set up on the device from the thermodynamic state by upload_thermo), advanced by 6 iterations.  For nmu = 1, 5 and
10 angles it times compute_rays, compute_rays_depth with every quantity, and compute_rays_depth with I only, the three
alternated within each of 5 rounds; every number is the best of those 5 CUDA-event timings of one call, after a warm-up
call of each.  The outputs are preallocated, so no allocation is timed.  The bytes are what the kernel must move:
every output written once, and for the all-quantities call the second pass's read and rewrite of tau and contrib.
The GPU's name, power limit and clocks are recorded with the numbers.
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

DEPTH_ARRAYS = ('I', 'chi', 'S', 'tau', 'contrib')


def call_bytes(quantities, ncol, N, Ns, nmu):
    """(bytes written, bytes of the second pass) of one compute_rays_depth call."""
    ray = ncol * Ns * nmu * 8
    written = sum(N * ray for q in quantities if q in DEPTH_ARRAYS) + (ray if 'z_tau1' in quantities else 0) + \
        (ncol * N * 8 if 'height' in quantities else 0)
    pass2 = 2 * N * ray * sum(q in quantities for q in ('tau', 'contrib')) if 'tau' in quantities else 0
    return written, pass2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--ncol', type=int, default=1024)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from test_gpu_rays import thermo_problems
    from lightspinner_b200.engine import RAYS_DEPTH_QUANTITIES, MaliEngine
    result = {'device': gpu_identity(), 'ncol': args.ncol,
              'workload': 'config 4 (CaII+H, 82 depths, 5 rays, 777 wavelengths), upload_thermo, 6 iterations; '
                          'compute_rays, compute_rays_depth (all quantities) and compute_rays_depth (I only) alternated; '
                          'best of %d CUDA-event timings after a warm-up; outputs preallocated' % args.reps}
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
    N, Ns, ncol = int(base['Nspace']), int(base['Nspect']), args.ncol
    rng = np.random.default_rng(0)
    rows = {}
    for nmu in (1, 5, 10):
        mus = np.sort(1.0 - rng.random(nmu))[::-1].copy()
        f64 = dict(dtype=torch.float64, device=eng.device)
        I_rays = torch.empty(ncol, Ns, nmu, **f64)
        full = {q: torch.empty((ncol, Ns, nmu) if q == 'z_tau1' else (ncol, N) if q == 'height'
                               else (ncol, N, Ns, nmu), **f64) for q in RAYS_DEPTH_QUANTITIES}
        only_I = {'I': full['I']}
        calls = {
            'compute_rays': lambda: eng.compute_rays_async(mus, out=I_rays),
            'depth_all': lambda: eng.compute_rays_depth_async(mus, out=full),
            'depth_I': lambda: eng.compute_rays_depth_async(mus, quantities=['I'], out=only_I),
        }
        times = {k: [] for k in calls}
        for fn in calls.values():                     # warm-up
            fn()
        torch.cuda.synchronize()
        for _ in range(args.reps):
            for k, fn in calls.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                e1.synchronize()
                times[k].append(e0.elapsed_time(e1))
        # the three calls agree where they overlap
        assert torch.equal(full['I'][:, 0], I_rays)
        row = {}
        for k, v in times.items():
            row[k] = {'ms': min(v), 'ms_all': v}
            if k != 'compute_rays':
                q = RAYS_DEPTH_QUANTITIES if k == 'depth_all' else ('I',)
                w, p2 = call_bytes(q, ncol, N, Ns, nmu)
                row[k].update(bytes_written=w, bytes_pass2=p2, GBps_written=w / (min(v) * 1e6),
                              GBps_moved=(w + p2) / (min(v) * 1e6))
            else:
                row[k].update(bytes_written=ncol * Ns * nmu * 8)
        row['depth_all_over_compute_rays'] = row['depth_all']['ms'] / row['compute_rays']['ms']
        row['depth_I_over_compute_rays'] = row['depth_I']['ms'] / row['compute_rays']['ms']
        rows[nmu] = row
        print('nmu=%2d: compute_rays %.3f ms; depth (all) %.3f ms, %.1f GB written, %.0f GB/s moved; depth (I) %.3f ms'
              % (nmu, row['compute_rays']['ms'], row['depth_all']['ms'], row['depth_all']['bytes_written'] / 1e9,
                 row['depth_all']['GBps_moved'], row['depth_I']['ms']), flush=True)
        del full, only_I, I_rays
        torch.cuda.empty_cache()
    result['nmu'] = rows
    ref = os.path.join(ROOT, 'profiles', 'rays_b200.json')
    if os.path.isfile(ref):
        old = json.load(open(ref))['compute_rays']
        result['compute_rays_vs_rays_b200_json'] = {n: rows[n]['compute_rays']['ms'] / old[str(n)]['ms'] for n in rows}
        print(json.dumps(result['compute_rays_vs_rays_b200_json']), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(result, f, indent=1)
    eng.close()


if __name__ == '__main__':
    main()
