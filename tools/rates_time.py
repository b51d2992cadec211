"""Device time of compute_rates (mali_compute_rates) beside one formal solution and compute_rays on the same batch.

    python tools/rates_time.py [--ncol 1024] [--out profiles/rates_b200.json]

The batch is that of tools/rays_time.py: BASELINE config 4 (CaII+H, every column jittered by synth.jitter_atmosphere
and set up on the device from the thermodynamic state by upload_thermo), advanced by 6 iterations.  Four calls are
timed with CUDA events, alternated within each of 5 rounds after a warm-up round, and the best of the 5 is kept:
compute_rates, one formal solution in exact and in contracted mode, and compute_rays at nmu = Nrays.  Every output is
preallocated.  The GPU's name, power limit and clocks are recorded with the numbers, and the registers and spills of
the two rates kernels are read from ptxas (-Xptxas -v) on a compile of mali_api.cu into a temporary directory.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from ng_converge import gpu_identity  # noqa: E402


def ptxas_resources(names=('rates_kernel', 'rates_finish_kernel')):
    """{kernel: {registers, spill_stores, spill_loads, stack}} of the library's flags, from ptxas -v."""
    from lightspinner_b200 import build
    src = os.path.join(build.CSRC, 'mali_api.cu')
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [build.nvcc_path()] + build.NVCC_FLAGS + ['-Xptxas', '-v', '-cubin', '-o', os.path.join(tmp, 'api.cubin'), src]
        log = subprocess.run(cmd, capture_output=True, text=True, check=True).stderr
    out = {}
    for name in names:
        m = re.search(r"Function properties for \S*\d%s\S*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                      r"(\d+) bytes spill loads\n.*?Used (\d+) registers" % name, log)
        out[name] = dict(registers=int(m.group(4)), spill_stores=int(m.group(2)), spill_loads=int(m.group(3)),
                         stack_bytes=int(m.group(1)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--ncol', type=int, default=1024)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from test_gpu_rays import thermo_problems
    from lightspinner_b200.engine import MaliEngine
    result = {'device': gpu_identity(), 'ncol': args.ncol, 'workload': 'config 4 (CaII+H, 82 depths, 5 rays, 777 '
              'wavelengths), upload_thermo, 6 iterations; the four calls alternated in each of 5 rounds after a '
              'warm-up round, best of 5 CUDA-event timings, outputs preallocated'}
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
    f64 = dict(dtype=torch.float64, device=eng.device)
    R = int(base['Nrays'])
    rates_out = tuple(torch.empty(args.ncol, eng.mt.Ntrans, eng.mt.Nspace, **f64) for _ in range(2))
    mus = np.asarray(base['muz'], dtype=np.float64)
    rays_out = torch.empty(args.ncol, int(base['Nspect']), R, **f64)

    def fs(mode):
        eng.set_arith(mode)
        eng.formal_sol_gamma_async()

    calls = {'compute_rates': lambda: eng.compute_rates_async(out=rates_out),
             'formal_sol_gamma_exact': lambda: fs('exact'),
             'formal_sol_gamma_contracted': lambda: fs('contracted'),
             'compute_rays_nmu%d' % R: lambda: eng.compute_rays_async(mus, out=rays_out)}
    times = {k: [] for k in calls}
    for rnd in range(6):
        for k, fn in calls.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            if rnd > 0:                      # round 0 is the warm-up
                times[k].append(e0.elapsed_time(e1))
    eng._raise_rays_faults(0)
    res = {k: {'ms': min(v), 'ms_all': v} for k, v in times.items()}
    for k, v in res.items():
        print('%-30s %.3f ms' % (k, v['ms']), flush=True)
    result['timings'] = res
    r = res['compute_rates']['ms']
    result['ratio_rates_to'] = {k: r / v['ms'] for k, v in res.items() if k != 'compute_rates'}
    print(json.dumps(result['ratio_rates_to']), flush=True)
    result['ptxas'] = ptxas_resources()
    print(json.dumps(result['ptxas']), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(result, f, indent=1)
    eng.close()


if __name__ == '__main__':
    main()
