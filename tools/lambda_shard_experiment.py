#!/usr/bin/env python
"""BASELINE config 5 (experiment): one stress column -- 10x refined wavelength grid, 10-point Gauss-Legendre mu,
512 depths -- wavelength-sharded over the GPUs of one box with an NCCL all-reduce of Gamma per iteration.

    python tools/lambda_shard_experiment.py [--check]                                  # 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        tools/lambda_shard_experiment.py [--check]                                     # N GPUs

Prints one JSON line (rank 0): ms per formal solution / per iteration, exchange size, and with --check the
agreement with the CPU oracle run on the same inputs (test infrastructure, not on the measured path)."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))


def build_problem(refine=10, nrays=10, ndepth=512, base_name='stress_r10_d512'):
    """The stress column: the reference-made 10-ray / 512-depth CaII column (tests/golden/stress_r10_d512.npz, built by
    the reference's own recipe with the x1 wavelength grid) with every wavelength interval refined `refine` times
    (lightspinner_b200.synth.stress_problem; the reference's x10 grid refines the lines only: Nspect 2627)."""
    from helpers import load_golden
    from lightspinner_b200 import synth
    base, _ = load_golden(base_name)
    return synth.stress_problem(base, refine=refine, nrays=nrays, ndepth=ndepth)


def run(q, iters=6, warmup=6, init_dist=True):
    """Times `iters` MALI iterations of the wavelength-sharded column on the ranks of the current torchrun launch, after
    a warm-up pass of `warmup` iterations (none when 0; each pass starts from fresh populations).
    Returns a dict (rank 0) with per-iteration times, split into formal solution / all-reduce / statistical equilibrium."""
    import torch
    import torch.distributed as dist
    from lightspinner_b200.lambda_shard import LambdaShardedColumn
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1 and init_dist and not dist.is_initialized():
        dist.init_process_group('nccl', device_id=dev)
    col = LambdaShardedColumn(q, device=local, specialize=True)
    info = col.eng.model_info()
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def one_pass(iters):
        col.eng.upload([col.sub])
        col.eng.reset_iteration_state()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        fs, ar, se, tot = [], [], [], []
        for it in range(1, iters + 1):
            e = [ev() for _ in range(4)]
            e[0].record()
            col.eng.formal_sol_gamma_async()
            e[1].record()
            col.exchange()              # one all-gather of [Gamma | dJ] + fixed-order sum / max (lambda_shard.GammaExchange)
            e[2].record()
            if it > 3:
                col.eng.stat_equil_async()
            e[3].record()
            torch.cuda.synchronize(dev)
            fs.append(e[0].elapsed_time(e[1]))
            ar.append(e[1].elapsed_time(e[2]))
            se.append(e[2].elapsed_time(e[3]))
            tot.append(e[0].elapsed_time(e[3]))
        return [float(np.median(x)) for x in (fs, ar, se, tot)]

    if warmup > 0:
        one_pass(warmup)                              # warm-up (library load, NCCL channels)
    med = one_pass(iters)
    ar_min = med[1]
    if world > 1:
        # the exchange segment of a rank includes its wait for the slowest rank's formal solution: the MIN over ranks (the
        # rank that arrives last) is the cost of the collective itself, the MAX is dominated by the load imbalance
        tmin = torch.tensor([med[1]], dtype=torch.float64, device=dev)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        ar_min = float(tmin[0])
        t = torch.tensor(med, dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        med = [float(x) for x in t]
    units = int(q['Nspect']) * int(q['Nrays']) * int(q['Nspace'])
    out = {'experiment': 'wavelength-sharded single column (BASELINE config 5)', 'n_gpus': world,
           'Nspect': int(q['Nspect']), 'Nrays': int(q['Nrays']), 'Nspace': int(q['Nspace']),
           'units_per_iteration': units, 'wavelengths_this_rank': col.hi - col.lo, 'tiles_this_rank': info['ntile'],
           'generic_tiles': info['generic_tiles'], 'ms_formal_solution': med[0], 'ms_gamma_allreduce': med[1],
           'ms_stat_equil': med[2], 'ms_per_iteration': med[3], 'ms_gamma_exchange_itself': ar_min,
           'note': 'ms_formal_solution / ms_gamma_allreduce are maxima over ranks of the two segments: the second one is '
                   'mostly the lighter ranks waiting for the slowest formal solution; ms_gamma_exchange_itself (minimum over '
                   'ranks) is the collective: one all-gather of [Gamma | dJ] + fixed-order sum',
           'allreduce_share_of_iteration': med[1] / med[3] if med[3] > 0 else None,
           'updates_per_s': units / (med[3] * 1e-3), 'exchange_bytes_per_iteration': int(col.eng.t_Gamma.numel()) * 8 + 8,
           'finite': bool(np.isfinite(col.n()).all())}
    col.close()
    return out if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--refine', type=int, default=10)
    ap.add_argument('--nrays', type=int, default=10)
    ap.add_argument('--ndepth', type=int, default=512)
    ap.add_argument('--iters', type=int, default=6)
    ap.add_argument('--check', action='store_true', help='compare with the CPU oracle (slow: ~10 s per iteration)')
    ap.add_argument('--prebuild', action='store_true', help='only build the specialised library (no GPU needed)')
    args = ap.parse_args()

    from helpers import load_golden
    from lightspinner_b200 import synth
    base, _ = load_golden('c1_falc_ca')
    t0 = time.perf_counter()
    q = synth.stress_problem(base, refine=args.refine, nrays=args.nrays, ndepth=args.ndepth)
    t_setup = time.perf_counter() - t0
    if args.prebuild:
        from lightspinner_b200 import specialize
        print(specialize.library_for(q, verbose=True))
        return

    import torch
    import torch.distributed as dist
    from lightspinner_b200.lambda_shard import LambdaShardedColumn
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ['NCCL_DEBUG'] = os.environ.get('MALI_NCCL_DEBUG', 'WARN')
        dist.init_process_group('nccl', device_id=dev)

    col = LambdaShardedColumn(q, device=local, specialize=True)
    info = col.eng.model_info()

    def run(record):
        col.eng.upload([col.sub])          # fresh populations, J = 0
        col.eng.reset_iteration_state()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        fs_ms, it_ms, hist, first = [], [], [], None
        for it in range(1, args.iters + 1):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            dJ = col.formal_sol_gamma_matrices()      # FS + all-reduce(Gamma, dJ) + one scalar read
            t1 = time.perf_counter()
            if record and it == 1:
                first = (col.eng.J(0), col.eng.I(0), col.eng.Gamma(0))
            t1b = time.perf_counter()
            dP = col.stat_equil() if it > 3 else None
            torch.cuda.synchronize(dev)
            t2 = time.perf_counter()
            fs_ms.append(1e3 * (t1 - t0))
            it_ms.append(1e3 * (t1 - t0 + t2 - t1b))
            hist.append((dJ, dP))
        return fs_ms, it_ms, hist, first

    run(False)                                        # warm-up (library load, NCCL channels)
    fs_ms, it_ms, hist, first = run(True)
    if world > 1:
        t = torch.tensor([float(np.median(fs_ms)), float(np.median(it_ms))], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        fs_med, it_med = float(t[0]), float(t[1])
    else:
        fs_med, it_med = float(np.median(fs_ms)), float(np.median(it_ms))

    check = None
    if args.check:
        ok = {}
        if rank == 0:
            from oracle import mali_oracle as O
            O.build()
            oc = O.OracleContext(q)
            t0 = time.perf_counter()
            for it in range(1, args.iters + 1):
                dJ = oc.formal_sol_gamma_matrices()
                if it == 1:
                    lo, hi = col.lo, col.hi
                    J, I, G = first
                    ok['J_slice_bitwise'] = bool(np.array_equal(J, oc.J[lo:hi]))
                    ok['I_slice_bitwise'] = bool(np.array_equal(I, oc.I[lo:hi]))
                    ok['J_slice_relerr'] = float(np.max(np.abs(J - oc.J[lo:hi]) / np.abs(oc.J[lo:hi])))
                    ok['Gamma_relerr'] = float(np.max(np.abs(G - oc.Gamma)) / np.max(np.abs(oc.Gamma)))
                if it > 3:
                    oc.stat_equil(use_scipy=False)
            ok['oracle_seconds'] = time.perf_counter() - t0
            n = col.n()
            ok['n_relerr_after_%d_iterations' % args.iters] = float(np.max(np.abs(n - oc.n) / np.abs(oc.n)))
        check = ok
    if world > 1:
        dist.barrier()

    if rank == 0:
        units = int(q['Nspect']) * int(q['Nrays']) * int(q['Nspace'])
        print(json.dumps({
            'experiment': 'wavelength-sharded single column (BASELINE config 5)', 'n_gpus': world,
            'Nspect': int(q['Nspect']), 'Nrays': int(q['Nrays']), 'Nspace': int(q['Nspace']),
            'units_per_iteration': units, 'wavelengths_this_rank': col.hi - col.lo, 'tiles_this_rank': info['ntile'],
            'generic_tiles': info['generic_tiles'], 'ms_per_formal_solution': fs_med, 'ms_per_iteration': it_med,
            'updates_per_s': units / (it_med * 1e-3), 'exchange_bytes_per_iteration': int(col.eng.t_Gamma.numel()) * 8 + 8,
            'host_setup_seconds': t_setup, 'history': hist, 'check': check}))
    col.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
