#!/usr/bin/env python
"""bench.py -- MALI ray-depth updates/s on B200 (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--ncol C] [--iters I] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --workload lambda_shard [--gpus N]        # BASELINE config 5 experiment (one column, wavelength-sharded)

Workload (config.workload): BASELINE config 4's per-GPU share -- a synthetic 1.5D batch of `ncol` perturbed FALC
columns per GPU (default 1024; 8 GPUs = the config's 8192), CaII + H 6-level both active (Nspect 777, 5 rays, 82 depths,
25 overlapping transitions), derived from the committed reference fixture tests/golden/c2_falc_cah.npz by
lightspinner_b200/synth.py.  Columns shard across ranks with no data-path collective (weak scaling); the only
exchange is the final gather of the emergent intensities, done inside the e2e region when N > 1.

A *step* is one fixed-length MALI solve of the whole batch: `iters` iterations of the device-resident loop
(mali_iterate, convergence test off), each = formal solution + Gamma (fs_gamma_kernel_m, gamma_finish_kernel,
j_finish_kernel) + statistical equilibrium (stat_equil_kernel).
  value : units / s with the inputs already resident in HBM (units = ncol_total * Nspect * Nrays * Nspace * iters)
  e2e   : the same solve through the public API from pinned HOST buffers: every step copies every column's
          inputs host->device (chunked, a copy stream running ahead of the compute stream), re-lays them out on
          the device, forms the Voigt line profiles there (upload_device_phi: the host hands over the damping
          parameters, Doppler widths and vlos the reference's compute_phi consumes), iterates, and reads I, n, dJ,
          dPops back to the host.  e2e_host_phi: the variant that ships host-computed profiles (2.5x the bytes).
  roofline : the fs_gamma_kernel_m launches only: algorithmic bytes per launch (SURVEY.md 8d formula) / their mean
             device time measured with CUDA events around every launch inside the timed region, vs
             MEASURED_PEAKS.json hbm_gbs; roofline.fp64: algorithmic flops vs the fp64 peak measured live.
  arith / exact_arith : the headline runs the library's default arithmetic (contracted); the same resident solve
             with the reference's rounding (MALI_ARITH_EXACT) is reported beside it.
  cpu_baseline : the oracle's C restatement (OpenMP over columns, all host cores) on a bounded sample of the same
                 columns and the same `iters` (rank 0, N = 1 only); reference_numpy: the unmodified reference's own
                 numpy path as timed in the build container (it does not exist on the GPU box).  --impl reference
                 prints that arm alone.
Side sections (N = 1 unless noted): single_column (configs 1/2), to_convergence (the batch run to the reference's
tolerances), response_function (config 3 from host tables), response_function_from_thermodynamic_state and
config4_from_thermodynamic_state (SURVEY.md 8f ranks 1-3 on the device: columns given as cmass, T, ne, nHTot, vturb,
vlos; config 4 by the reference's own jitter recipe with columns 0 and 1 checked against the reference fixtures).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

METRIC = 'MALI ray-depth updates/s'
UNIT = 'updates/s'


def load_base(name):
    from helpers import load_golden
    return load_golden(name)[0]


def algorithmic_bytes_per_column(p):
    """SURVEY.md 8(d): every distinct input read once and every output written once per iteration, fp64."""
    N, S, R = int(p['Nspace']), int(p['Nspect']), int(p['Nrays'])
    tr = np.asarray(p['trans'])
    line_nl = int(tr[tr[:, 3] == 1, 5].sum())
    nl = np.asarray(p['Nlevel'], dtype=np.int64)
    return 8 * (2 * line_nl * R * N + 5 * S * N + int(((2 * nl * nl + 2 * nl + 1) * N).sum()) + S * R)


def algorithmic_flops_per_column(p):
    """SURVEY.md 8(d): F = 2 [31 + 28 A] fp64 operations per unit, A = mean active transitions per wavelength."""
    tr = np.asarray(p['trans'])
    S, R, N = int(p['Nspect']), int(p['Nrays']), int(p['Nspace'])
    abar = float(tr[:, 5].sum()) / S
    return 2.0 * (31.0 + 28.0 * abar) * S * R * N


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(path):
        try:
            return float(json.load(open(path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, pw = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax.append(float(r[1]))
                pw.append(float(r[2]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(nm)
            except Exception:
                continue
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(smax) if smax else None,
                'power_w_max': max(pw) if pw else None, 'samples': len(sm), 'reasons': sorted(reasons)}


def host_threads():
    """Host cores this process may use (launchers such as torchrun export OMP_NUM_THREADS=1: not a core count)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def cpu_oracle_rate(base, ncol_cpu, iters, col0=0):
    """Times the oracle's C restatement (OpenMP over columns) on synthetic columns [col0, col0+ncol_cpu)."""
    from oracle import mali_oracle as mo
    from lightspinner_b200 import synth
    mo.build()
    mo.set_threads(host_threads())
    ctxs = [mo.OracleContext(synth.jitter_problem(base, col0 + c)) for c in range(ncol_cpu)]
    t0 = time.perf_counter()
    mo.iterate_batch(ctxs, iters, start_iter=3)     # start_iter=3: every iteration does formal solution + stat-eq
    dt = time.perf_counter() - t0
    units = ncol_cpu * int(base['Nspect']) * int(base['Nrays']) * int(base['Nspace']) * iters
    return units / dt, dt, mo.max_threads(), ctxs


def run_reference(args, base):
    """--impl reference: the reference's algorithm on the host cores (the oracle port; the reference itself is
    pure Python and is not present on the GPU box).  Rank 0 only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    threads = host_threads()
    # bounded sample: calibrate on one column per thread x 1 iteration, then size the step so that the whole
    # --steps K --warmup W run stays within about a minute of CPU time whatever the box's core count
    cpu_oracle_rate(base, threads, 1)                      # first touch (library load, page faults)
    _, dt_cal, _, _ = cpu_oracle_rate(base, threads, 1)
    budget = 60.0 / (args.steps + 1)
    per_thread = int(budget / max(dt_cal * args.iters, 1e-6))
    ncol_cpu = threads * max(1, min(16, per_thread))
    for _ in range(args.warmup and 1):
        cpu_oracle_rate(base, threads, 1)
    rates, times = [], []
    for _ in range(args.steps):
        r, dt, th, _ = cpu_oracle_rate(base, ncol_cpu, args.iters)
        rates.append(r)
        times.append(dt)
    units = ncol_cpu * int(base['Nspect']) * int(base['Nrays']) * int(base['Nspace']) * args.iters
    value = units * len(times) / sum(times)
    sample = '%d synthetic columns x %d MALI iterations per step (of the %d-column batch)' % (
        ncol_cpu, args.iters, args.ncol * args.gpus)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * sum(times) / len(times),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(args, base),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': th, 'kind': 'port', 'sample': sample,
                         'reference_numpy': reference_numpy_side_number()},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


def reference_numpy_side_number():
    """The UNMODIFIED reference's own numpy / numba path cannot run on the GPU box (it is not there); it was timed in
    the build container where /root/reference is mounted (tools/time_reference_here.py) and is quoted from
    profiles/ as a stated side number next to the C port that is timed live."""
    for name in ('r02_reference_numpy_timing.json', 'r01_reference_numpy_timing.json'):
        try:
            d = json.load(open(os.path.join(ROOT, 'profiles', name)))
            c2 = [c for c in d['cases'] if c['case'].startswith('C2')][0]
            out = {'updates_per_s_one_core': c2['updates_per_s_one_core'], 'case': c2['case'],
                   'where': d['where'], 'source': 'profiles/' + name}
            if 'pool' in d:
                out['pool'] = d['pool']
            return out
        except Exception:
            continue
    return None


def run_lambda_shard(args):
    """BASELINE config 5 (an experiment, not the production path): one stress column -- 10x refined wavelength grid,
    10-point quadrature, 512 depths -- split over the GPUs by wavelength (ranges balanced by work); every iteration exchanges Gamma (one NCCL all-gather of
    [Gamma | dJ] + a fixed-order sum, lambda_shard.GammaExchange).
    A step is one MALI iteration of the column (strong scaling: the column is fixed); a warm-up pass of --warmup
    iterations precedes the --steps timed ones."""
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import lambda_shard_experiment as ls
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    json_fd = None
    if world > 1:
        if os.environ.get('NCCL_DEBUG', '').upper() not in ('INFO', 'TRACE'):
            os.environ['NCCL_DEBUG'] = 'INFO'      # (the GPU boxes preset WARN: a round-2 run logged no rank lines)
        sys.stdout.flush()
        json_fd = os.dup(1)
        os.dup2(2, 1)
    q = ls.build_problem()
    out = ls.run(q, iters=args.steps, warmup=args.warmup)
    if rank == 0:
        line = {'metric': METRIC, 'value': out['updates_per_s'], 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': out['ms_per_iteration'], 'higher_is_better': True,
                'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
                'config': {'workload': 'EXPERIMENT: wavelength-sharded single stress column (BASELINE config 5), Gamma '
                                       'exchange (one NCCL all-gather + fixed-order sum) every iteration', 'Nspect': out['Nspect'], 'Nrays': out['Nrays'],
                           'Nspace': out['Nspace'], 'parallelism': 'wavelengths sharded over %d GPU(s)' % world},
                'lambda_shard': out, 'e2e': None, 'gpu_launches': None}
        if json_fd is not None:
            os.write(json_fd, (json.dumps(line) + '\n').encode())
        else:
            print(json.dumps(line))
    import torch.distributed as dist
    if dist.is_initialized():
        dist.destroy_process_group()


DUMP_BYTES = 60 * 10**6      # array bytes of --dump-outputs: with the .npy headers, under 64 MB


def dump_outputs(out_dir, eng, col_global0, world, rank):
    """Writes what the resident solve hands its caller, in the reference's shapes and float64: emergent intensity
    I [col, Nspect, Nrays], populations n [col, sum Nlevel, Nspace], dJ and dPops [col] with `columns`, the global
    index of each column, and the mean intensity J [col, Nspect, Nspace] with `J_columns`.  At most DUMP_BYTES in all
    (two thirds of it at most for I, n, dJ, dPops, the rest for J, which is 13x larger per column): what does not fit
    is represented by a fixed, seeded sample of the columns.  With several ranks each writes its share of the budget
    as <name>_rank<r>.npy."""
    import torch
    mt, ncol = eng.mt, eng.ncol
    rng = np.random.default_rng(0)

    def sample(bytes_per_col, budget):
        k = min(ncol, budget // bytes_per_col)
        return np.arange(ncol) if k == ncol else np.sort(rng.choice(ncol, k, replace=False))

    budget = DUMP_BYTES // world
    per_col = 8 * (mt.Nspect * mt.Nrays + eng.lay.pops + 3)
    cols = sample(per_col, 2 * budget // 3)
    jcols = sample(8 * (mt.Nspect * mt.Nspace + 1), budget - len(cols) * per_col)
    idx, jidx = (torch.from_numpy(c).to(eng.device) for c in (cols, jcols))
    out = {'columns': torch.from_numpy((col_global0 + cols).astype(np.float64)),
           'I': eng.t_I.view(ncol, mt.Nspect, mt.Nrays).index_select(0, idx),
           'n': eng.t_pops.view(ncol, -1, mt.Nspace).index_select(0, idx),
           'dJ': eng.t_dJ.index_select(0, idx), 'dPops': eng.t_dPops.index_select(0, idx),
           'J_columns': torch.from_numpy((col_global0 + jcols).astype(np.float64)),
           'J': eng.t_J.view(ncol, mt.Nspace, mt.Nspect).index_select(0, jidx).transpose(1, 2)}
    os.makedirs(out_dir, exist_ok=True)
    suffix = '_rank%d' % rank if world > 1 else ''
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + suffix + '.npy'), np.ascontiguousarray(t.cpu().numpy()))


def workload_config(args, base):
    return {
        'workload': 'synthetic 1.5D batch of perturbed FALC columns, CaII + H 6-level active '
                    '(BASELINE config 4 per-GPU share), fixed-length MALI solve',
        'fixture': args.fixture, 'columns_per_gpu': args.ncol, 'columns_total': args.ncol * args.gpus,
        'iters_per_solve': args.iters, 'Nspace': int(base['Nspace']), 'Nrays': int(base['Nrays']),
        'Nspect': int(base['Nspect']), 'Ntrans': int(np.asarray(base['trans']).shape[0]),
        'parallelism': 'columns sharded over %d GPU(s), no data-path collective' % args.gpus,
        'arithmetic': 'fp64; formal-solution kernels in the library default mode (contracted a*b+c, shared reciprocals; '
                      'MALI_ARITH=exact gives the reference\'s rounding, reported as exact_arith)',
        'l2_policy': 'inputs larger than L2 (%.1f GB of per-column tables per GPU)' % (
            args.ncol * algorithmic_bytes_per_column(base) / 1e9),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--ncol', type=int, default=1024, help='columns per GPU')
    ap.add_argument('--iters', type=int, default=16, help='MALI iterations per solve (= per step)')
    ap.add_argument('--fixture', default='c2_falc_cah')
    ap.add_argument('--chunk', type=int, default=512, help='columns per upload chunk in the e2e path')
    ap.add_argument('--e2e-steps', type=int, default=0, help='timed steps of the e2e paths (default: --steps)')
    ap.add_argument('--first-chunk', type=int, default=0,
                    help='e2e path: size of a smaller first chunk (shortens the exposed first host->device copy)')
    ap.add_argument('--sched', default='',
                    help='explicit e2e upload schedule: comma-separated chunk sizes (the last one repeats); overrides '
                         '--chunk / --first-chunk')
    ap.add_argument('--split', type=int, default=0,
                    help='experiment: also time the resident solve issued as K column ranges on K streams')
    ap.add_argument('--workload', default='columns', choices=['columns', 'lambda_shard'],
                    help='columns: the headline column-sharded batch; lambda_shard: BASELINE config 5 experiment, one '
                         'stress column wavelength-sharded over the GPUs with a Gamma all-reduce per iteration')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the timed resident solve computed in its last step to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or args.workload != 'columns'):
        ap.error('--dump-outputs applies to the column workload of --impl ours')
    args.warmup = max(args.warmup, 0)
    base = load_base(args.fixture)

    if args.impl == 'reference':
        run_reference(args, base)
        return
    if args.workload == 'lambda_shard':
        run_lambda_shard(args)
        return

    import torch
    import torch.distributed as dist
    from lightspinner_b200 import synth
    from lightspinner_b200.engine import MaliEngine
    from lightspinner_b200.tables import pack_column

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus and world > 1:
        raise SystemExit('--gpus %d but WORLD_SIZE=%d' % (args.gpus, world))
    if args.gpus > 1 and world == 1:
        raise SystemExit('launch with torch.distributed.run --nproc-per-node %d for --gpus %d' % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    json_fd = None
    if world > 1:
        # NCCL's own log (rank / channel lines: NCCL_DEBUG=INFO unless the launcher asks for INFO / TRACE itself) is written to the
        # process's stdout by NCCL; point fd 1 at stderr for everything but the one JSON line, which goes to the real one
        if os.environ.get('NCCL_DEBUG', '').upper() not in ('INFO', 'TRACE'):
            os.environ['NCCL_DEBUG'] = 'INFO'      # (the GPU boxes preset WARN: a round-2 run logged no rank lines)
        sys.stdout.flush()
        json_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group('nccl', device_id=dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ncol, iters = args.ncol, args.iters
    N, S, R = int(base['Nspace']), int(base['Nspect']), int(base['Nrays'])
    units_per_col_iter = S * R * N
    sched_sizes = [int(x) for x in args.sched.split(',') if x] if args.sched else None
    if sched_sizes:
        args.chunk = max(sched_sizes)
    eng = MaliEngine(base, ncol, device=local, max_upload_chunk=args.chunk)
    lay, mt = eng.lay, eng.mt
    hp = int(lay.hostpack)
    chunk = min(args.chunk, ncol)
    # e2e schedule: [(first column, count)]; an optional small first chunk, then `chunk`-sized ones
    sched, c0 = [], 0
    if sched_sizes:        # growing chunks: only the first (small) upload is exposed, every later one hides behind a solve
        for i, n in enumerate(sched_sizes[:-1]):
            if c0 + n < ncol:
                sched.append((c0, n))
                c0 += n
        chunk = min(sched_sizes[-1], ncol)
    elif 0 < args.first_chunk < chunk and args.first_chunk < ncol:
        sched.append((0, args.first_chunk))
        c0 = args.first_chunk
    while c0 < ncol:
        sched.append((c0, min(chunk, ncol - c0)))
        c0 += chunk
    chunk = max(n for _, n in sched)     # what the staging buffers are sized by
    col_global0 = rank * ncol        # this rank's slice of the global batch

    # ---- build the resident batch: base host pack -> device, jitter on the device, re-layout
    base_pack = torch.from_numpy(pack_column(mt, lay, base)).to(dev)
    staging = [torch.empty(chunk * hp, dtype=torch.float64, device=dev) for _ in range(2)]
    want_e2e = not args.no_e2e
    host_in = torch.empty(ncol * hp, dtype=torch.float64, pin_memory=True) if want_e2e else None
    def fill_batch(keep_host_copy):
        for c0 in range(0, ncol, chunk):
            nc = min(chunk, ncol - c0)
            synth.jitter_staging(staging[0], lay, mt, base_pack, [col_global0 + c for c in range(c0, c0 + nc)])
            eng.repack_from_staging(staging[0], c0, nc)
            if keep_host_copy:
                host_in[c0 * hp:(c0 + nc) * hp].copy_(staging[0][:nc * hp])
        torch.cuda.synchronize(dev)

    fill_batch(want_e2e)
    eng.reset_iteration_state()
    eng.iterate_async(4, tolJ=-1.0)      # brings every column's iteration counter past 3 (test.py:27)

    def solve_resident():
        # the device-resident loop with the convergence test off: `iters` iterations of formal solution + Gamma +
        # statistical equilibrium for every column (the columns' iteration counters are past 3 after the warm-up, so
        # every iteration solves the populations, as in the CPU arm)
        eng.iterate_async(iters, tolJ=-1.0)

    # ---- value: inputs resident in HBM
    for _ in range(args.warmup):
        solve_resident()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = eng.launch_count()
    eng.profile_begin(args.steps * iters)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        solve_resident()
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    fs_ms, fs_n = eng.profile_end()
    launches = eng.launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    finite = bool(torch.isfinite(eng.t_pops).all().item() and torch.isfinite(eng.t_I).all().item())
    if args.dump_outputs:      # before the side sections below run the solve again
        dump_outputs(args.dump_outputs, eng, col_global0, world, rank)
    total_units = world * ncol * units_per_col_iter * iters * args.steps
    value = total_units / (ms * 1e-3)

    # ---- experiment (--split K): the same resident solve issued as K column ranges on K streams, so that one range's
    # DRAM-bound finish kernels (gamma_finish, j_finish, statistical equilibrium: 13 % of an iteration, SMs mostly idle)
    # can run under another range's formal solution; compared with the single-range solve replayed the same way (both as
    # CUDA graphs, the per-launch profiling events off)
    split_side = None
    if args.split > 1:
        try:
            sts = [torch.cuda.Stream(dev) for _ in range(args.split)]
            per = (ncol + args.split - 1) // args.split

            def solve_split():
                cur = torch.cuda.current_stream(dev)
                for i, st_ in enumerate(sts):
                    c0_, nc_ = i * per, min(per, ncol - i * per)
                    if nc_ <= 0:
                        continue
                    st_.wait_stream(cur)
                    with torch.cuda.stream(st_):
                        eng.iterate_async(iters, tolJ=-1.0, col0=c0_, ncol=nc_)
                for st_ in sts:
                    cur.wait_stream(st_)

            def timed(fn):
                for _ in range(max(2, args.warmup)):
                    fn()
                barrier()
                e0.record()
                for _ in range(args.steps):
                    fn()
                e1.record()
                barrier()
                return max_over_ranks(e0.elapsed_time(e1)) / args.steps

            ms_one = timed(solve_resident)
            ms_spl = timed(solve_split)
            split_side = {'ranges': args.split, 'ms_per_step_single_range': ms_one, 'ms_per_step_split': ms_spl,
                          'value_single_range': world * ncol * units_per_col_iter * iters / (ms_one * 1e-3),
                          'value_split': world * ncol * units_per_col_iter * iters / (ms_spl * 1e-3),
                          'finite': bool(torch.isfinite(eng.t_pops).all().item())}
        except Exception as ex:
            split_side = {'error': repr(ex)}

    # ---- the same resident solve with the reference's rounding (MALI_ARITH_EXACT): a side number next to the
    # headline, which runs the library's default arithmetic (contracted; both modes are parity-tested)
    arith_default = eng.arith
    exact_side = None
    try:
        eng.set_arith('exact')
        solve_resident()
        barrier()
        eng.profile_begin(iters)
        e0.record()
        solve_resident()
        e1.record()
        barrier()
        ms_x = max_over_ranks(e0.elapsed_time(e1))
        fx_ms, fx_n = eng.profile_end()
        exact_side = {'arith': 'exact', 'value': world * ncol * units_per_col_iter * iters / (ms_x * 1e-3), 'unit': UNIT,
                      'ms_per_step': ms_x, 'mean_launch_ms': fx_ms / max(fx_n, 1), 'steps': 1}
    except Exception as ex:
        exact_side = {'error': repr(ex)}
    finally:
        eng.set_arith(arith_default)

    # ---- roofline of the dominant kernel
    peak, peak_src = measured_peaks()
    fs_ms_mean = fs_ms / max(fs_n, 1)
    alg_bytes = algorithmic_bytes_per_column(base) * ncol
    achieved = alg_bytes / (fs_ms_mean * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:    # DRAM bytes per launch from the committed ncu capture of this very configuration (profiles/): ncu cannot
        # run inside a timed bench, so this field is read from the capture, not measured in this run
        tj = json.load(open(os.path.join(ROOT, 'profiles', 'traffic_latest.json')))
        if int(tj['ncol']) == ncol and tj['fixture'] == args.fixture:
            traffic = float(tj['traffic_bytes_per_launch'])
            traffic_src = 'from profiles/traffic_latest.json (%s), not measured in this run' % tj.get('source', 'ncu --set full')
    except Exception:
        pass
    roofline = {'kernel': 'fs_gamma_kernel_m<0,1,2> (formal solution + Gamma stage: 3 launches)', 'bound': 'hbm',
                'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                'frac': achieved / peak, 'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peak_src,
                'algorithmic_bytes_per_launch': alg_bytes, 'mean_launch_ms': fs_ms_mean, 'launches_timed': fs_n,
                'share_of_step': fs_ms / ms if ms > 0 else None, 'arith': arith_default,
                'binding_unit': 'L1 data pipe (shared-memory / shuffle wavefronts): 91-93 % of peak in the two large '
                                'kernel classes, dispatch ports 85-90 % (ncu --set full, profiles/r02_v18_fs_kernel_ncu_summary.txt; '
                                'from that capture, not measured in this run)',
                'note': 'neither HBM nor the fp64 pipe binds this path: the per-depth warp-wide Gamma sums saturate the '
                        "SM's L1 data pipe first (DESIGN.md section 4); fp64 CUDA-core work would bind next, well "
                        'before HBM (SURVEY.md 7.3-2)'}
    try:    # the roof that actually binds: unfused fp64 on the CUDA cores, peak measured live
        from lightspinner_b200.engine import fp64_peak
        pk = fp64_peak(local)
        fl = algorithmic_flops_per_column(base) * ncol / (fs_ms_mean * 1e-3)
        roofline['fp64'] = {'achieved': fl / 1e12, 'peak': pk / 1e12, 'unit': 'Tflop/s (unfused mul/add)',
                            'frac': fl / pk, 'algorithmic_flops_per_launch': algorithmic_flops_per_column(base) * ncol,
                            'peak_source': 'measured live (mali_fp64_peak: 8 independent mul+add chains per thread)'}
    except Exception as ex:
        roofline['fp64'] = {'error': repr(ex)}

    # ---- e2e: host buffers -> H2D -> re-layout -> iterate -> D2H, double-buffered over column chunks
    e2e = None
    if want_e2e:
        # [0] copy stream (H2D, re-layout, line profiles), [1] compute stream (the solves), the latter at high priority so
        # that the upload kernels of the next chunk only fill what the solve leaves idle
        streams = [torch.cuda.Stream(dev), torch.cuda.Stream(dev, priority=-1)]
        out_I = torch.empty(ncol * lay.I, dtype=torch.float64, pin_memory=True)
        out_n = torch.empty(ncol * lay.pops, dtype=torch.float64, pin_memory=True)
        out_d = torch.empty(2 * ncol, dtype=torch.float64, pin_memory=True)
        gathered = torch.empty(world * ncol * lay.I, dtype=torch.float64, device=dev) if world > 1 else None

        chunk_done = [None] * len(sched)    # per chunk: its previous solve + read-back finished (buffers are reused)

        def solve_from_host():
            for ci, (c0, nc) in enumerate(sched):
                with torch.cuda.stream(streams[0]):      # copy stream: H2D + re-layout, runs ahead of the solves
                    if chunk_done[ci] is not None:
                        streams[0].wait_event(chunk_done[ci])
                    eng.upload_packed(host_in[c0 * hp:(c0 + nc) * hp], c0, nc, staging=staging[ci & 1])
                    ready = torch.cuda.Event()
                    ready.record()
                with torch.cuda.stream(streams[1]):      # compute stream: the solves, one chunk after the other
                    streams[1].wait_event(ready)
                    eng.iterate_async(iters, tolJ=-1.0, col0=c0, ncol=nc)
                    out_I[c0 * lay.I:(c0 + nc) * lay.I].copy_(eng.t_I[c0 * lay.I:(c0 + nc) * lay.I], non_blocking=True)
                    out_n[c0 * lay.pops:(c0 + nc) * lay.pops].copy_(eng.t_pops[c0 * lay.pops:(c0 + nc) * lay.pops],
                                                                  non_blocking=True)
                    out_d[c0:c0 + nc].copy_(eng.t_dJ[c0:c0 + nc], non_blocking=True)
                    out_d[ncol + c0:ncol + c0 + nc].copy_(eng.t_dPops[c0:c0 + nc], non_blocking=True)
                    chunk_done[ci] = torch.cuda.Event()
                    chunk_done[ci].record()
            for st in streams:
                torch.cuda.current_stream(dev).wait_stream(st)
            if world > 1:     # the path's only exchange: final gather of the emergent intensities (SURVEY.md 8e)
                dist.all_gather_into_tensor(gathered, eng.t_I)

        solve_from_host()
        barrier()
        l0 = eng.launch_count()
        k_e2e = args.e2e_steps if args.e2e_steps > 0 else args.steps
        e0.record()
        for _ in range(k_e2e):
            solve_from_host()
        e1.record()
        barrier()
        ms_e = max_over_ranks(e0.elapsed_time(e1))
        launches_e2e = eng.launch_count() - l0
        e_units = world * ncol * units_per_col_iter * iters * k_e2e
        e2e = {'value': e_units / (ms_e * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': world * ncol * hp * 8,
               'd2h_bytes_per_step': world * (ncol * (lay.I + lay.pops) + 2 * ncol) * 8, 'steps': k_e2e,
               'ms_per_step': ms_e / k_e2e, 'gpu_launches': launches_e2e,
               'finite': bool(np.isfinite(out_I.numpy()).all() and np.isfinite(out_n.numpy()).all()),
               'pipeline': 'column chunks %s; a copy stream (H2D + re-layout) runs ahead of the compute stream' % [n for _, n in sched]}
        if world > 1:
            e2e['gather_bytes_per_step'] = world * ncol * lay.I * 8

    # ---- e2e with the line profiles formed on the device (mali_compute_phi, SURVEY.md 8f rank 2): the host hands over
    # what ComputationalTransition.compute_phi consumes (damping parameters, Doppler widths, vlos) instead of phi, so
    # 60 % fewer bytes cross PCIe and the Voigt evaluation happens inside the timed region.  Columns: same jittered
    # backgrounds / rates; the up/down asymmetry now comes from vlos = 2 km/s * g3 (BASELINE config 4's recipe).
    e2e_dev = None
    if want_e2e and all(k in base for k in ('aDamp', 'vBroad')):
        try:
            hpp = int(lay.hp_phi)
            host_pre = torch.empty(ncol * hpp, dtype=torch.float64, pin_memory=True)
            host_pre.view(ncol, hpp).copy_(host_in.view(ncol, hp)[:, :hpp])
            nT, nA = mt.Ntrans, mt.Natom
            aux_np = np.empty((ncol, nT + nA + 1, N))
            aux_np[:, :nT] = np.asarray(base['aDamp'], dtype=np.float64).reshape(1, nT, N)
            aux_np[:, nT:nT + nA] = np.asarray(base['vBroad'], dtype=np.float64).reshape(1, nA, N)
            for c in range(ncol):
                fv = synth.jitter_factors(col_global0 + c, N)[2]
                aux_np[c, nT + nA] = 2.0e3 * (fv - 1.0) / 0.02
            host_aux = torch.from_numpy(aux_np).pin_memory()
            dev_aux = [torch.empty((chunk, nT + nA + 1, N), dtype=torch.float64, device=dev) for _ in range(2)]
            dev_split = [(torch.empty((chunk, nT, N), dtype=torch.float64, device=dev),
                          torch.empty((chunk, nA, N), dtype=torch.float64, device=dev),
                          torch.empty((chunk, 1, N), dtype=torch.float64, device=dev)) for _ in range(2)]

            def solve_from_host_device_phi():
                for ci, (c0, nc) in enumerate(sched):
                    with torch.cuda.stream(streams[0]):
                        if chunk_done[ci] is not None:
                            streams[0].wait_event(chunk_done[ci])
                        dev_aux[ci & 1][:nc].copy_(host_aux[c0:c0 + nc], non_blocking=True)
                        aD, vB, vL = dev_split[ci & 1]
                        aD[:nc].copy_(dev_aux[ci & 1][:nc, :nT])
                        vB[:nc].copy_(dev_aux[ci & 1][:nc, nT:nT + nA])
                        vL[:nc].copy_(dev_aux[ci & 1][:nc, nT + nA:])
                        eng.upload_packed_device_phi(host_pre[c0 * hpp:(c0 + nc) * hpp], aD, vB, vL, c0, nc,
                                                     staging=staging[ci & 1])
                        ready = torch.cuda.Event()
                        ready.record()
                    with torch.cuda.stream(streams[1]):
                        streams[1].wait_event(ready)
                        eng.iterate_async(iters, tolJ=-1.0, col0=c0, ncol=nc)
                        out_I[c0 * lay.I:(c0 + nc) * lay.I].copy_(eng.t_I[c0 * lay.I:(c0 + nc) * lay.I], non_blocking=True)
                        out_n[c0 * lay.pops:(c0 + nc) * lay.pops].copy_(eng.t_pops[c0 * lay.pops:(c0 + nc) * lay.pops],
                                                                      non_blocking=True)
                        out_d[c0:c0 + nc].copy_(eng.t_dJ[c0:c0 + nc], non_blocking=True)
                        out_d[ncol + c0:ncol + c0 + nc].copy_(eng.t_dPops[c0:c0 + nc], non_blocking=True)
                        chunk_done[ci] = torch.cuda.Event()
                        chunk_done[ci].record()
                for st in streams:
                    torch.cuda.current_stream(dev).wait_stream(st)
                if world > 1:
                    dist.all_gather_into_tensor(gathered, eng.t_I)

            solve_from_host_device_phi()
            barrier()
            l0 = eng.launch_count()
            e0.record()
            for _ in range(k_e2e):
                solve_from_host_device_phi()
            e1.record()
            barrier()
            ms_d = max_over_ranks(e0.elapsed_time(e1))
            # diagnostic: the copy stream's work of one step on its own (H2D + re-layout + line profiles, no solve)
            e0.record()
            for ci, (c0, nc) in enumerate(sched):
                dev_aux[ci & 1][:nc].copy_(host_aux[c0:c0 + nc], non_blocking=True)
                aD, vB, vL = dev_split[ci & 1]
                aD[:nc].copy_(dev_aux[ci & 1][:nc, :nT])
                vB[:nc].copy_(dev_aux[ci & 1][:nc, nT:nT + nA])
                vL[:nc].copy_(dev_aux[ci & 1][:nc, nT + nA:])
                eng.upload_packed_device_phi(host_pre[c0 * hpp:(c0 + nc) * hpp], aD, vB, vL, c0, nc, staging=staging[ci & 1])
            e1.record()
            barrier()
            ms_up = e0.elapsed_time(e1)
            e2e_dev = {'value': e_units / (ms_d * 1e-3), 'unit': UNIT,
                       'h2d_bytes_per_step': world * ncol * (hpp + (nT + nA + 1) * N) * 8,
                       'd2h_bytes_per_step': e2e['d2h_bytes_per_step'], 'steps': k_e2e, 'ms_per_step': ms_d / k_e2e,
                       'gpu_launches': eng.launch_count() - l0, 'upload_only_ms_per_step': ms_up,
                       'finite': bool(np.isfinite(out_I.numpy()).all() and np.isfinite(out_n.numpy()).all()),
                       'pipeline': e2e['pipeline'] + '; line profiles computed on the device (mali_compute_phi) '
                                   'from aDamp / vBroad / vlos'}
        except Exception as ex:
            e2e_dev = {'error': repr(ex)}

    # ---- CPU baseline on the host cores (rank 0, N = 1)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = host_threads()
        cpu_oracle_rate(base, threads, 1, col0=col_global0)     # first touch
        _, dt_cal, _, _ = cpu_oracle_rate(base, threads, 1, col0=col_global0)
        per_thread = int(20.0 / max(dt_cal * iters, 1e-6))          # about 20 s of CPU work
        ncol_cpu = max(1, min(ncol, threads * max(1, min(16, per_thread))))
        rate, dt, th, ctxs = cpu_oracle_rate(base, ncol_cpu, iters, col0=col_global0)
        cpu = {'value': rate, 'unit': UNIT, 'cores': th, 'kind': 'port',
               'sample': '%d of the %d synthetic columns x %d MALI iterations, oracle C restatement with OpenMP '
                         'over columns, %.1f s' % (ncol_cpu, ncol, iters, dt),
               'reference_numpy': reference_numpy_side_number()}

    # ---- BASELINE configs 1/2 on the side: one CaII/FALC column to convergence (latency-bound by construction)
    single = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            c1 = load_base('c1_falc_ca')
            e1 = MaliEngine(c1, 1, device=local)
            e1.upload([c1])
            out = {}
            for mode in ('host_loop', 'device_loop'):
                best = None
                for rep in range(3):              # best of 3: the first device loop also captures its CUDA graph
                    e1.upload([c1])
                    e1.reset_iteration_state()
                    torch.cuda.synchronize(dev)
                    t0 = time.perf_counter()
                    if mode == 'host_loop':       # test.py:20-29 driven from Python, two scalar reads per iteration
                        dJ, dP, it = 1.0, 1.0, 0
                        while (dJ > 2e-3 or dP > 1e-3) and it < 500:
                            it += 1
                            dJ = float(e1.formal_sol_gamma_matrices()[0])
                            if it > 3:
                                dP = float(e1.stat_equil()[0])
                    else:                         # mali_iterate: the loop stays on the device (a replayed CUDA graph);
                        for _ in range(8):        # the host looks at the convergence flag every 16 iterations
                            e1.iterate_async(16)
                            if bool((e1.t_done != 0).all().item()):
                                break
                        it = int(e1.t_iter.cpu()[0])
                    dt = time.perf_counter() - t0
                    best = dt if best is None else min(best, dt)
                out[mode] = {'iterations': it, 'seconds': best}
            single = {'config': 'CaII/FALC single column (test.py problem), to convergence', **out}
            e1.close()
        except Exception as ex:   # never let the side measurement break the main line
            single = {'error': repr(ex)}

    # ---- second half of BASELINE's metric: seconds to converge.  The same batch, from its start populations, run
    # by the device-resident loop until every column meets the reference's tolerances (test.py:20: dJ <= 2e-3 and
    # dPops <= 1e-3, statistical equilibrium from the 4th iteration on); converged columns drop out of the launches.
    conv = None
    if not args.no_cpu:
        try:
            fill_batch(False)
            eng.reset_iteration_state()
            barrier()
            t0 = time.perf_counter()
            n_it = 0
            while n_it < 400:          # 16 iterations per host round trip; converged columns skip their work
                eng.iterate_async(16)
                n_it += 16
                if bool((eng.t_done != 0).all().item()):
                    break
            barrier()
            dt = max_over_ranks(time.perf_counter() - t0)
            eng.raise_on_faults()
            its = eng.t_iter.cpu().numpy().astype(np.int64)
            tot = torch.tensor([float(its.sum()), float(its.max()), float(-its.min()),
                                float((eng.t_done.cpu().numpy() != 0).sum())], dtype=torch.float64, device=dev)
            if world > 1:
                s2 = tot.clone()
                dist.all_reduce(s2, op=dist.ReduceOp.SUM)
                dist.all_reduce(tot, op=dist.ReduceOp.MAX)
                tot[0], tot[3] = s2[0], s2[3]
            conv = {'config': 'the %d-column batch to convergence (dJ <= 2e-3, dPops <= 1e-3), device-resident loop' % (world * ncol),
                    'seconds_to_converge': dt, 'columns': world * ncol, 'columns_converged': int(tot[3].item()),
                    'iterations_max': int(tot[1].item()), 'iterations_min': int(-tot[2].item()),
                    'iterations_mean': float(tot[0].item()) / (world * ncol),
                    'updates_per_s': float(tot[0].item()) * units_per_col_iter / dt}
        except Exception as ex:
            conv = {'error': repr(ex)}

    # ---- BASELINE config 3 on the side: the response-function batch (164 perturbed CaII/FALC columns, warm-started
    # from the converged base populations, response_fn.py:23-39), columns sharded over the ranks, each column run to
    # the reference's convergence tolerance by the device-resident loop.  The columns cycle through the two
    # response-function problems generated with the unmodified reference (tests/golden/rf_*.npz), so the iteration
    # counts and emergent intensities can be checked against the reference's own.
    rf = None
    if not args.no_cpu:
        try:
            from helpers import load_golden
            from lightspinner_b200.sharding import shard_range
            gold = [load_golden(nm) for nm in ('rf_k40p', 'rf_k10m')]
            n_rf = 164
            lo, cnt = shard_range(n_rf, world, rank)
            hi = lo + cnt
            mine = [gold[c % 2] for c in range(lo, hi)]
            e3 = MaliEngine(gold[0][0], max(len(mine), 1), device=local)
            # host side of a column: its block without the line profiles + what compute_phi consumes (the profiles
            # are formed on the device, as in the headline e2e path)
            hp3 = int(e3.lay.hp_phi)
            packs = [torch.from_numpy(pack_column(e3.mt, e3.lay, g[0], with_phi=False)) for g in gold]
            nmine, N3 = max(len(mine), 1), int(gold[0][0]['Nspace'])
            host3 = torch.empty(nmine * hp3, dtype=torch.float64, pin_memory=True)
            aux3 = [torch.empty((nmine,) + np.asarray(gold[0][0][k]).reshape(-1, N3).shape, dtype=torch.float64).pin_memory()
                    for k in ('aDamp', 'vBroad', 'vlos')]
            for i in range(len(mine)):
                host3[i * hp3:(i + 1) * hp3].copy_(packs[(lo + i) % 2])
                for t, k in zip(aux3, ('aDamp', 'vBroad', 'vlos')):
                    t[i].copy_(torch.from_numpy(np.asarray(gold[(lo + i) % 2][0][k], dtype=np.float64).reshape(-1, N3)))
            dev3 = [torch.empty_like(t, device=dev) for t in aux3]
            times, its = [], None
            for rep in range(3):
                barrier()
                t0 = time.perf_counter()
                if mine:
                    for t, h in zip(dev3, aux3):
                        t.copy_(h, non_blocking=True)
                    for c0 in range(0, len(mine), 64):      # H2D + re-layout + profiles + solve, as a user runs it
                        nc = min(64, len(mine) - c0)
                        e3.upload_packed_device_phi(host3[c0 * hp3:(c0 + nc) * hp3], dev3[0][c0:c0 + nc],
                                                    dev3[1][c0:c0 + nc], dev3[2][c0:c0 + nc], c0, nc)
                    e3.reset_iteration_state()
                    for _ in range(8):                      # 8 iterations per host round trip
                        e3.iterate_async(8, ncol=len(mine))
                        if bool((e3.t_done[:len(mine)] != 0).all().item()):
                            break
                barrier()
                times.append(max_over_ranks(time.perf_counter() - t0))
            if mine:
                e3.raise_on_faults(0, len(mine))
            ok = True
            if mine:
                its = e3.t_iter.cpu().numpy()[:len(mine)]
                for i in range(len(mine)):
                    g = mine[i][1]
                    ok = ok and int(its[i]) == int(g['niter'])
                    if i < 2:
                        ref_I = np.asarray(g['final_I'])
                        ok = ok and float(np.max(np.abs(e3.I(i) - ref_I) / np.abs(ref_I))) < 1e-10
            okt = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(okt, op=dist.ReduceOp.MIN)
            g0 = gold[0][0]
            units_rf = sum(int(gold[c % 2][1]['niter']) for c in range(n_rf)) * int(g0['Nspect']) * int(g0['Nrays']) * int(g0['Nspace'])
            rf = {'config': 'response-function batch: 164 perturbed CaII/FALC columns (T[k] +/- 25 K, warm start), '
                            'to convergence, host buffers -> H2D -> line profiles on the device -> solve (device-resident loop)',
                  'columns': n_rf, 'columns_this_rank': len(mine), 'seconds_to_converge': min(times),
                  'seconds_all_reps': times, 'updates_per_s': units_rf / min(times),
                  'iterations': sorted(set(int(x) for x in its)) if its is not None else [],
                  'matches_reference': bool(okt.item() > 0.5),
                  'check': 'iteration count of every column == the reference\'s; I(lambda, mu) of the first two '
                           'columns within 1e-10 of the reference\'s converged output (tests/golden/rf_*.npz)'}
            e3.close()
        except Exception as ex:
            rf = {'error': repr(ex)}

    # ---- BASELINE config 3 from the thermodynamic state alone (SURVEY.md 8f ranks 1-3 on the device): the 164 columns
    # of response_fn.py -- FALC with T[k] +- 25 K -- given as (column mass, T, ne, nHTot, vturb, vlos) per column; the
    # EOS, background opacities, heights, LTE populations, collisional rates, g_ij and line profiles are formed on the
    # GPU (mali_background, mali_setup_columns, mali_compute_phi), then the warm-started columns are solved.  Set-up
    # and solve seconds are reported separately; the reference spends ~3.4 s of Python per column on this set-up.
    rf_thermo = None
    if not args.no_cpu:
        try:
            from helpers import load_golden, load_setup_inputs
            from lightspinner_b200.atoms import AtomTables
            from lightspinner_b200.eos import EosTables
            from lightspinner_b200.sharding import shard_range
            zeos = np.load(os.path.join(ROOT, 'tests', 'golden', 'eos.npz'))
            c1p, c1r = load_golden('c1_falc_ca')
            rfg = {40: load_golden('rf_k40p'), -10: load_golden('rf_k10m')}
            atoms, _ = load_setup_inputs('c1_falc_ca')
            N1 = int(c1p['Nspace'])
            cols = [(k, s) for k in range(N1) for s in (+1, -1)]          # response_fn.py:24: 164 perturbed columns
            lo, cnt = shard_range(len(cols), world, rank)
            mine = cols[lo:lo + cnt]
            base1 = {k: c1p[k] for k in ('Nspace', 'Nrays', 'Nspect', 'wavelength', 'muz', 'wmu', 'Nlevel', 'trans',
                                         'linepar', 'alpha', 'vturb', 'vlos', 'atom_names')}
            probs = []
            for k, sgn in mine:
                q = dict(base1)
                T = np.array(zeos['falc_T'])
                T[k] += 25.0 * sgn
                q['temperature'], q['ne'], q['nHTot'], q['cmass'] = T, zeos['falc_ne'], zeos['falc_nHTot'], zeos['falc_cmass']
                q['nTotal'] = (atoms['CA']['abundance'] * q['nHTot'])[None, :]
                # the damping parameters are the model objects' business (atomic_model.py:491-502, host): the two columns
                # that exist as reference fixtures carry their own, the others the unperturbed column's
                key = k * sgn
                q['aDamp'] = rfg[key][0]['aDamp'] if key in rfg else c1p['aDamp']
                q['n'] = c1r['final_n']                                   # warm start, response_fn.py:33
                probs.append(q)
            e4 = MaliEngine(c1p, max(len(probs), 1), device=local, max_upload_chunk=max(len(probs), 1))
            e4.set_eos(EosTables.from_arrays(zeos))
            e4.set_atoms(AtomTables.from_arrays([dict(atoms['CA'])]))
            t_setup, t_solve = [], []
            for rep in range(3):
                barrier()
                t0 = time.perf_counter()
                if probs:
                    e4.upload_thermo(probs, start_from_lte=False)
                torch.cuda.synchronize(dev)
                t1 = time.perf_counter()
                if probs:
                    e4.reset_iteration_state()
                    for _ in range(8):
                        e4.iterate_async(8, ncol=len(probs))
                        if bool((e4.t_done[:len(probs)] != 0).all().item()):
                            break
                barrier()
                t_setup.append(max_over_ranks(t1 - t0))
                t_solve.append(max_over_ranks(time.perf_counter() - t1))
            ok, its4 = True, []
            if probs:
                e4.raise_on_faults(0, len(probs))
                its4 = e4.t_iter.cpu().numpy()[:len(probs)]
                for i, (k, sgn) in enumerate(mine):
                    if k * sgn in rfg:       # the two columns the reference itself ran: same count, same I to 1e-10
                        g = rfg[k * sgn][1]
                        ok = ok and int(its4[i]) == int(g['niter'])
                        ok = ok and float(np.max(np.abs(e4.I(i) - g['final_I']) / np.abs(g['final_I']))) < 1e-10
            okt = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(okt, op=dist.ReduceOp.MIN)
            rf_thermo = {'config': 'response-function batch from the thermodynamic state alone: 164 columns (FALC, T[k] +- 25 K) '
                                   'given as column mass, T, ne, nHTot, vturb, vlos; EOS, background opacity, heights, LTE '
                                   'populations, collisional rates and line profiles formed on the device',
                         'columns': len(cols), 'columns_this_rank': len(probs), 'setup_seconds': min(t_setup),
                         'solve_seconds': min(t_solve), 'seconds_total': min(a + b for a, b in zip(t_setup, t_solve)),
                         'setup_seconds_all_reps': t_setup, 'solve_seconds_all_reps': t_solve,
                         'iterations': sorted(set(int(x) for x in its4)),
                         'matches_reference': bool(okt.item() > 0.5),
                         'check': 'columns (k=40, +25 K) and (k=10, -25 K) against the reference fixtures: iteration count and '
                                  'I(lambda, mu) within 1e-10',
                         'reference_setup_seconds_per_column': 3.4}
            e4.close()
        except Exception as ex:
            rf_thermo = {'error': repr(ex)}

    # ---- BASELINE config 4 by its own recipe (SURVEY.md 8d item 4), from the thermodynamic state: every column is FALC
    # with T *= exp(0.01 g1), ne *= exp(0.05 g2), vlos = 2 km/s g3 (lightspinner_b200.synth.jitter_atmosphere -- bit
    # identical to the reference's columns 0 and 1), set up entirely on the device (EOS, background, heights, LTE
    # populations, collisional rates, profiles) and run to convergence by the device-resident loop.  Columns 0 and 1
    # exist as reference fixtures (tests/golden/c2v_jitter_cah_*.npz): their iteration counts and converged I, n are
    # checked against the reference's inside this run.  (The lines' damping parameters are host inputs: columns 0 and 1
    # carry their own, the others the unperturbed column's.)
    c4 = None
    if not args.no_cpu:
        try:
            from helpers import load_golden, load_setup_inputs
            from lightspinner_b200.atoms import AtomTables
            from lightspinner_b200.eos import EosTables
            zeos = np.load(os.path.join(ROOT, 'tests', 'golden', 'eos.npz'))
            atoms4, _ = load_setup_inputs('c2_falc_cah')
            fx = {c: load_golden('c2v_jitter_cah_%d' % c) for c in (0, 1)}
            n4 = min(ncol, 1024)
            names4 = [str(x).strip().upper() for x in base['atom_names']]
            ab4 = [atoms4[nm]['abundance'] for nm in names4]
            probs = []
            for c in range(n4):
                gc = col_global0 + c
                T4, ne4, vl4 = synth.jitter_atmosphere(gc, zeos['falc_T'], zeos['falc_ne'])
                probs.append(dict(temperature=T4, ne=ne4, vlos=vl4, nHTot=zeos['falc_nHTot'], cmass=zeos['falc_cmass'],
                                  vturb=base['vturb'], nTotal=np.stack([a * zeos['falc_nHTot'] for a in ab4]),
                                  aDamp=fx[gc][0]['aDamp'] if gc in fx else base['aDamp']))
            e5 = MaliEngine(base, n4, device=local, max_upload_chunk=256)
            e5.set_eos(EosTables.from_arrays(zeos))
            e5.set_atoms(AtomTables.from_arrays([dict(atoms4[nm]) for nm in names4]))
            t_setups = []
            for rep in range(2):      # the first call also allocates the engine's staging / pinned buffers
                barrier()
                t0 = time.perf_counter()
                e5.upload_thermo(probs)
                torch.cuda.synchronize(dev)
                t_setups.append(max_over_ranks(time.perf_counter() - t0))
            t_setup = min(t_setups)
            e5.reset_iteration_state()
            barrier()
            t0 = time.perf_counter()
            for _ in range(25):
                e5.iterate_async(16)
                if bool((e5.t_done != 0).all().item()):
                    break
            barrier()
            t_solve = max_over_ranks(time.perf_counter() - t0)
            e5.raise_on_faults()
            its5 = e5.t_iter.cpu().numpy().astype(np.int64)
            ok, detail = True, {}
            for c in range(n4):
                gc = col_global0 + c
                if gc in fx:
                    r5 = fx[gc][1]
                    eI = float(np.max(np.abs(e5.I(c) - r5['final_I']) / np.abs(r5['final_I'])))
                    en = float(np.max(np.abs(e5.n(c) - r5['final_n']) / np.abs(r5['final_n'])))
                    detail['column_%d' % gc] = {'iterations': int(its5[c]), 'reference_iterations': int(r5['niter']),
                                                'rel_err_I': eI, 'rel_err_n': en}
                    ok = ok and int(its5[c]) == int(r5['niter']) and eI < 1e-10 and en < 1e-10
            c4 = {'config': 'BASELINE config 4 by its own recipe: %d columns per GPU from (cmass, T, ne, nHTot, vturb, vlos), '
                            'device-side set-up, to convergence' % n4,
                  'columns_per_gpu': n4, 'setup_seconds': t_setup, 'setup_seconds_all_reps': t_setups,
                  'seconds_to_converge': t_solve,
                  'iterations_min': int(its5.min()), 'iterations_max': int(its5.max()), 'iterations_mean': float(its5.mean()),
                  'updates_per_s': float(its5.sum()) * units_per_col_iter * world / t_solve,
                  'reference_columns': detail, 'matches_reference': bool(ok) if detail else None}
            e5.close()
        except Exception as ex:
            c4 = {'error': repr(ex)}

    # headline e2e: the path a user of the batch API takes -- upload_device_phi (the host hands over what the
    # reference's compute_phi consumes; profiles are formed on the device inside the timed region).  The variant that
    # ships host-computed profiles over PCIe is reported beside it.
    e2e_host = e2e
    if e2e_dev is not None and 'value' in e2e_dev:
        e2e, e2e_host = e2e_dev, e2e

    if rank == 0:
        cfg = workload_config(args, base)
        line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'config': cfg, 'clocks': clocks,
                'e2e': e2e, 'e2e_host_phi': e2e_host, 'gpu_launches': launches, 'roofline': roofline, 'cpu_baseline': cpu,
                'single_column': single, 'to_convergence': conv, 'response_function': rf,
                'response_function_from_thermodynamic_state': rf_thermo, 'config4_from_thermodynamic_state': c4,
                'results_finite': finite,
                'arith': arith_default, 'exact_arith': exact_side}
        if split_side is not None:
            line['split_streams_experiment'] = split_side
        if json_fd is not None:
            sys.stdout.flush()
            os.write(json_fd, (json.dumps(line) + '\n').encode())
        else:
            print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
