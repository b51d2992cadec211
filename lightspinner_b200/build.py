"""In-tree build of libmali_b200.so with nvcc for sm_100a (no torch, no JIT cache).

    python -m lightspinner_b200.build [--force] [--verbose]

--fmad=false is part of the numerical contract (see csrc/mali_device.cuh); -lineinfo keeps the ncu source page
usable.  Seven translation units -- the host API with the small kernels, and one per register class and arithmetic
mode of the structure-specialised formal-solution kernels -- are compiled in parallel and linked into one shared library, which
lives in lightspinner_b200/_lib/ (git-ignored).  The checked build (CHECK_LIB, -DMALI_CHECK) is built next to it.
"""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIBDIR = os.path.join(HERE, '_lib')
LIB = os.path.join(LIBDIR, os.environ.get('MALI_LIB_NAME', 'libmali_b200.so'))
# every lane verifies each record the TMA ring delivers against global memory (tests/test_gpu_checked_build.py)
CHECK_LIB = os.path.join(LIBDIR, 'libmali_b200_check.so')
CHECK_DEFINES = ['MALI_CHECK=1']
DEPS = ['mali_api.cu', 'mali_fs_class.cu', 'mali_fs_launch.h', 'mali_kernels.cuh', 'mali_device.cuh', 'mali_types.cuh',
        'exp_table.inc', 'mali_solve.h', 'mali_voigt.h', 'mali_fs_spec.cuh', 'mali_fs_step.inc', 'spec_instances.inc',
        'mali_rays.cuh', 'mali_rates.cuh', 'mali_perturb.cuh', 'mali_eos.h', 'mali_eos_tables.inc',
        os.path.join('..', '..', 'include', 'mali_b200.h')]

EXTRA = os.environ.get('MALI_NVCC_EXTRA', '').split()
NVCC_FLAGS = EXTRA + ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '--fmad=false', '-std=c++20',
                      '-Xcompiler', '-fPIC', '-Xcompiler', '-ffp-contract=off', '-Xcompiler', '-O2']
# (mali_voigt.h is reached by every unit through mali_device.cuh, but only compute_phi_kernel in mali_kernels.cuh and
# rays_kernel in mali_rays.cuh call it)
API_ONLY = {'mali_api.cu', 'mali_kernels.cuh', 'mali_rays.cuh', 'mali_rates.cuh', 'mali_perturb.cuh', 'mali_eos.h',
            'mali_eos_tables.inc', 'mali_voigt.h', os.path.join('..', '..', 'include', 'mali_b200.h')}
FS_ONLY = {'mali_fs_class.cu', 'mali_fs_step.inc', 'spec_instances.inc'}
# (object name, source, extra flags)
UNITS = [('fs1', 'mali_fs_class.cu', ['-DMALI_CLS=1']), ('fs1f', 'mali_fs_class.cu', ['-DMALI_CLS=1', '-DMALI_FAST=1']),
         ('fs2', 'mali_fs_class.cu', ['-DMALI_CLS=2']), ('fs2f', 'mali_fs_class.cu', ['-DMALI_CLS=2', '-DMALI_FAST=1']),
         ('fs0', 'mali_fs_class.cu', ['-DMALI_CLS=0']), ('fs0f', 'mali_fs_class.cu', ['-DMALI_CLS=0', '-DMALI_FAST=1']),
         ('api', 'mali_api.cu', [])]


def nvcc_path():
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError('nvcc not found')


def stale(lib=LIB):
    if not os.path.isfile(lib):
        return True
    t = os.path.getmtime(lib)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS) or os.path.getmtime(__file__) > t


def build(force=False, verbose=False, lib=None, spec_inc=None, defines=(), objdir=None):
    """Build libmali_b200.so, or (lib, spec_inc / defines given) a variant with other kernel instances / options.
    objdir: where the objects are kept for incremental builds (default lightspinner_b200/_obj/<library name>)."""
    lib = LIB if lib is None else lib
    if lib in (LIB, CHECK_LIB) and not force and not stale(lib):
        return lib
    os.makedirs(os.path.dirname(lib), exist_ok=True)
    extra = (['-DMALI_SPEC_INC="%s"' % spec_inc] if spec_inc else []) + ['-D' + d for d in defines]
    nvcc = nvcc_path()
    ccbin = ['-ccbin', '/usr/bin/g++' if os.path.isfile('/usr/bin/g++') else 'g++']
    if objdir is None:
        objdir = os.path.join(HERE, '_obj', os.path.basename(lib))
    os.makedirs(objdir, exist_ok=True)

    class _Ok:
        returncode, stdout, stderr = 0, '', ''

    def compile_unit(u):
        name, src, flags = u
        obj = os.path.join(objdir, name + '.o')
        cmd = [nvcc] + NVCC_FLAGS + extra + flags + (['-Xptxas', '-v'] if verbose else []) + ccbin + \
            ['-c', '-o', obj, os.path.join(CSRC, src)]
        # incremental: an object is kept while none of ITS sources (and no option) changed
        deps = [d for d in DEPS if d not in (FS_ONLY if name == 'api' else API_ONLY)]
        stamp = obj + '.cmd'
        if (os.path.isfile(obj) and os.path.isfile(stamp) and open(stamp).read() == ' '.join(cmd)
                and all(os.path.getmtime(os.path.join(CSRC, d)) <= os.path.getmtime(obj) for d in deps)
                and (not spec_inc or os.path.getmtime(spec_inc) <= os.path.getmtime(obj))):
            return obj, _Ok
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode == 0:
            open(stamp, 'w').write(' '.join(cmd))
        return obj, res

    with ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
        results = list(ex.map(compile_unit, UNITS))
    ok = True
    for obj, res in results:
        if verbose or res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
        ok = ok and res.returncode == 0
    if not ok:
        raise RuntimeError('nvcc failed building %s' % os.path.basename(lib))
    cmd = [nvcc, '-shared', '-cudart', 'static', '-gencode', 'arch=compute_100a,code=sm_100a'] + ccbin + \
        ['-o', lib + '.tmp'] + [obj for obj, _ in results]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError('link failed for %s' % os.path.basename(lib))
    os.replace(lib + '.tmp', lib)
    return lib


def build_checked(force=False, verbose=False):
    """Build CHECK_LIB (same ABI as libmali_b200.so, every ring delivery verified on the device)."""
    return build(force=force, verbose=verbose, lib=CHECK_LIB, defines=CHECK_DEFINES)


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
    print(build_checked(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
