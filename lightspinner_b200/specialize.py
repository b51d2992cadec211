"""Model-specific kernel specialisation.

The fast formal-solution kernels are specialised on the *structure* of a wavelength tile (which transitions overlap
it and which atomic levels they share; csrc/mali_fs_spec.cuh).  libmali_b200.so ships instances for the models of the
committed fixtures; any other model still runs -- on the generic kernel, a few times slower.  This module closes the
gap when nvcc is available: it lists the tile structures of a model, writes an instance file for them and builds a
model-specific variant of the library (same C ABI), cached under a hash of its structures, sources and compiler
options in a private per-user temporary directory (the package tree is left as the build left it; it may be read-only).

    lib_path = specialize.library_for(problem)      # None when nothing had to be (or could be) built
    eng = MaliEngine(problem, ncol, specialize=True)   # does it for you
"""
import fcntl
import hashlib
import os
import stat
import sys
import tempfile

import numpy as np

from . import build as _build

MAXS = 8


def tile_structures(p):
    """Structure keys of every tile of the model, in the textual form mali_api.cu's structure_key() produces."""
    tr = np.asarray(p['trans']).reshape(-1, 6)
    Nspect, Nrays = int(p['Nspect']), int(p['Nrays'])
    Nlevel = np.asarray(p['Nlevel'], dtype=int)
    lvloff = np.concatenate([[0], np.cumsum(Nlevel)])
    natom = len(Nlevel)
    Lw = 32 // Nrays
    pw = (1 + int(Nlevel.sum()) + 3) // 4 * 4        # width of a popsT row (csrc/mali_types.cuh)
    keys = []
    for ti in range((Nspect + Lw - 1) // Lw):
        la0, la1 = ti * Lw, min(Nspect, ti * Lw + Lw)
        slots = [t for t in range(len(tr)) if tr[t, 4] < la1 and tr[t, 4] + tr[t, 5] > la0]
        if len(slots) > MAXS or natom > 4:
            continue
        lev = {}
        kind, atom, lvI, lvJ, rowI, rowJ = ([0] * MAXS for _ in range(6))
        for q, t in enumerate(slots):
            a, i, j, isLine = (int(v) for v in tr[t, :4])
            for lv in (i, j):
                lev.setdefault((a, lv), len(lev))
            kind[q], atom[q] = isLine, a
            lvI[q], lvJ[q] = lev[(a, i)], lev[(a, j)]
            rowI[q], rowJ[q] = int(lvloff[a] + i), int(lvloff[a] + j)
        arr = lambda x: '{' + ','.join(str(v) for v in x) + '}'
        keys.append('{%d,%d,%d,%d,%s,%s,%s,%s,%s,%s,%d,%d}' % (Lw, len(slots), natom, len(lev), arr(kind), arr(atom),
                                                             arr(lvI), arr(lvJ), arr(rowI), arr(rowJ), Nrays, pw))
    return keys


def write_instances(keys, path, comment=''):
    nslot = lambda k: int(k[1:].split(',')[1])
    keys = sorted(set(keys), key=lambda k: (-nslot(k), k))
    with open(path, 'w') as f:
        f.write('// generated -- %d tile structures %s\n' % (len(keys), comment))
        for q, k in enumerate(keys):
            f.write('MALI_SPEC(%d, "%s", %s)\n' % (q, k, k[1:-1]))
    return keys


def stock_keys():
    inc = os.path.join(_build.CSRC, 'spec_instances.inc')
    keys = []
    for line in open(inc):
        if line.startswith('MALI_SPEC('):
            keys.append(line.split('"')[1])
    return keys


def cache_dir():
    """Per-user directory of the model-specific libraries built at run time.  Libraries found there are loaded, so
    it must be this user's own private directory (a predictable name in a shared temporary directory)."""
    d = os.path.join(tempfile.gettempdir(), 'lightspinner_b200-%d' % os.getuid())
    try:
        os.mkdir(d, 0o700)
    except FileExistsError:
        pass
    st = os.lstat(d)
    if not stat.S_ISDIR(st.st_mode) or st.st_uid != os.getuid() or st.st_mode & 0o077:
        raise RuntimeError('%s is not a private directory of this user: refusing to load libraries from it' % d)
    return d


def variant_tag(keys):
    """Content hash of everything a model-specific library is built from: its tile structures, the kernel sources,
    the build script and the compiler with its options.  Checkouts of different commits never share a library."""
    h = hashlib.sha256()
    for part in ['\n'.join(keys), _build.nvcc_path(), ' '.join(_build.NVCC_FLAGS)]:
        h.update(part.encode() + b'\0')
    for f in [os.path.join(_build.CSRC, d) for d in _build.DEPS] + [_build.__file__]:
        with open(f, 'rb') as src:
            h.update(src.read() + b'\0')
    return h.hexdigest()[:16]


def library_for(problem, verbose=False):
    """Path of a library whose kernel instances cover every tile structure of `problem`; builds it with nvcc when
    the stock library does not (returns None if nothing is needed, or if nvcc is missing)."""
    need = set(tile_structures(problem))
    have = set(stock_keys())
    if need <= have:
        return None
    try:
        _build.nvcc_path()
    except RuntimeError:
        return None
    keys = sorted(need | have)
    tag = variant_tag(keys)
    cache = cache_dir()
    lib = os.path.join(cache, 'libmali_b200_spec_%s.so' % tag)
    with open(lib + '.lock', 'w') as lock:      # the ranks of one job ask for the same library at the same time
        fcntl.flock(lock, fcntl.LOCK_EX)
        if os.path.isfile(lib):                 # the name is the hash of all its inputs; build() writes it atomically
            return lib
        inc = os.path.join(cache, 'spec_instances_%s.inc' % tag)
        write_instances(keys, inc, '(stock + model-specific)')
        if verbose:
            sys.stderr.write('lightspinner_b200: building %s for %d new tile structures\n'
                             % (os.path.basename(lib), len(need - have)))
        return _build.build(force=True, verbose=False, lib=lib, spec_inc=inc,
                            objdir=os.path.join(cache, '_obj', os.path.basename(lib)))
