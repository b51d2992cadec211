"""The C-ABI shared library loads on a machine without a GPU and exports every entry point that include/mali_b200.h
declares; compute entry points must fail loudly (no CPU fallback) when there is no CUDA device."""
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    text = open(os.path.join(ROOT, 'include', 'mali_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(mali_[a-z0-9_]+)\s*\(', text)))


def test_header_and_library_agree():
    from lightspinner_b200 import _capi, build
    build.build()
    L = _capi.load()
    names = declared_functions()
    assert len(names) >= 15
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing
    assert set(_capi.EXPORTS) <= set(names)


def test_host_helper_planck_matches_oracle(oracle):
    """mali_planck_bc is host code (libm exp, as numba calls it): bit-identical to the oracle's planck."""
    from lightspinner_b200 import tables
    wav = np.array([30.0, 121.567, 393.366, 500.0, 854.209, 868.186])
    T = np.array([9000.0, 9400.0])
    out = tables.planck_bc(wav, T)
    for i, w in enumerate(wav):
        assert out[i, 0] == oracle.planck(T[0], w) and out[i, 1] == oracle.planck(T[1], w)


NO_GPU_CHECK = '''
import ctypes as C
import pytest
from helpers import load_golden
from lightspinner_b200.engine import MaliEngine
p, _ = load_golden('c1_falc_ca')
with pytest.raises(RuntimeError, match='no CPU fallback'):
    MaliEngine(p, 1)
from lightspinner_b200 import _capi
L = _capi.load()
assert L.mali_device_count() == 0
h = C.c_void_p()
from lightspinner_b200.tables import ModelTables
desc = ModelTables(p).desc()
assert L.mali_model_create(C.byref(desc), 0, C.byref(h)) != 0
assert b'cuda' in L.mali_last_error().lower() or len(L.mali_last_error()) > 0
print('NO_GPU_CHECK_OK')
'''


def test_no_cpu_fallback():
    """Run in a process that sees no CUDA device (CUDA_VISIBLE_DEVICES=''), so that it also runs on a GPU machine."""
    path = [ROOT, os.path.join(ROOT, 'tests'), os.environ.get('PYTHONPATH')]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='', PYTHONPATH=os.pathsep.join(p for p in path if p))
    cmd = [sys.executable] + (['-s'] if sys.flags.no_user_site else []) + ['-c', NO_GPU_CHECK]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
    assert res.returncode == 0 and 'NO_GPU_CHECK_OK' in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]
