"""Response functions of the emergent spectrum (response_fn.py; definition in include/mali_b200.h and DESIGN.md): the
host side of MaliEngine.compute_response.

For every depth k of a base column and s = -1, +1 the perturbed column is the base with X[k] -> X[k] + s * step, X one
of RESPONSE_PARAMS; its damping at k is row k of aDamp_minus / aDamp_plus (the damping of the base atmosphere with X
shifted by -step / +step everywhere: damping is local in depth), elsewhere the base's; a temperature change at
k >= Nspace - 2 changes the boundary Planck pair as well.  perturbed_problem builds such a column as an upload_thermo
problem dict: it is the reference the device path (mali_perturb_columns) is tested against.
"""
from dataclasses import dataclass

import numpy as np

RESPONSE_PARAMS = ('temperature', 'vturb', 'vlos')
BASE_KEYS = ('temperature', 'ne', 'nHTot', 'vturb', 'vlos', 'nTotal', 'aDamp')


def base_arrays(base, Nspace, Natom, Ntrans):
    """The base column's upload_thermo inputs as float64 arrays of the model's shapes (ValueError naming what is missing
    or misshapen)."""
    missing = [k for k in BASE_KEYS if k not in base]
    if missing or ('cmass' not in base and 'height' not in base):
        raise ValueError('base needs %s and cmass or height: missing %s'
                         % (', '.join(BASE_KEYS), missing + ([] if 'cmass' in base or 'height' in base else ['cmass / height'])))
    shapes = dict(nTotal=(Natom, Nspace), aDamp=(Ntrans, Nspace))
    out = {}
    for k in BASE_KEYS + tuple(x for x in ('cmass', 'height') if x in base):
        a = np.asarray(base[k], dtype=np.float64)
        want = shapes.get(k, (Nspace,))
        if a.size != int(np.prod(want)):
            raise ValueError('base[%r] must be %s, got shape %s' % (k, list(want), a.shape))
        out[k] = np.ascontiguousarray(a.reshape(want))
    return out


def response_args(param, step, aDamp_minus, aDamp_plus, depths, Nspace, Ntrans):
    """Validated (step, depths [ndepth] int32, aDamp_minus, aDamp_plus) of a compute_response call; the damping arrays are
    None for 'vlos', which does not use them."""
    if param not in RESPONSE_PARAMS:
        raise ValueError('param must be one of %s, got %r' % (', '.join(RESPONSE_PARAMS), param))
    try:
        step = float(step)
    except (TypeError, ValueError):
        raise ValueError('step must be a finite number > 0, got %r' % (step,)) from None
    if not (np.isfinite(step) and step > 0.0):
        raise ValueError('step must be a finite number > 0, got %r' % step)
    if depths is None:
        d = np.arange(Nspace, dtype=np.int64)
    else:
        d = np.asarray(depths)
        if d.ndim == 0:
            d = d.reshape(1)
        if d.ndim != 1 or d.shape[0] == 0 or not np.issubdtype(d.dtype, np.integer):
            raise ValueError('depths must be a non-empty 1-D sequence of integers, got %r' % (depths,))
        if ((d < 0) | (d >= Nspace)).any():
            raise ValueError('depths must lie in [0, %d): got %s' % (Nspace, d[(d < 0) | (d >= Nspace)][:8].tolist()))
        if np.unique(d).shape[0] != d.shape[0]:
            raise ValueError('depths must be unique')
    damp = [None, None]
    if param != 'vlos':
        for q, (name, a) in enumerate((('aDamp_minus', aDamp_minus), ('aDamp_plus', aDamp_plus))):
            if a is None:
                raise ValueError('%s [Ntrans, Nspace] is required for param=%r: the damping of the base atmosphere with '
                                 '%s shifted by %sstep' % (name, param, param, '-' if q == 0 else '+'))
            a = np.asarray(a, dtype=np.float64)
            if a.shape != (Ntrans, Nspace):
                raise ValueError('%s must be [Ntrans, Nspace] = %s, got shape %s' % (name, [Ntrans, Nspace], a.shape))
            damp[q] = a
    return step, d.astype(np.int32), damp[0], damp[1]


def perturbed_value(x0, step, k, s):
    """X[k] + s * step, the perturbed column's value at its depth (the same expression on every path)."""
    return x0[k] + s * step


def perturbed_bbc(wavelength, temperature, param, step, k, s):
    """[Nspect, 2] boundary Planck pair of the perturbed column when it differs from the base's (a temperature change at
    one of the last two depths), else None."""
    T = np.asarray(temperature, dtype=np.float64)
    if param != 'temperature' or k < T.shape[0] - 2:
        return None
    from .tables import planck_bc
    Tp = T.copy()
    Tp[k] = perturbed_value(T, step, k, s)
    return planck_bc(wavelength, Tp)


def perturbed_problem(base, param, step, k, s, aDamp_minus=None, aDamp_plus=None):
    """The upload_thermo problem dict of the column (k, s): a shallow copy of `base` with X[k] -> X[k] + s * step and,
    for 'temperature' / 'vturb', aDamp row k taken from aDamp_plus (s = +1) or aDamp_minus (s = -1)."""
    if param not in RESPONSE_PARAMS or s not in (-1, 1):
        raise ValueError('param must be one of %s and s -1 or +1' % (RESPONSE_PARAMS,))
    q = dict(base)
    x = np.array(base[param], dtype=np.float64).reshape(-1)
    x[k] = perturbed_value(x, step, k, s)
    q[param] = x
    if param != 'vlos':
        src = aDamp_plus if s > 0 else aDamp_minus
        a = np.array(base['aDamp'], dtype=np.float64)
        a[:, k] = np.asarray(src, dtype=np.float64)[:, k]
        q['aDamp'] = a
    return q


@dataclass
class ResponseFunction:
    """What MaliEngine.compute_response returns.  rf[d][la][m] = (I_plus - I_minus) / (2 step) of the columns perturbed at
    depths[d]; I_minus, I_plus [ndepth, Nspect, nmu]; I0 [Nspect, nmu] the solved base at the same angles; mu the angles
    of compute_rays, or None for the model's quadrature angles (I of the last formal solution, as response_fn.py reads
    ctx.I); iterations [ndepth, 2] and converged [ndepth, 2] per column (s = -1, +1); base_iterations, base_converged.
    The reference's normalised form is (I_plus - I_minus) / I0."""
    param: str
    step: float
    depths: np.ndarray
    mu: np.ndarray
    rf: np.ndarray
    I_minus: np.ndarray
    I_plus: np.ndarray
    I0: np.ndarray
    iterations: np.ndarray
    converged: np.ndarray
    base_iterations: int
    base_converged: bool
