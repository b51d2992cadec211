"""ctypes binding of libmali_b200.so (include/mali_b200.h).  Thin on purpose: plain pointers and sizes.

There is no CPU fallback: if the library is missing or was not built, importing the compute layer fails loudly.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, '_lib', os.environ.get('MALI_LIB_NAME', 'libmali_b200.so'))

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class MaliError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__('libmali_b200 error %d: %s' % (code, msg))
        self.code = code


class ModelDesc(C.Structure):
    _fields_ = [('Nspace', C.c_int32), ('Nrays', C.c_int32), ('Nspect', C.c_int32), ('Natom', C.c_int32),
                ('Ntrans', C.c_int32), ('Nlevel', _ip), ('trans', _ip), ('wavelength', _dp), ('muz', _dp),
                ('wmu', _dp), ('lineconst', _dp), ('wlambda', _dp), ('alpha', _dp), ('twohc_l3', _dp),
                ('wlacont', _dp), ('lambda0', _dp)]


class AtomDesc(C.Structure):
    _fields_ = [('Natom', C.c_int32), ('Nlevel', _ip), ('dE', _dp), ('gi0', _dp), ('dZ', _ip), ('nDebye', _dp), ('g', _dp),
                ('vTherm', _dp), ('c1', C.c_double), ('c2', C.c_double), ('Ncoll', C.c_int32), ('coll', _ip),
                ('knots', _dp), ('coef', _dp), ('fill', _dp), ('par', _dp)]


class EosDesc(C.Structure):
    _fields_ = [('npf', C.c_int32), ('tpf', _dp), ('pf', _dp), ('eion', _dp), ('stage_off', _ip), ('abund', _dp),
                ('avw', C.c_double), ('rho_from_H', C.c_double), ('ab_others', C.c_double), ('saha_fac', C.c_double),
                ('prec', C.c_double), ('amu_weight_per_H', C.c_double), ('cm_to_m_cubed', C.c_double),
                ('thomson_sigma', C.c_double)]


class Layout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in (
        'hostpack', 'colconst', 'pops', 'J', 'I', 'Gamma', 'scratch', 'hp_height', 'hp_bbc', 'hp_bg_chi',
        'hp_bg_eta', 'hp_bg_sca', 'hp_C', 'hp_nTotal', 'hp_gijcont', 'hp_n', 'hp_phi', 'hp_wphi')] + \
        [(n, C.c_int32) for n in ('sumNlevel', 'sumNlevel2', 'ntile', 'lambda_per_warp')]


class Buffers(C.Structure):
    _fields_ = [('ncol', C.c_int32), ('colconst', C.c_void_p), ('pops', C.c_void_p), ('J', C.c_void_p),
                ('I', C.c_void_p), ('Gamma', C.c_void_p), ('scratch', C.c_void_p), ('dJ', C.c_void_p),
                ('dPops', C.c_void_p), ('status', C.c_void_p), ('iter', C.c_void_p), ('done', C.c_void_p)]


class RaysDepthOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('I', 'chi', 'S', 'tau', 'contrib', 'z_tau1', 'height')]


class PerturbDesc(C.Structure):
    _fields_ = [('depth', _ip)] + [(n, C.c_void_p) for n in (
        'T', 'ne', 'nHTot', 'vturb', 'vlos', 'cmass', 'aDamp', 'bbc', 'pops0', 'src_work', 'src_nStar', 'src_vBroad',
        'work', 'nStar', 'vBroad')]


class NgParams(C.Structure):
    _fields_ = [('order', C.c_int32), ('delay', C.c_int32), ('period', C.c_int32)]


class NgBuffers(C.Structure):
    _fields_ = [('hist', C.c_void_p), ('nse', C.c_void_p), ('accepted', C.c_void_p)]


EXPORTS = ['mali_last_error', 'mali_device_count', 'mali_model_create', 'mali_model_destroy', 'mali_model_layout', 'mali_model_info',
           'mali_planck_bc', 'mali_upload_columns', 'mali_upload_columns_nophi', 'mali_compute_phi', 'mali_formal_sol_gamma', 'mali_stat_equil', 'mali_iterate',
           'mali_piecewise_linear_1d', 'mali_uv', 'mali_exp_hook', 'mali_div_hook', 'mali_profile_begin',
           'mali_profile_end', 'mali_launch_count', 'mali_fp64_peak', 'mali_line_layout', 'mali_model_set_arith', 'mali_model_get_arith',
           'mali_upload_columns_atmos', 'mali_model_set_atoms', 'mali_setup_columns',
           'mali_upload_columns_thermo', 'mali_model_set_eos', 'mali_background', 'mali_graph_iterations',
           'mali_ng_layout', 'mali_stat_equil_ng', 'mali_iterate_ng', 'mali_ng_hook', 'mali_compute_rays',
           'mali_compute_rays_depth', 'mali_compute_rates', 'mali_perturb_columns']

RAYS_MAX_MU = 64   # MALI_RAYS_MAX_MU

ARITH_EXACT, ARITH_CONTRACTED = 0, 1

_libs = {}


def load(path=None):
    """Load the shared library (building it is the job of lightspinner_b200.build / __graft_entry__.build).
    `path`: a model-specific variant built by lightspinner_b200.specialize (same ABI, other kernel instances)."""
    path = LIB_PATH if path is None else path
    if path in _libs:
        return _libs[path]
    if not os.path.isfile(path):
        raise ImportError('%s is missing: run `python -m lightspinner_b200.build` (nvcc, sm_100a). '
                          'There is no CPU fallback for the MALI hot path.' % path)
    L = C.CDLL(path)
    L.mali_last_error.restype = C.c_char_p
    L.mali_device_count.restype = C.c_int
    L.mali_model_create.argtypes = [C.POINTER(ModelDesc), C.c_int, C.POINTER(C.c_void_p)]
    L.mali_model_destroy.argtypes = [C.c_void_p]
    L.mali_model_destroy.restype = None
    L.mali_model_layout.argtypes = [C.c_void_p, C.POINTER(Layout)]
    L.mali_model_info.argtypes = [C.c_void_p, C.POINTER(C.c_int32)]
    L.mali_planck_bc.argtypes = [_dp, C.c_int32, C.c_double, C.c_double, _dp]
    L.mali_upload_columns.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                      C.c_void_p]
    L.mali_upload_columns_nophi.argtypes = L.mali_upload_columns.argtypes
    L.mali_upload_columns_atmos.argtypes = L.mali_upload_columns.argtypes
    L.mali_model_set_atoms.argtypes = [C.c_void_p, C.POINTER(AtomDesc)]
    L.mali_upload_columns_thermo.argtypes = L.mali_upload_columns.argtypes
    L.mali_model_set_eos.argtypes = [C.c_void_p, C.POINTER(EosDesc)]
    L.mali_background.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_int32, C.c_int32] + [C.c_void_p] * 6
    L.mali_setup_columns.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_int32, C.c_int32] + [C.c_void_p] * 5 + \
        [C.c_int32, C.c_void_p]
    L.mali_compute_phi.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p]
    for name in ('mali_formal_sol_gamma', 'mali_stat_equil'):
        getattr(L, name).argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_int32, C.c_int32, C.c_void_p]
    L.mali_iterate.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_int32, C.c_int32, C.c_int32, C.c_double,
                               C.c_double, C.c_void_p]
    L.mali_piecewise_linear_1d.argtypes = [C.c_int32, C.c_int32] + [C.c_void_p] * 10
    L.mali_profile_begin.argtypes = [C.c_void_p, C.c_int32]
    L.mali_profile_end.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int32)]
    L.mali_launch_count.argtypes = [C.c_void_p]
    L.mali_model_set_arith.argtypes = [C.c_void_p, C.c_int32]
    L.mali_model_get_arith.argtypes = [C.c_void_p]
    L.mali_line_layout.argtypes = [C.c_void_p, C.c_int32, _ip, _ip, _ip, C.c_int32, C.POINTER(C.c_int64)]
    L.mali_launch_count.restype = C.c_longlong
    L.mali_graph_iterations.argtypes = [C.c_void_p]
    L.mali_graph_iterations.restype = C.c_longlong
    L.mali_div_hook.argtypes = [C.c_int32] + [C.c_void_p] * 5
    L.mali_fp64_peak.argtypes = [C.c_int32, C.c_void_p, C.POINTER(C.c_double)]
    L.mali_exp_hook.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mali_ng_layout.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int64)]
    L.mali_stat_equil_ng.argtypes = [C.c_void_p, C.POINTER(Buffers), C.POINTER(NgBuffers), C.POINTER(NgParams), C.c_int32,
                                     C.c_int32, C.c_void_p]
    L.mali_iterate_ng.argtypes = [C.c_void_p, C.POINTER(Buffers), C.POINTER(NgBuffers), C.POINTER(NgParams), C.c_int32,
                                  C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_void_p]
    L.mali_ng_hook.argtypes = [C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mali_compute_rays.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_int32, C.c_int32, C.c_int32, _dp] + \
        [C.c_void_p] * 6
    L.mali_compute_rays_depth.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_int32, C.c_int32, C.c_int32, _dp] + \
        [C.c_void_p] * 3 + [C.POINTER(RaysDepthOut), C.c_void_p, C.c_void_p]
    L.mali_compute_rates.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_int32, C.c_int32] + [C.c_void_p] * 4
    L.mali_perturb_columns.argtypes = [C.c_void_p, C.POINTER(Buffers), C.c_int32, C.c_int32, C.c_int32,
                                       C.POINTER(PerturbDesc), C.c_void_p]
    L.mali_uv.argtypes = [C.c_void_p, C.POINTER(Buffers)] + [C.c_int32] * 5 + [C.c_void_p] * 4
    _libs[path] = L
    return L


def check(code, lib=None):
    """Raise MaliError for a non-zero return code.  `lib`: the library that produced it (the message lives in a
    thread-local of that very .so; model-specific variants are separate libraries)."""
    if code != 0:
        L = load() if lib is None else lib
        raise MaliError(code, L.mali_last_error().decode('utf-8', 'replace'))
