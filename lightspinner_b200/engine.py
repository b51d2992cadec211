"""Batched MALI engine: owns the device buffers (torch tensors as carriers) of a batch of columns that share one
radiative model, and drives libmali_b200.so through its C ABI.

    eng = MaliEngine(problem_or_ModelTables, ncol)       # Context.__init__ for ncol columns
    eng.upload([problem0, problem1, ...])                 # host pack -> H2D -> device re-layout
    dJ = eng.formal_sol_gamma_matrices()                  # [ncol] numpy   (rh_method.py:565-708)
    dP = eng.stat_equil()                                 # [ncol] numpy   (rh_method.py:710-745)
    eng.J(col), eng.I(col), eng.Gamma(col), eng.n(col)    # numpy, reference shapes
    I = eng.compute_rays([1.0, 0.5])                      # [ncol, Nspect, nmu] emergent intensity at user angles
    d = eng.compute_rays_depth([1.0, 0.5])                # RayDepthData: I, chi, S, tau, contrib per depth, z_tau1
    r = eng.compute_rates()                               # RadiativeRates: Rij, Rji, net [ncol, Ntrans, Nspace]
    rf = eng.compute_response(base, 'temperature', 25.0, aDamp_minus=.., aDamp_plus=..)   # ResponseFunction

Columns are independent (no cross-column arithmetic anywhere), which is what makes the path data-parallel:
ranks of a multi-GPU job each own a contiguous slice of columns (see lightspinner_b200/sharding.py).
"""
import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _capi
from .tables import ModelTables, pack_column


class MaliEngine:
    def __init__(self, model, ncol, device=None, max_upload_chunk=64, specialize=False, arith=None, library=None, ng=None):
        """arith: 'exact' | 'contracted' | None (the library's default / the MALI_ARITH environment variable) -- the
        arithmetic mode of the formal-solution kernels, see include/mali_b200.h (mali_model_set_arith).
        library: path of another build of the library with the same ABI (e.g. the checked build of tools/build_variants.py).
        specialize=True: if the model has wavelength tiles without a specialised kernel instance and nvcc is
        available, build (once, cached) a model-specific variant of the library; otherwise those tiles run on the
        generic kernel.  specialize=<problem dict>: build / pick the variant that covers THAT model (e.g. the full
        column when `model` is one wavelength shard of it, so that every rank loads the same library).
        ng: an NgOptions to enable Ng acceleration of the population iteration (stat_equil, iterate_async); None: off,
        and every launch and result is that of the plain iteration."""
        if not torch.cuda.is_available():
            raise RuntimeError('lightspinner_b200 needs a CUDA device: the MALI hot path has no CPU fallback')
        self.mt = model if isinstance(model, ModelTables) else ModelTables(model)
        self.ncol = int(ncol)
        self.device = torch.device('cuda', torch.cuda.current_device() if device is None else device)
        lib_path = library
        if isinstance(specialize, dict) or (specialize and not isinstance(model, ModelTables)):
            from . import specialize as _spec
            lib_path = _spec.library_for(specialize if isinstance(specialize, dict) else model)
        self.lib = _capi.load(lib_path)
        self._handle = C.c_void_p()
        desc = self.mt.desc()
        self._check(self.lib.mali_model_create(C.byref(desc), self.device.index, C.byref(self._handle)))
        if arith is not None:
            self.set_arith(arith)
        info = self.model_info()
        if info['generic_tiles'] > 0 and lib_path is None:
            import warnings
            warnings.warn('%d of %d wavelength tiles of this model have no structure-specialised kernel instance and run '
                          'on the generic kernel (~4x slower): pass specialize=True to build a model-specific library, '
                          'or add the model to tools/gen_spec_instances.py' % (info['generic_tiles'], info['ntile']),
                          RuntimeWarning, stacklevel=2)
        self.lay = _capi.Layout()
        self._check(self.lib.mali_model_layout(self._handle, C.byref(self.lay)))
        L = self.lay
        f64 = dict(dtype=torch.float64, device=self.device)
        i32 = dict(dtype=torch.int32, device=self.device)
        n = self.ncol
        self.t_colconst = torch.zeros(n * L.colconst, **f64)
        self.t_pops = torch.zeros(n * L.pops, **f64)
        self.t_J = torch.zeros(n * L.J, **f64)
        self.t_I = torch.zeros(n * L.I, **f64)
        self.t_Gamma = torch.zeros(n * L.Gamma, **f64)
        self.t_scratch = torch.zeros(n * L.scratch, **f64)
        self.t_dJ = torch.zeros(n, **f64)
        self.t_dPops = torch.ones(n, **f64)
        self.t_status = torch.zeros(n, **i32)
        self.t_iter = torch.zeros(n, **i32)
        self.t_done = torch.zeros(n, **i32)
        self.bufs = _capi.Buffers(n, *(t.data_ptr() for t in (
            self.t_colconst, self.t_pops, self.t_J, self.t_I, self.t_Gamma, self.t_scratch, self.t_dJ,
            self.t_dPops, self.t_status, self.t_iter, self.t_done)))
        # each column's line-profile inputs, kept for compute_rays (which forms the profiles at new angles); the
        # uploads that take host profiles instead leave a column without them (_has_profile False)
        N = self.mt.Nspace
        self.t_aDamp = torch.zeros(n, self.mt.Ntrans, N, **f64)
        self.t_vBroad = torch.zeros(n, self.mt.Natom, N, **f64)
        self.t_vlos = torch.zeros(n, N, **f64)
        self._has_profile = np.zeros(n, dtype=bool)
        self._rays_bad = None
        self.chunk = max(1, min(int(max_upload_chunk), n))
        self._staging = None
        self._pinned = None
        self.ng = ng
        if ng is not None:
            from .ng import NgOptions
            if not isinstance(ng, NgOptions):
                raise TypeError('ng must be an NgOptions (or None)')
            per = C.c_int64(0)
            self._check(self.lib.mali_ng_layout(self._handle, ng.order, C.byref(per)))
            self.t_ng_hist = torch.zeros(n * per.value, **f64)
            self.t_ng_nse = torch.zeros(n, **i32)
            self.t_ng_accepted = torch.zeros(n * self.mt.Natom, **i32)
            self.ng_bufs = _capi.NgBuffers(*(t.data_ptr() for t in (self.t_ng_hist, self.t_ng_nse, self.t_ng_accepted)))
            self.ng_params = _capi.NgParams(ng.order, ng.delay, ng.period)

    def _check(self, code):
        _capi.check(code, self.lib)

    def set_arith(self, mode):
        modes = {'exact': _capi.ARITH_EXACT, 'contracted': _capi.ARITH_CONTRACTED}
        if mode not in modes:
            raise ValueError("arith must be 'exact' or 'contracted'")
        self._check(self.lib.mali_model_set_arith(self._handle, modes[mode]))

    @property
    def arith(self):
        return 'contracted' if self.lib.mali_model_get_arith(self._handle) == _capi.ARITH_CONTRACTED else 'exact'

    def close(self):
        if self._handle:
            self.lib.mali_model_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _staging_bufs(self, per_column=None):
        """Device staging of `chunk` host-pack blocks and a pinned host buffer of `chunk * per_column` doubles
        (default: whole blocks).  The upload paths that send only a prefix of each block pin only that much:
        page-locking gigabytes takes a good fraction of a second."""
        if self._staging is None:
            self._staging = torch.empty(self.chunk * self.lay.hostpack, dtype=torch.float64, device=self.device)
        need = self.chunk * int(self.lay.hostpack if per_column is None else per_column)
        if self._pinned is None or self._pinned.numel() < need:
            self._pinned = torch.empty(need, dtype=torch.float64, pin_memory=True)
        return self._staging, self._pinned

    def hostpack_size(self):
        return int(self.lay.hostpack)

    # ------------------------------------------------------------------ upload
    def upload(self, problems, col0=0):
        """Pack and upload a list of problem dicts into columns [col0, col0+len(problems))."""
        staging, pinned = self._staging_bufs()
        hp = self.lay.hostpack
        pin_np = pinned.numpy()
        for c0 in range(0, len(problems), self.chunk):
            chunk = problems[c0:c0 + self.chunk]
            torch.cuda.current_stream(self.device).synchronize()  # pinned buffer reuse
            for q, p in enumerate(chunk):
                pack_column(self.mt, self.lay, p, out=pin_np[q * hp:(q + 1) * hp])
            self.upload_packed(pinned, col0 + c0, len(chunk))
            for q, p in enumerate(chunk):    # keep the profile inputs when the dict carries them
                if all(k in p for k in ('aDamp', 'vBroad', 'vlos')):
                    self._keep_profile_inputs(col0 + c0 + q, 1, *(np.asarray(p[k], dtype=np.float64)[None]
                                                                  for k in ('aDamp', 'vBroad', 'vlos')))
        torch.cuda.current_stream(self.device).synchronize()

    def _keep_profile_inputs(self, col0, ncol, aDamp, vBroad, vlos):
        """Copies a range of columns' aDamp / vBroad / vlos (numpy arrays or device tensors) into the persistent
        tensors compute_rays reads, and returns those slices.  Inputs that are not of the model's shape (e.g. the aDamp
        rows of lines a derived model dropped; compute_phi reads nothing of a model without lines) are not kept: the
        columns are then marked as having no profile inputs and None is returned."""
        c1 = col0 + ncol
        ins = [torch.as_tensor(a, dtype=torch.float64) for a in (aDamp, vBroad, vlos)]
        if any(a.numel() != ncol * t[0].numel() for a, t in zip(ins, (self.t_aDamp, self.t_vBroad, self.t_vlos))):
            self._has_profile[col0:c1] = False
            return None
        out = []
        for t, a in zip((self.t_aDamp, self.t_vBroad, self.t_vlos), ins):
            dst = t[col0:c1]
            if a.data_ptr() != dst.data_ptr() or a.device != dst.device:
                dst.copy_(a.reshape(dst.shape), non_blocking=a.device == dst.device)
            out.append(dst)
        self._has_profile[col0:c1] = True
        return out

    def upload_device_phi(self, problems, col0=0):
        """Like upload(), but the Voigt line profiles are formed on the device (ComputationalTransition.compute_phi,
        rh_method.py:198-243 -> mali_compute_phi) from each problem's damping parameters `aDamp` [Ntrans, Nspace],
        Doppler widths `vBroad` [Natom, Nspace] and `vlos` [Nspace]: only the blocks without phi / wphi (about 40 %
        of the bytes) cross PCIe.  Profiles agree with the reference's to ~1e-13 (the accuracy of scipy's wofz)."""
        self.ng_reset(col0, len(problems))
        hpp = int(self.lay.hp_phi)
        staging, pinned = self._staging_bufs(hpp)
        pin_np = pinned.numpy()
        N = self.mt.Nspace
        for c0 in range(0, len(problems), self.chunk):
            chunk = problems[c0:c0 + self.chunk]
            torch.cuda.current_stream(self.device).synchronize()  # pinned buffer reuse
            for q, p in enumerate(chunk):
                pack_column(self.mt, self.lay, p, out=pin_np[q * hpp:(q + 1) * hpp], with_phi=False)
            aux = [np.stack([np.asarray(p[k], dtype=np.float64).reshape(-1, N) for p in chunk])
                   for k in ('aDamp', 'vBroad', 'vlos')]
            if aux[0].shape[1] != self.mt.Ntrans or aux[1].shape[1] != self.mt.Natom or aux[2].shape[1] != 1:
                raise ValueError('aDamp / vBroad / vlos must be [Ntrans, Nspace] / [Natom, Nspace] / [Nspace]')
            dev = self._keep_profile_inputs(col0 + c0, len(chunk), *aux)      # (shapes checked above)
            with torch.cuda.device(self.device):
                self._check(self.lib.mali_upload_columns_nophi(self._handle, C.byref(self.bufs), col0 + c0, len(chunk),
                                                               C.c_void_p(pinned.data_ptr()),
                                                               C.c_void_p(staging.data_ptr()), self._stream()))
                self._check(self.lib.mali_compute_phi(self._handle, C.byref(self.bufs), col0 + c0, len(chunk),
                                                      *(C.c_void_p(t.data_ptr()) for t in dev), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()

    def set_atoms(self, atom_tables):
        """Registers the model-level atom data (lightspinner_b200.atoms.AtomTables) the device-side column set-up needs."""
        self._atom_tables = atom_tables
        desc = atom_tables.desc()
        self._check(self.lib.mali_model_set_atoms(self._handle, C.byref(desc)))

    def upload_atmos(self, problems, col0=0, start_from_lte=True):
        """Like upload_device_phi(), with everything the device can form from the atmosphere formed there: each
        problem supplies height, temperature, ne, vturb, vlos, nTotal, the background (bg_chi / bg_eta / bg_sca) and the
        lines' damping parameters aDamp; LTE populations, collisional rates, Doppler widths, the continua's g_ij
        (mali_setup_columns) and the Voigt profiles (mali_compute_phi) are computed on the GPU.  start_from_lte=False
        keeps the populations given in problem['n'] (a warm start, response_fn.py:33).  Needs set_atoms()."""
        self.ng_reset(col0, len(problems))
        hpc = int(self.lay.hp_C)
        staging, pinned = self._staging_bufs(hpc)
        pin_np = pinned.numpy()
        N = self.mt.Nspace
        self.nStar = getattr(self, 'nStar', None)
        if self.nStar is None:
            self.nStar = torch.zeros(self.ncol * self.lay.sumNlevel * N, dtype=torch.float64, device=self.device)
        for c0 in range(0, len(problems), self.chunk):
            chunk = problems[c0:c0 + self.chunk]
            nc = len(chunk)
            torch.cuda.current_stream(self.device).synchronize()  # pinned buffer reuse
            for q, p in enumerate(chunk):
                pack_column(self.mt, self.lay, p, out=pin_np[q * hpc:(q + 1) * hpc], with_derived=False)
            aux = {k: torch.from_numpy(np.ascontiguousarray(np.stack(
                [np.asarray(p[k], dtype=np.float64).reshape(-1, N) for p in chunk]))).to(self.device)
                for k in ('temperature', 'ne', 'vturb', 'vlos', 'aDamp')}
            # mali_setup_columns writes the Doppler widths straight into the persistent slice compute_rays reads
            vBroad = self.t_vBroad[col0 + c0:col0 + c0 + nc]
            self._keep_profile_inputs(col0 + c0, nc, aux['aDamp'], vBroad, aux['vlos'])
            ns = self.nStar[(col0 + c0) * self.lay.sumNlevel * N:(col0 + c0 + nc) * self.lay.sumNlevel * N]
            P = lambda t: C.c_void_p(t.data_ptr())
            with torch.cuda.device(self.device):
                self._check(self.lib.mali_upload_columns_atmos(self._handle, C.byref(self.bufs), col0 + c0, nc,
                                                               P(pinned), P(staging), self._stream()))
                self._check(self.lib.mali_setup_columns(self._handle, C.byref(self.bufs), col0 + c0, nc,
                                                        P(aux['temperature']), P(aux['ne']), P(aux['vturb']), P(ns),
                                                        P(vBroad), 1 if start_from_lte else 0, self._stream()))
                self._check(self.lib.mali_compute_phi(self._handle, C.byref(self.bufs), col0 + c0, nc, P(aux['aDamp']),
                                                      P(vBroad), P(aux['vlos']), self._stream()))
            if not start_from_lte:
                for q, p in enumerate(chunk):
                    self.set_n(col0 + c0 + q, p['n'])
            torch.cuda.current_stream(self.device).synchronize()
            self._last_vBroad = vBroad

    def set_eos(self, eos_tables):
        """Registers the EOS / background tables (lightspinner_b200.eos.EosTables) mali_background needs."""
        self._eos_tables = eos_tables
        desc = eos_tables.desc()
        self._check(self.lib.mali_model_set_eos(self._handle, C.byref(desc)))

    def upload_thermo(self, problems, col0=0, start_from_lte=True):
        """The whole per-column set-up on the device, from the thermodynamic state: each problem supplies temperature,
        ne, nHTot, vturb, vlos, nTotal, the lines' damping parameters aDamp and either `cmass` (a column-mass depth
        scale: the heights come from convert_scales' recurrence on the device) or `height`.  The EOS, the background
        opacities (mali_background), LTE populations, collisional rates, Doppler widths, the continua's g_ij
        (mali_setup_columns) and the Voigt profiles (mali_compute_phi) are all formed on the GPU.
        Needs set_eos() and set_atoms()."""
        self.ng_reset(col0, len(problems))
        hpb = int(self.lay.hp_bg_chi)
        staging, pinned = self._staging_bufs(hpb)
        pin_np = pinned.numpy()
        N = self.mt.Nspace
        if getattr(self, 'nStar', None) is None:
            self.nStar = torch.zeros(self.ncol * self.lay.sumNlevel * N, dtype=torch.float64, device=self.device)
        for c0 in range(0, len(problems), self.chunk):
            chunk = problems[c0:c0 + self.chunk]
            nc = len(chunk)
            torch.cuda.current_stream(self.device).synchronize()  # pinned buffer reuse
            for q, p in enumerate(chunk):
                pack_column(self.mt, self.lay, p, out=pin_np[q * hpb:(q + 1) * hpb], with_background=False)
            keys = ['temperature', 'ne', 'nHTot', 'vturb', 'vlos', 'aDamp'] + (['cmass'] if 'cmass' in chunk[0] else [])
            aux = {k: torch.from_numpy(np.ascontiguousarray(np.stack(
                [np.asarray(p[k], dtype=np.float64).reshape(-1, N) for p in chunk]))).to(self.device) for k in keys}
            vBroad = self.t_vBroad[col0 + c0:col0 + c0 + nc]
            self._keep_profile_inputs(col0 + c0, nc, aux['aDamp'], vBroad, aux['vlos'])
            work = torch.empty(nc * N * 21, dtype=torch.float64, device=self.device)
            ns = self.nStar[(col0 + c0) * self.lay.sumNlevel * N:(col0 + c0 + nc) * self.lay.sumNlevel * N]
            P = lambda t: C.c_void_p(t.data_ptr())
            with torch.cuda.device(self.device):
                self._check(self.lib.mali_upload_columns_thermo(self._handle, C.byref(self.bufs), col0 + c0, nc,
                                                                P(pinned), P(staging), self._stream()))
                self._check(self.lib.mali_background(self._handle, C.byref(self.bufs), col0 + c0, nc,
                                                     P(aux['temperature']), P(aux['ne']), P(aux['nHTot']),
                                                     P(aux['cmass']) if 'cmass' in aux else None, P(work), self._stream()))
                self._check(self.lib.mali_setup_columns(self._handle, C.byref(self.bufs), col0 + c0, nc,
                                                        P(aux['temperature']), P(aux['ne']), P(aux['vturb']), P(ns),
                                                        P(vBroad), 1 if start_from_lte else 0, self._stream()))
                self._check(self.lib.mali_compute_phi(self._handle, C.byref(self.bufs), col0 + c0, nc, P(aux['aDamp']),
                                                      P(vBroad), P(aux['vlos']), self._stream()))
            if not start_from_lte:
                for q, p in enumerate(chunk):
                    self.set_n(col0 + c0 + q, p['n'])
            torch.cuda.current_stream(self.device).synchronize()
            self._last_vBroad = vBroad
            self._last_work = work

    def upload_packed_device_phi(self, host_prefix_pinned, aDamp, vBroad, vlos, col0, ncol, staging=None):
        """Asynchronous form of upload_device_phi: `host_prefix_pinned` holds [ncol][lay.hp_phi] doubles (pinned),
        aDamp / vBroad / vlos are device tensors [ncol][Ntrans|Natom|1][Nspace]."""
        self.ng_reset(col0, ncol)
        self._keep_profile_inputs(col0, ncol, aDamp, vBroad, vlos)
        if staging is None:
            staging, _ = self._staging_bufs(0)
        if ncol * self.lay.hostpack > staging.numel():
            raise ValueError('staging buffer too small for %d columns' % ncol)
        with torch.cuda.device(self.device):
            self._check(self.lib.mali_upload_columns_nophi(self._handle, C.byref(self.bufs), col0, ncol,
                                                           C.c_void_p(host_prefix_pinned.data_ptr()),
                                                           C.c_void_p(staging.data_ptr()), self._stream()))
            self._check(self.lib.mali_compute_phi(self._handle, C.byref(self.bufs), col0, ncol,
                                                  C.c_void_p(aDamp.data_ptr()), C.c_void_p(vBroad.data_ptr()),
                                                  C.c_void_p(vlos.data_ptr()), self._stream()))

    def upload_packed(self, host_pinned, col0, ncol, staging=None):
        """H2D copy of `ncol` host-pack blocks (a pinned torch tensor) + device re-layout; asynchronous.  The blocks
        carry the line profiles, not their inputs: compute_rays refuses these columns (upload() keeps the inputs
        when the problem dicts have them)."""
        self.ng_reset(col0, ncol)
        self._has_profile[col0:col0 + ncol] = False
        if staging is None:
            staging, _ = self._staging_bufs(0)
        if ncol * self.lay.hostpack > staging.numel():
            raise ValueError('staging buffer too small for %d columns' % ncol)
        with torch.cuda.device(self.device):
            self._check(self.lib.mali_upload_columns(self._handle, C.byref(self.bufs), col0, ncol,
                                                     C.c_void_p(host_pinned.data_ptr()),
                                                     C.c_void_p(staging.data_ptr()), self._stream()))

    def repack_from_staging(self, staging, col0, ncol):
        """Device re-layout only (the staging tensor already holds host-pack blocks on the device)."""
        self.ng_reset(col0, ncol)
        self._has_profile[col0:col0 + ncol] = False
        with torch.cuda.device(self.device):
            self._check(self.lib.mali_upload_columns(self._handle, C.byref(self.bufs), col0, ncol, None,
                                                     C.c_void_p(staging.data_ptr()), self._stream()))

    # ------------------------------------------------------------------ the hot path
    def formal_sol_gamma_async(self, col0=0, ncol=None):
        ncol = self.ncol - col0 if ncol is None else ncol
        with torch.cuda.device(self.device):
            self._check(self.lib.mali_formal_sol_gamma(self._handle, C.byref(self.bufs), col0, ncol, self._stream()))

    def stat_equil_async(self, col0=0, ncol=None):
        ncol = self.ncol - col0 if ncol is None else ncol
        with torch.cuda.device(self.device):
            if self.ng is not None:
                self._check(self.lib.mali_stat_equil_ng(self._handle, C.byref(self.bufs), C.byref(self.ng_bufs),
                                                        C.byref(self.ng_params), col0, ncol, self._stream()))
            else:
                self._check(self.lib.mali_stat_equil(self._handle, C.byref(self.bufs), col0, ncol, self._stream()))

    def formal_sol_gamma_matrices(self, col0=0, ncol=None):
        """One Lambda iteration for columns [col0, col0+ncol) (default: all); returns their dJ (device->host read)."""
        ncol = self.ncol - col0 if ncol is None else ncol
        self.formal_sol_gamma_async(col0, ncol)
        dJ = self.t_dJ[col0:col0 + ncol].cpu().numpy()
        status = self.t_status[col0:col0 + ncol].cpu().numpy()
        if (status & 2).any():
            bad = col0 + np.nonzero(status & 2)[0]
            self.t_status[col0:col0 + ncol].bitwise_and_(~2)
            raise FloatingPointError('opacity or optical-depth step outside the formal solver\'s numeric domain '
                                     '(zero, subnormal, infinite or NaN) in column(s) %s' % bad[:8].tolist())
        return dJ

    def stat_equil(self, col0=0, ncol=None):
        """Statistical equilibrium for columns [col0, col0+ncol) (default: all); returns their dPops."""
        ncol = self.ncol - col0 if ncol is None else ncol
        self.stat_equil_async(col0, ncol)
        dP = self.t_dPops[col0:col0 + ncol].cpu().numpy()
        status = self.t_status[col0:col0 + ncol].cpu().numpy()
        if (status & 1).any():
            bad = col0 + np.nonzero(status & 1)[0]
            self.t_status[col0:col0 + ncol].zero_()
            raise np.linalg.LinAlgError('singular statistical-equilibrium system in column(s) %s' % bad[:8].tolist())
        return dP

    def iterate_async(self, max_iter, tolJ=2e-3, tolPops=1e-3, col0=0, ncol=None):
        """The loop of test.py:20-29 on the device with per-column convergence (tolJ < 0: fixed iteration count)."""
        ncol = self.ncol - col0 if ncol is None else ncol
        with torch.cuda.device(self.device):
            if self.ng is not None:
                self._check(self.lib.mali_iterate_ng(self._handle, C.byref(self.bufs), C.byref(self.ng_bufs),
                                                     C.byref(self.ng_params), col0, ncol, int(max_iter), float(tolJ),
                                                     float(tolPops), self._stream()))
            else:
                self._check(self.lib.mali_iterate(self._handle, C.byref(self.bufs), col0, ncol, int(max_iter),
                                                  float(tolJ), float(tolPops), self._stream()))

    def raise_on_faults(self, col0=0, ncol=None):
        """What the reference would have raised during the loop: LinAlgError for a singular statistical-equilibrium
        system (status bit 0), FloatingPointError for an opacity / optical-depth step outside the formal solver's
        domain (status bit 1) or a NaN in dJ / dPops (done == 2).  mali_iterate stops such a column where it fails."""
        ncol = self.ncol - col0 if ncol is None else ncol
        status = self.t_status[col0:col0 + ncol].cpu().numpy()
        done = self.t_done[col0:col0 + ncol].cpu().numpy()
        if (status & 1).any():
            bad = col0 + np.nonzero(status & 1)[0]
            raise np.linalg.LinAlgError('singular statistical-equilibrium system in column(s) %s' % bad[:8].tolist())
        if (status & 2).any() or (done == 2).any():
            bad = col0 + np.nonzero((status & 2) | (done == 2))[0]
            raise FloatingPointError('non-finite result or opacity / optical-depth step outside the formal solver\'s '
                                     'numeric domain in column(s) %s' % bad[:8].tolist())

    # ------------------------------------------------------------------ emergent intensity at user angles
    def _rays_setup(self, mus, col0, ncol):
        """The checks compute_rays_async and compute_rays_depth_async share (the angles, the column range, every column
        with its profile inputs); returns the angles, ncol and the profile-input pointers, and zeroes the fault words."""
        mus = rays_angles(mus)
        ncol = self.ncol - col0 if ncol is None else ncol
        if col0 < 0 or ncol < 1 or col0 + ncol > self.ncol:
            raise ValueError('columns [%d, %d) outside the batch of %d' % (col0, col0 + ncol, self.ncol))
        if (self.mt.trans[:, 3] != 0).any() and not self._has_profile[col0:col0 + ncol].all():
            bad = col0 + np.nonzero(~self._has_profile[col0:col0 + ncol])[0]
            raise ValueError('column(s) %s were uploaded with host line profiles and without their inputs (aDamp, vBroad, '
                             'vlos): compute_rays needs those to form the profiles at new angles' % bad[:8].tolist())
        self._rays_bad = torch.zeros(ncol, dtype=torch.int32, device=self.device)
        P = lambda t: C.c_void_p(t.data_ptr()) if t.numel() else None
        return mus, ncol, [P(self.t_aDamp[col0:]), P(self.t_vBroad[col0:]), P(self.t_vlos[col0:])]

    def _raise_rays_faults(self, col0):
        bad = self._rays_bad.cpu().numpy()
        if (bad & 2).any():
            cols = col0 + np.nonzero(bad & 2)[0]
            raise FloatingPointError('opacity or optical-depth step outside the formal solver\'s numeric domain '
                                     '(zero, subnormal, infinite or NaN) in column(s) %s' % cols[:8].tolist())

    def compute_rays_async(self, mus, col0=0, ncol=None, out=None):
        """Emergent intensity at the angles `mus` (0 < mu <= 1; a scalar is one angle) from the current populations and
        J of columns [col0, col0+ncol) (mali_compute_rays): a device tensor [ncol, Nspect, nmu], `out` if given.  It is
        what the next formal solution would return as I if those angles were its quadrature angles; nothing else is
        written, so it can be called between any two iterations.  Lists longer than MALI_RAYS_MAX_MU are split into
        several launches.  Domain faults are collected for compute_rays (see there)."""
        mus, ncol, args = self._rays_setup(mus, col0, ncol)
        nmu, S = mus.shape[0], self.mt.Nspect
        if out is None:
            out = torch.empty(ncol, S, nmu, dtype=torch.float64, device=self.device)
        elif (tuple(out.shape) != (ncol, S, nmu) or out.dtype != torch.float64 or out.device != self.device
              or not out.is_contiguous()):
            raise ValueError('out must be a contiguous float64 tensor [%d, %d, %d] on %s' % (ncol, S, nmu, self.device))
        P = lambda t: C.c_void_p(t.data_ptr())
        step = _capi.RAYS_MAX_MU
        with torch.cuda.device(self.device):
            for q0 in range(0, nmu, step):
                part = mus[q0:q0 + step]
                dst = out if nmu <= step else torch.empty(ncol, S, part.shape[0], dtype=torch.float64, device=self.device)
                self._check(self.lib.mali_compute_rays(self._handle, C.byref(self.bufs), col0, ncol, part.shape[0],
                                                       part.ctypes.data_as(C.POINTER(C.c_double)), *args, P(dst),
                                                       P(self._rays_bad), self._stream()))
                if dst is not out:
                    out[:, :, q0:q0 + part.shape[0]].copy_(dst)
        return out

    def compute_rays(self, mus, col0=0, ncol=None):
        """compute_rays_async as numpy [ncol, Nspect, nmu]; raises FloatingPointError if an opacity / optical-depth step
        of a column left the formal solver's numeric domain (status bit 1 of the formal solution)."""
        col0 = int(col0)
        out = self.compute_rays_async(mus, col0, ncol)
        res = out.cpu().numpy()
        self._raise_rays_faults(col0)
        return res

    def compute_rays_depth_async(self, mus, col0=0, ncol=None, quantities=None, out=None):
        """Depth-resolved data of the rays compute_rays sweeps (mali_compute_rays_depth; definitions in
        include/mali_b200.h): a dict of device tensors, one per name in `quantities` (default RAYS_DEPTH_QUANTITIES):
        'I', 'chi', 'S', 'tau', 'contrib' [ncol, Nspace, Nspect, nmu] (depth 0 at the top), 'z_tau1' [ncol, Nspect, nmu]
        (the height of tau = 1 along each ray, NaN if it is never reached) and 'height' [ncol, Nspace].  `out` may map
        some of those names to contiguous float64 device tensors of those shapes to be filled.  The same checks as
        compute_rays_async; nothing else is written.  Lists longer than MALI_RAYS_MAX_MU are split into several
        launches.  Domain faults are collected for compute_rays_depth."""
        want = rays_depth_quantities(quantities)
        mus, ncol, args = self._rays_setup(mus, col0, ncol)
        nmu, N, S = mus.shape[0], self.mt.Nspace, self.mt.Nspect

        def shape(k, n):
            return (ncol, S, n) if k == 'z_tau1' else (ncol, N) if k == 'height' else (ncol, N, S, n)

        def empty(k, n):
            return torch.empty(shape(k, n), dtype=torch.float64, device=self.device)

        res = {}
        for k, t in (out or {}).items():
            if k not in want:
                raise ValueError('out[%r] was given but %r is not among the requested quantities %s' % (k, k, want))
            if (tuple(t.shape) != shape(k, nmu) or t.dtype != torch.float64 or t.device != self.device
                    or not t.is_contiguous()):
                raise ValueError('out[%r] must be a contiguous float64 tensor %s on %s' % (k, list(shape(k, nmu)),
                                                                                          self.device))
            res[k] = t
        for k in want:
            if k not in res:
                res[k] = empty(k, nmu)
        # contrib and z_tau1 are formed from the optical-depth steps the kernel keeps in the tau buffer
        launch = list(want) + (['tau'] if 'tau' not in want and ('contrib' in want or 'z_tau1' in want) else [])
        P = lambda t: C.c_void_p(t.data_ptr())
        step = _capi.RAYS_MAX_MU
        with torch.cuda.device(self.device):
            for q0 in range(0, nmu, step):
                part = mus[q0:q0 + step]
                n = part.shape[0]
                dst = {}
                for k in launch:
                    if k == 'height':
                        if q0 == 0:
                            dst[k] = res[k]
                    else:
                        dst[k] = res[k] if k in res and n == nmu else empty(k, n)
                if not dst:     # only the heights were asked for, and the first launch wrote them
                    break
                desc = _capi.RaysDepthOut(**{k: P(t) for k, t in dst.items()})
                self._check(self.lib.mali_compute_rays_depth(self._handle, C.byref(self.bufs), col0, ncol, n,
                                                             part.ctypes.data_as(C.POINTER(C.c_double)), *args,
                                                             C.byref(desc), P(self._rays_bad), self._stream()))
                for k, t in dst.items():
                    if k in res and t is not res[k]:
                        res[k][..., q0:q0 + n].copy_(t)
        return {k: res[k] for k in want}

    def compute_rays_depth(self, mus, col0=0, ncol=None, quantities=None):
        """compute_rays_depth_async as a RayDepthData of numpy arrays (the angles, the heights, and the requested
        quantities; the others are None).  Raises FloatingPointError on a domain fault, as compute_rays does."""
        col0 = int(col0)
        want = rays_depth_quantities(quantities)
        dev = self.compute_rays_depth_async(mus, col0, ncol, tuple(want) + (() if 'height' in want else ('height',)))
        host = {k: t.cpu().numpy() for k, t in dev.items()}
        self._raise_rays_faults(col0)
        return RayDepthData(mu=rays_angles(mus), height=host['height'],
                            **{k: host.get(k) for k in RAYS_DEPTH_QUANTITIES if k != 'height'})

    # ------------------------------------------------------------------ radiative rates
    def compute_rates_async(self, col0=0, ncol=None, out=None):
        """Radiative rates R_ij, R_ji (s^-1) of every transition from the current populations and J of columns
        [col0, col0+ncol) (mali_compute_rates; definition in include/mali_b200.h): a pair of device tensors
        [ncol, Ntrans, Nspace], `out` (a pair of contiguous float64 tensors of that shape) if given.  The intensity is
        the one the next formal solution computes, with the line profiles already in the tables, so columns uploaded
        with host profiles are served too.  The call overwrites the formal-solution scratch (which holds nothing
        between calls) and nothing else the iteration uses.  Domain faults are collected for compute_rates."""
        ncol = self.ncol - col0 if ncol is None else ncol
        if col0 < 0 or ncol < 1 or col0 + ncol > self.ncol:
            raise ValueError('columns [%d, %d) outside the batch of %d' % (col0, col0 + ncol, self.ncol))
        shape = (ncol, self.mt.Ntrans, self.mt.Nspace)
        if out is None:
            out = tuple(torch.empty(shape, dtype=torch.float64, device=self.device) for _ in range(2))
        elif (not isinstance(out, (tuple, list)) or len(out) != 2
              or any(not isinstance(t, torch.Tensor) or tuple(t.shape) != shape or t.dtype != torch.float64
                     or t.device != self.device or not t.is_contiguous() for t in out)):
            raise ValueError('out must be a pair (Rij, Rji) of contiguous float64 tensors %s on %s'
                             % (list(shape), self.device))
        self._rays_bad = torch.zeros(ncol, dtype=torch.int32, device=self.device)
        P = lambda t: C.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            self._check(self.lib.mali_compute_rates(self._handle, C.byref(self.bufs), col0, ncol, P(out[0]), P(out[1]),
                                                    P(self._rays_bad), self._stream()))
        return out[0], out[1]

    def compute_rates(self, col0=0, ncol=None):
        """compute_rates_async as a RadiativeRates of numpy arrays [ncol, Ntrans, Nspace], with the net radiative rates
        n_i R_ij - n_j R_ji (m^-3 s^-1) from the same populations.  Raises FloatingPointError on a domain fault, as
        compute_rays does."""
        col0 = int(col0)
        Rij, Rji = self.compute_rates_async(col0, ncol)
        ncol = Rij.shape[0]
        L = self.lay.pops
        n = self.t_pops[col0 * L:(col0 + ncol) * L].view(ncol, -1, self.mt.Nspace)
        tr = self.mt.trans
        rowI = torch.as_tensor(self.mt.lvloff[tr[:, 0]] + tr[:, 1], dtype=torch.int64, device=self.device)
        rowJ = torch.as_tensor(self.mt.lvloff[tr[:, 0]] + tr[:, 2], dtype=torch.int64, device=self.device)
        net = n[:, rowI] * Rij - n[:, rowJ] * Rji
        res = RadiativeRates(Rij=Rij.cpu().numpy(), Rji=Rji.cpu().numpy(), net=net.cpu().numpy())
        self._raise_rays_faults(col0)
        return res

    # ------------------------------------------------------------------ response functions
    def compute_response(self, base, param, step, *, aDamp_minus=None, aDamp_plus=None, depths=None, mus=None,
                         max_iter=500, tolJ=2e-3, tolPops=1e-3, col0=0, ncol=None):
        """Response function of the emergent intensity to `param` ('temperature' K, 'vturb' or 'vlos' m/s) at every
        depth in `depths` (default all), by central differences with step `step` (response_fn.py; definition in
        include/mali_b200.h at mali_perturb_columns and DESIGN.md): a ResponseFunction.

        base: an upload_thermo problem dict (temperature, ne, nHTot, vturb, vlos, nTotal, aDamp and cmass or height),
        solved from LTE, or from base['n'] if given.  aDamp_minus / aDamp_plus [Ntrans, Nspace]: the damping of the
        base atmosphere with `param` shifted by -step / +step at every depth (required for 'temperature' and 'vturb',
        not used for 'vlos').  Every perturbed column starts from the solved base's populations with J = 0 and runs
        the loop of iterate_async (per-column convergence at tolJ / tolPops, at most max_iter iterations, the engine's
        Ng option).  mus: the angles of compute_rays for I, or None for I at the quadrature angles after each loop.

        Columns [col0, col0+ncol) (default: all from col0) are the workspace and everything in them is overwritten:
        col0 holds the base as set up, col0 + 1 the base solve, the rest take the perturbed columns in chunks, each
        formed from col0 by mali_perturb_columns.  At least 3 columns.  Needs set_eos() and set_atoms().  Raises
        LinAlgError / FloatingPointError as raise_on_faults does."""
        from .response import ResponseFunction, base_arrays, response_args
        if getattr(self, '_eos_tables', None) is None or getattr(self, '_atom_tables', None) is None:
            raise ValueError('compute_response needs set_eos() and set_atoms()')
        mt = self.mt
        N, S = mt.Nspace, mt.Nspect
        col0 = int(col0)
        ncol = self.ncol - col0 if ncol is None else int(ncol)
        if col0 < 0 or ncol < 1 or col0 + ncol > self.ncol:
            raise ValueError('columns [%d, %d) outside the batch of %d' % (col0, col0 + ncol, self.ncol))
        if ncol < 3:
            raise ValueError('the workspace needs at least 3 columns (the base as set up, the base solve and one '
                             'perturbed column), got %d' % ncol)
        step, depths, adm, adp = response_args(param, step, aDamp_minus, aDamp_plus, depths, N, mt.Ntrans)
        b = base_arrays(base, N, mt.Natom, mt.Ntrans)
        if mus is not None:
            mus = rays_angles(mus)
        if int(max_iter) < 1:
            raise ValueError('max_iter must be >= 1, got %r' % (max_iter,))
        src, bcol, w0, W = col0, col0 + 1, col0 + 2, ncol - 2

        # the source column: set up once, never iterated; the base solve beside it
        self.upload_thermo([b], src)
        src_work = self._last_work
        if 'n' in base:
            b['n'] = base['n']
        self.upload_thermo([b], bcol, start_from_lte='n' not in base)
        self._solve_range(bcol, 1, max_iter, tolJ, tolPops)
        I0 = self._response_intensity(mus, bcol, 1)[0]
        base_iter, base_conv = int(self.t_iter[bcol].item()), bool(self.t_done[bcol].item() == 1)

        pops0 = self.t_pops[bcol * self.lay.pops:(bcol + 1) * self.lay.pops]
        cols = [(int(d), s) for d in depths for s in (-1, 1)]
        nd = depths.shape[0]
        nmu = mt.Nrays if mus is None else mus.shape[0]
        I = np.empty((nd, 2, S, nmu))
        its = np.empty((nd, 2), dtype=np.int64)
        conv = np.empty((nd, 2), dtype=bool)
        for i0 in range(0, len(cols), W):
            chunk = cols[i0:i0 + W]
            nc = len(chunk)
            self._perturb_chunk(b, param, step, chunk, adm, adp, src, src_work, pops0, w0)
            self._solve_range(w0, nc, max_iter, tolJ, tolPops)
            Ic = self._response_intensity(mus, w0, nc)
            it = self.t_iter[w0:w0 + nc].cpu().numpy()
            dn = self.t_done[w0:w0 + nc].cpu().numpy()
            for q, (k, s) in enumerate(chunk):
                d, j = (i0 + q) // 2, (s + 1) // 2
                I[d, j], its[d, j], conv[d, j] = Ic[q], it[q], dn[q] == 1
        return ResponseFunction(param=param, step=step, depths=depths, mu=mus, rf=(I[:, 1] - I[:, 0]) / (2.0 * step),
                                I_minus=I[:, 0], I_plus=I[:, 1], I0=I0, iterations=its, converged=conv,
                                base_iterations=base_iter, base_converged=base_conv)

    def _perturb_chunk(self, b, param, step, chunk, adm, adp, src, src_work, pops0, w0):
        """Columns [w0, w0+len(chunk)) become the columns (k, s) of `chunk` (mali_perturb_columns from the source column
        `src`, set up from the base arrays `b` by upload_thermo, whose EOS work rows are `src_work`), starting from the
        populations pops0; their profile inputs are kept for compute_rays."""
        from .response import perturbed_bbc, perturbed_value
        from .tables import planck_bc
        mt, N, SL = self.mt, self.mt.Nspace, int(self.lay.sumNlevel)
        nc = len(chunk)
        dev = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64).to(self.device)
        P = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        keys = ('temperature', 'ne', 'nHTot', 'vturb', 'vlos') + (('cmass',) if 'cmass' in b else ())
        # the base repeated, plus one indexed write per column
        ins = {k: dev(b[k]).reshape(1, N).repeat(nc, 1) for k in keys}
        ks = np.array([k for k, _ in chunk], dtype=np.int32)
        ar = torch.arange(nc, device=self.device)
        kt = torch.as_tensor(ks, dtype=torch.int64, device=self.device)
        x = b[param]
        ins[param][ar, kt] = dev([perturbed_value(x, step, k, s) for k, s in chunk])
        aD = dev(b['aDamp']).reshape(1, mt.Ntrans, N).repeat(nc, 1, 1)
        if param != 'vlos':
            aD[ar, :, kt] = dev(np.stack([(adp if s > 0 else adm)[:, k] for k, s in chunk]))
        bbc = None
        if param == 'temperature':
            bbc0 = planck_bc(mt.wavelength, x)
            bbc = dev(np.stack([bb if bb is not None else bbc0 for bb in
                                (perturbed_bbc(mt.wavelength, x, param, step, k, s) for k, s in chunk)]))
        aD, vBroad, vlos = self._keep_profile_inputs(w0, nc, aD, self.t_vBroad[w0:w0 + nc], ins['vlos'])
        work = torch.empty(nc * N * 21, dtype=torch.float64, device=self.device)
        desc = _capi.PerturbDesc(ks.ctypes.data_as(C.POINTER(C.c_int32)),
                                 *(P(ins[k]) for k in ('temperature', 'ne', 'nHTot', 'vturb')), P(vlos),
                                 P(ins.get('cmass')), P(aD), P(bbc), P(pops0), P(src_work),
                                 P(self.nStar[src * SL * N:(src + 1) * SL * N]), P(self.t_vBroad[src]), P(work),
                                 P(self.nStar[w0 * SL * N:(w0 + nc) * SL * N]), P(vBroad))
        with torch.cuda.device(self.device):
            self._check(self.lib.mali_perturb_columns(self._handle, C.byref(self.bufs), src, w0, nc, C.byref(desc),
                                                      self._stream()))
        torch.cuda.current_stream(self.device).synchronize()    # (the inputs above are freed on return)

    def _solve_range(self, col0, ncol, max_iter, tolJ, tolPops):
        """Fresh iteration state for columns [col0, col0+ncol), then the device loop in rounds of 16 iterations until
        every column is done or max_iter iterations ran; raises as raise_on_faults."""
        self.reset_iteration_state(col0, ncol)
        left = int(max_iter)
        while left > 0:
            n = min(16, left)
            self.iterate_async(n, tolJ, tolPops, col0, ncol)
            left -= n
            if bool((self.t_done[col0:col0 + ncol] != 0).all().item()):
                break
        self.raise_on_faults(col0, ncol)

    def _response_intensity(self, mus, col0, ncol):
        """[ncol, Nspect, nmu]: I of the last formal solution (mus None) or compute_rays at mus."""
        if mus is None:
            L = self.lay.I
            return self.t_I[col0 * L:(col0 + ncol) * L].view(ncol, self.mt.Nspect, self.mt.Nrays).cpu().numpy()
        return self.compute_rays(mus, col0, ncol)

    def reset_iteration_state(self, col0=0, ncol=None):
        """Fresh loop state (iterations, done, dPops, dJ, status and the Ng history) for columns [col0, col0+ncol),
        default all."""
        ncol = self.ncol - col0 if ncol is None else ncol
        c = slice(col0, col0 + ncol)
        self.t_iter[c].zero_()
        self.t_done[c].zero_()
        self.t_dPops[c].fill_(1.0)
        self.t_dJ[c].fill_(1.0)
        self.t_status[c].zero_()
        if self.ng is not None:
            self.t_ng_nse[c].zero_()
            self.t_ng_accepted[col0 * self.mt.Natom:(col0 + ncol) * self.mt.Natom].zero_()

    def ng_reset(self, col0=0, ncol=None):
        """Restart the Ng history of columns [col0, col0+ncol): needed after their populations were edited between
        per-call iterations (the extrapolation would otherwise mix the edited vector with the older ones)."""
        if self.ng is not None:
            ncol = self.ncol - col0 if ncol is None else ncol
            self.t_ng_nse[col0:col0 + ncol].zero_()

    def ng_accepted(self):
        """[ncol, Natom] numpy: Ng extrapolations applied since the last reset_iteration_state (None without Ng)."""
        if self.ng is None:
            return None
        return self.t_ng_accepted.view(self.ncol, self.mt.Natom).cpu().numpy()

    # ------------------------------------------------------------------ measurement
    def profile_begin(self, max_launches):
        self._check(self.lib.mali_profile_begin(self._handle, int(max_launches)))

    def profile_end(self):
        """(summed device ms of the fs_gamma_kernel launches since profile_begin, number of launches)"""
        ms, n = C.c_double(0.0), C.c_int32(0)
        self._check(self.lib.mali_profile_end(self._handle, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def model_info(self):
        out = (C.c_int32 * 8)()
        self._check(self.lib.mali_model_info(self._handle, out))
        keys = ('ntile', 'spec_tiles', 'generic_tiles', 'max_slots', 'max_levels', 'row_stride', 'smem_per_warp', 'tma')
        return dict(zip(keys, list(out)))

    def launch_count(self):
        return int(self.lib.mali_launch_count(self._handle))

    def graph_iterations(self):
        """Iterations of iterate_async that were replayed from a captured CUDA graph."""
        return int(self.lib.mali_graph_iterations(self._handle))

    # ------------------------------------------------------------------ results, reference shapes
    def J(self, col=0):
        N, S = self.mt.Nspace, self.mt.Nspect
        return self.t_J[col * self.lay.J:(col + 1) * self.lay.J].view(N, S).t().contiguous().cpu().numpy()

    def I(self, col=0):
        return self.t_I[col * self.lay.I:(col + 1) * self.lay.I].view(self.mt.Nspect, self.mt.Nrays).cpu().numpy()

    def Gamma(self, col=0):
        return self.t_Gamma[col * self.lay.Gamma:(col + 1) * self.lay.Gamma].view(-1, self.mt.Nspace).cpu().numpy()

    def n(self, col=0):
        return self.t_pops[col * self.lay.pops:(col + 1) * self.lay.pops].view(-1, self.mt.Nspace).cpu().numpy()

    def set_n(self, col, n):
        t = torch.from_numpy(np.ascontiguousarray(n, dtype=np.float64).reshape(-1))
        self.t_pops[col * self.lay.pops:(col + 1) * self.lay.pops].copy_(t)

    def atom_Gamma(self, col, a):
        NL = int(self.mt.Nlevel[a])
        g = self.Gamma(col)
        return g[self.mt.g2off[a]:self.mt.g2off[a + 1]].reshape(NL, NL, self.mt.Nspace)

    def atom_n(self, col, a):
        return self.n(col)[self.mt.lvloff[a]:self.mt.lvloff[a + 1]]

    def line_profile(self, col, t):
        """(phi [Nlambda, Nrays, 2, Nspace], wphi [Nspace]) of line t of column col, read back from the device table
        (rh_method.py:224, 235): the table holds hc/4pi*Bij*phi and wlambda*wphi/HC, so the values returned are those
        quantities divided by their constant factors (equal to the profiles the device formed to an ulp)."""
        mt = self.mt
        if not mt.trans[t, 3]:
            raise ValueError('transition %d is a continuum: it has no line profile' % t)
        tile0, ntile, off_tab = C.c_int32(0), C.c_int32(0), C.c_int64(0)
        self._check(self.lib.mali_line_layout(self._handle, t, C.byref(tile0), C.byref(ntile), None, 0, C.byref(off_tab)))
        ent = np.zeros((ntile.value, 4), dtype=np.int32)
        self._check(self.lib.mali_line_layout(self._handle, t, C.byref(tile0), C.byref(ntile),
                                              ent.ctypes.data_as(C.POINTER(C.c_int32)), ntile.value, C.byref(off_tab)))
        N, R, Lw = mt.Nspace, mt.Nrays, int(self.lay.lambda_per_warp)
        Nblue, Nlam = int(mt.trans[t, 4]), int(mt.trans[t, 5])
        cc = self.t_colconst[col * self.lay.colconst:(col + 1) * self.lay.colconst].cpu().numpy()
        tab = cc[off_tab.value:]
        phi = np.zeros((Nlam, R, 2, N))
        wphi = np.zeros(N)
        c0 = mt.lineconst[t, 0]
        from .tables import HC
        kk = np.arange(N)
        for q in range(ntile.value):
            v0, vDir, f, stride = (int(x) for x in ent[q])
            for ls in range(Lw):
                lt = (tile0.value + q) * Lw + ls - Nblue
                if lt < 0 or lt >= Nlam:
                    continue
                for mu in range(R):
                    for d in range(2):
                        phi[lt, mu, d] = tab[v0 + d * vDir + ls * R + mu + kk * stride] / c0
                if lt == 0:
                    wphi = tab[f + ls + kk * stride] * HC / mt.wlambda[mt.toff[t]]
        return phi, wphi

    # ------------------------------------------------------------------ test hooks
    def uv(self, col, t, la, mu, toFrom):
        N = self.mt.Nspace
        out = torch.empty(3, N, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            self._check(self.lib.mali_uv(self._handle, C.byref(self.bufs), col, t, la, mu, int(bool(toFrom)),
                                         C.c_void_p(out[0].data_ptr()), C.c_void_p(out[1].data_ptr()),
                                         C.c_void_p(out[2].data_ptr()), self._stream()))
        o = out.cpu().numpy()
        return o[0], o[1], o[2]   # Uji, Vij, Vji


def rays_angles(mus):
    """The angles of a compute_rays call as a 1-D float64 array: a scalar is one angle; every angle must be finite
    and in (0, 1] (ValueError otherwise)."""
    a = np.asarray(mus, dtype=np.float64)
    if a.ndim == 0:
        a = a.reshape(1)
    if a.ndim != 1 or a.shape[0] == 0:
        raise ValueError('mus must be a scalar or a non-empty 1-D sequence of angles, got shape %s' % (a.shape,))
    ok = np.isfinite(a) & (a > 0.0) & (a <= 1.0)
    if not ok.all():
        raise ValueError('every mu must lie in (0, 1]: got %s' % a[~ok][:8].tolist())
    return np.ascontiguousarray(a)


RAYS_DEPTH_QUANTITIES = ('I', 'chi', 'S', 'tau', 'contrib', 'z_tau1', 'height')


def rays_depth_quantities(quantities):
    """The quantities of a compute_rays_depth call as a tuple in RAYS_DEPTH_QUANTITIES order: None means all of them,
    a string is one name; unknown names, repeats and an empty selection raise ValueError."""
    if quantities is None:
        return RAYS_DEPTH_QUANTITIES
    q = [quantities] if isinstance(quantities, str) else list(quantities)
    unknown = [k for k in q if k not in RAYS_DEPTH_QUANTITIES]
    if unknown:
        raise ValueError('unknown quantities %s (known: %s)' % (unknown, ', '.join(RAYS_DEPTH_QUANTITIES)))
    if not q or len(set(q)) != len(q):
        raise ValueError('quantities must name each of %s at most once, and at least one: got %s'
                         % (', '.join(RAYS_DEPTH_QUANTITIES), q))
    return tuple(k for k in RAYS_DEPTH_QUANTITIES if k in q)


@dataclass
class RayDepthData:
    """Depth-resolved data of up-going rays at the angles `mu` (MaliEngine / Context / BatchContext.compute_rays_depth;
    definitions in include/mali_b200.h).  With a leading column axis from MaliEngine and BatchContext, without it from
    Context: I, chi, S, tau, contrib [.., Nspace, Nspect, nmu] (depth 0 at the top), z_tau1 [.., Nspect, nmu] (NaN where
    tau = 1 is never reached), height [.., Nspace].  Quantities that were not requested are None."""
    mu: np.ndarray
    height: np.ndarray
    I: np.ndarray = None
    chi: np.ndarray = None
    S: np.ndarray = None
    tau: np.ndarray = None
    contrib: np.ndarray = None
    z_tau1: np.ndarray = None

    def column(self, c):
        """The data of column c of a batched result, without the column axis."""
        return RayDepthData(mu=self.mu, **{k: None if v is None else v[c] for k, v in vars(self).items() if k != 'mu'})


@dataclass
class RadiativeRates:
    """Radiative rates of every transition (MaliEngine / Context / BatchContext.compute_rates; definition in
    include/mali_b200.h): Rij, Rji (s^-1) and net = n_i Rij - n_j Rji (m^-3 s^-1), [.., Ntrans, Nspace] in the model's
    transition order, with a leading column axis from MaliEngine and BatchContext, without it from Context."""
    Rij: np.ndarray
    Rji: np.ndarray
    net: np.ndarray

    def column(self, c):
        """The rates of column c of a batched result, without the column axis."""
        return RadiativeRates(Rij=self.Rij[c], Rji=self.Rji[c], net=self.net[c])


def piecewise_linear_1d_batch(z, muz, toFrom, bbc0, bbc1, chi, S, device=None):
    """formal_solver.piecewise_linear_1d for nray independent rays on the GPU (test hook of the fused sweep)."""
    if not torch.cuda.is_available():
        raise RuntimeError('lightspinner_b200 needs a CUDA device: the MALI hot path has no CPU fallback')
    dev = torch.device('cuda', torch.cuda.current_device() if device is None else device)
    lib = _capi.load()
    chi = np.ascontiguousarray(chi, dtype=np.float64)
    nray, N = chi.shape
    td = lambda a, dt=torch.float64: torch.as_tensor(np.ascontiguousarray(a), dtype=dt).to(dev)
    tz, tmu, ttf = td(z), td(muz), td(np.asarray(toFrom, dtype=np.int32), torch.int32)
    tb0, tb1, tchi, tS = td(bbc0), td(bbc1), td(chi), td(S)
    tI = torch.empty(nray, N, dtype=torch.float64, device=dev)
    tP = torch.empty(nray, N, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _capi.check(lib.mali_piecewise_linear_1d(N, nray, *(C.c_void_p(t.data_ptr()) for t in
                                                           (tz, tmu, ttf, tb0, tb1, tchi, tS, tI, tP)),
                                                 C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return tI.cpu().numpy(), tP.cpu().numpy()


def exp_hook(x, device=None):
    """The kernel's exp() on the GPU (test hook): must be bit-identical to libm's exp for 2^-54 <= |x| < 512."""
    dev = torch.device('cuda', torch.cuda.current_device() if device is None else device)
    tx = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64)).to(dev)
    ty = torch.empty_like(tx)
    with torch.cuda.device(dev):
        _capi.check(_capi.load().mali_exp_hook(tx.numel(), C.c_void_p(tx.data_ptr()), C.c_void_p(ty.data_ptr()),
                                               C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return ty.cpu().numpy()


def div_hook(a, b, device=None):
    """The kernels' shared-reciprocal division on the GPU (test hook): returns (q, bad)."""
    dev = torch.device('cuda', torch.cuda.current_device() if device is None else device)
    ta = torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
    tb = torch.as_tensor(np.ascontiguousarray(b, dtype=np.float64)).to(dev)
    tq = torch.empty_like(ta)
    tbad = torch.zeros(ta.numel(), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _capi.check(_capi.load().mali_div_hook(ta.numel(), *(C.c_void_p(t.data_ptr()) for t in (ta, tb, tq, tbad)),
                                               C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return tq.cpu().numpy(), tbad.cpu().numpy()


def fp64_peak(device=None, iters=4096):
    """Measured unfused fp64 mul+add throughput of the device (operations / s)."""
    dev = torch.device('cuda', torch.cuda.current_device() if device is None else device)
    scratch = torch.zeros(8, dtype=torch.float64, device=dev)
    out = C.c_double(0.0)
    with torch.cuda.device(dev):
        _capi.check(_capi.load().mali_fp64_peak(int(iters), C.c_void_p(scratch.data_ptr()), C.byref(out)))
    return out.value


def ng_hook(hist, order, device=None):
    """One Ng extrapolation with the kernels' own code (test hook of mali_iterate_ng): hist [order+2, nvec], newest
    first.  Returns (x*, True) if accepted, else (the newest vector, False)."""
    dev = torch.device('cuda', torch.cuda.current_device() if device is None else device)
    th = torch.as_tensor(np.ascontiguousarray(hist, dtype=np.float64)).to(dev)
    if th.dim() != 2 or th.shape[0] != int(order) + 2:
        raise ValueError('hist must be [order + 2, nvec]')
    out = torch.empty(th.shape[1], dtype=torch.float64, device=dev)
    acc = torch.zeros(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _capi.check(_capi.load().mali_ng_hook(int(order), th.shape[1], C.c_void_p(th.data_ptr()), C.c_void_p(out.data_ptr()),
                                              C.c_void_p(acc.data_ptr()), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return out.cpu().numpy(), bool(acc.item())
