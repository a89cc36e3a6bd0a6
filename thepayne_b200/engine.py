"""Batched likelihood engine: one CUDA context per (emulators, observation, parameter layout).

Thin host-side wrapper over the C ABI (include/payne_b200.h).  PyTorch is used only as the
device-memory / stream provider; the arithmetic all happens inside libpayne_b200.so.

The parameter-vector convention is the reference's (Payne/fitting/likelihood.py:35-72): a
row of ``theta`` holds the free parameters in ``fitpars_i`` order, fixed ones come from
``fixedpars``, and spectral parameters that are neither are NaN.

One context may hold the observations of many stars (``stars=[...]``): the emulators are shared, and
every row of a batch names its star.  Each star may bring its own fixed parameter values, its own subset
of the photometric bands, its own LSF vector and its own parameter layout (free parameters and their
order, continuum order, photometry).  A single-star engine is the case of one star.

Consecutive stars of a set may form a *target* (``targets=[...]``): one physical star observed in several spectra
(echelle orders, spectrograph arms, epochs) that share its labels.  A row of a target batch is evaluated with one
emulator row and one rotation stage, then once per spectrum (member): Doppler shift, instrumental stage (scalar R or
the member's LSF vector), resampling, continuum and chi2.

``binary=True`` models every spectrum as a double-lined binary: the flux-weighted sum of two stars (``set_binary``).

``cont_box=[(lo, hi), ...]`` (per star, or for the single star) integrates the continuum polynomial out instead of
sampling its coefficients (``set_cont_marg``).

A fixed ``Inst_R`` that is a 1-D array is an LSF vector, the dispersion (AA) at every observed pixel,
as in the reference (genmod.py:82-85 passes a non-float inst_R on to getspec's LSF branch,
predictspec.py:265-286).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import PAR_INDEX, PREC


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _pf(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _pd(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _i32(a):
    return np.ascontiguousarray(np.asarray(a).astype(np.int32, casting='same_kind'))


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _nan(want, shape, dev):
    """A NaN-filled float64 output on ``dev``, or None when not wanted."""
    return torch.full(shape, float('nan'), dtype=torch.float64, device=dev) if want else None


# the secondary's own parameters of a binary (``Engine(binary=True)``) and the primary's parameter each one replaces
# (names ending in ``_<digit>`` already mean "spectrum s" in the multi-spectrum fit)
BINARY_PARS = {'Teff_sec': 'Teff', 'log(g)_sec': 'log(g)', '[Fe/H]_sec': '[Fe/H]', '[a/Fe]_sec': '[a/Fe]',
               'Vmic_sec': 'Vmic', 'Vrad_sec': 'Vrad', 'Vrot_sec': 'Vrot'}


def _binary(fitpars_i, fixedpars):
    """PayneBinary (include/payne_b200.h): each secondary parameter and ``Rratio`` from its column in ``fitpars_i`` or
    its value in ``fixedpars``; a secondary parameter in neither is the primary's."""
    b = _lib.PayneBinary()
    for k in range(_lib.NPAR):
        b.col[k], b.fixed[k] = -1, np.nan
    for name, base in BINARY_PARS.items():
        k = PAR_INDEX[base]
        if name in fitpars_i:
            b.col[k] = fitpars_i.index(name)
        elif name in fixedpars:
            b.fixed[k] = float(fixedpars[name])
    b.rratio_col = fitpars_i.index('Rratio') if 'Rratio' in fitpars_i else -1
    b.rratio_fixed = float(fixedpars.get('Rratio', np.nan)) if b.rratio_col < 0 else np.nan
    return b


def _split_fixed(fixedpars):
    """fixedpars -> (PAYNE_NPAR fixed values with NaN where absent, LSF vector or None)."""
    vals = np.full(_lib.NPAR, np.nan)
    lsf = None
    for name, k in PAR_INDEX.items():
        if name not in fixedpars:
            continue
        v = fixedpars[name]
        if name == 'Inst_R' and np.ndim(v) == 1:
            lsf = _f64(v)
        else:
            vals[k] = float(v)
    return vals, lsf


def _layout(fitpars_i, fixed_vals, runbools, precision):
    """PayneLayout (include/payne_b200.h) of one parameter layout (likelihood.py:42-72)."""
    spec_bool, phot_bool, modpoly_bool, photscale_bool = [bool(b) for b in runbools[:4]]
    lay = _lib.PayneLayout()
    lay.ndim = len(fitpars_i)
    for name, k in PAR_INDEX.items():
        lay.col[k] = fitpars_i.index(name) if name in fitpars_i else -1
        lay.fixed[k] = fixed_vals[k]
    pcs = [i for i, p in enumerate(fitpars_i) if 'pc' in p]   # likelihood.py:56-57
    if modpoly_bool and len(pcs) > _lib.MAX_POLY:
        raise ValueError('at most %d continuum coefficients' % _lib.MAX_POLY)
    lay.n_poly = len(pcs) if modpoly_bool else 0
    for i, c in enumerate(pcs[:_lib.MAX_POLY]):
        lay.poly_col[i] = c
    lay.spec_bool, lay.phot_bool = int(spec_bool), int(phot_bool)
    lay.modpoly_bool, lay.photscale_bool = int(modpoly_bool), int(photscale_bool)
    lay.precision = PREC[precision] if isinstance(precision, str) else int(precision)
    return lay


def _specnet_struct(spec, keep):
    """PayneSpecNet (include/payne_b200.h) for a ``synth.SpecNet``-like container; the numpy buffers the
    struct points into are appended to ``keep``."""
    sp = _lib.PayneSpecNet()
    W = [_f32(w) for w in spec.weights]
    b = [_f32(v) for v in spec.biases]
    keep += W + b
    nl = len(W)
    nntype = getattr(spec, 'nntype', 'LinNet')
    if (nl, nntype) not in [(6, 'LinNet'), (4, 'SMLP'), (3, 'YST1'), (4, 'MultiNet')]:
        raise ValueError('unsupported emulator: %d layers of type %s' % (nl, nntype))
    sp.D_in, sp.H1, sp.D_out = W[0].shape[-1], W[0].shape[-2], W[-1].shape[0]
    if nntype == 'MultiNet':   # trainspec_multi.py:29-36, chunk nets stacked along axis 0
        sp.H2 = sp.H3 = sp.H1
        sp.n_groups, sp.group_size = int(W[0].shape[0]), int(spec.chunk)
    elif nl == 6:        # NNmodels.py:147-152
        sp.H2, sp.H3 = W[3].shape[0], W[4].shape[0]
    elif nl == 4:        # NNmodels.py:99-107
        sp.H2, sp.H3 = W[1].shape[0], W[2].shape[0]
    else:                # ystpred.py:25-30
        sp.H2, sp.H3 = W[1].shape[0], 0
    sp.n_layers = nl
    sp.activation = 0 if nntype in ('LinNet', 'MultiNet') else 1
    sp.label_fp32_cast = 0 if nntype == 'YST1' else 1      # ystpred.py:47-50 stays in float64
    for k in range(nl):
        sp.W[k], sp.b[k] = _pf(W[k]), _pf(b[k])
    xmin, xmax, wave = _f64(spec.xmin), _f64(spec.xmax), _f64(spec.wavelength)
    keep += [xmin, xmax, wave]
    sp.xmin, sp.xmax, sp.wavelength = _pd(xmin), _pd(xmax), _pd(wave)
    sp.resolution = float(spec.resolution)
    sp.encode_offset = float(getattr(spec, 'encode_offset', 0.5))
    return sp


class Engine:
    def __init__(self, spec=None, phot=None, obs_wave=None, obs_flux=None, obs_eflux=None,
                 obs_phot=None, fitpars_i=(), fixedpars=None, runbools=(True, False, False, False, False),
                 precision='parity', device=None, stars=None, targets=None, binary=False, cont_box=None):
        """``stars``: instead of ``obs_wave``, ``obs_flux``, ``obs_eflux`` and ``obs_phot``, a list of
        ``{'wave', 'flux', 'eflux', 'phot': {band: (mag, err)}}``, one per star; ``lnlike_batch`` and
        ``model_batch`` then take the star index of every row.  A star may also carry
          ``'fixedpars'``: its fixed parameter values, in place of the shared ``fixedpars``;
          ``'bands'``: the order of its magnitudes (its SED chi2 is summed in that order, likelihood.py:109-112);
          ``'fitpars_i'`` / ``'runbools'``: its own free parameters in its theta order (``pc_k`` among them) and
          run booleans, in place of the shared ones;
          ``'cont_box'``: the box [(lo, hi), ...] of its continuum coefficients, which are then integrated out
          (``set_cont_marg``).
        Its ``'phot'`` keys may be any subset of the photometry net's bands; without ``'bands'`` they go in the
        net's order.  In a photometry engine a star without ``'phot'`` is a star without photometry.  A fixed
        ``Inst_R`` that is a 1-D array is the star's LSF vector (one dispersion per observed pixel); every star
        has one or none does.  ``ndim`` is the largest star's: a row of ``theta`` holds its star's
        ``star_fitpars_i[k]`` in its first ``star_ndim[k]`` columns, and the columns after those are ignored.

        ``targets``: member counts [n_0, n_1, ...] summing to the number of stars; target t is the next n_t stars
        (see ``set_targets``).  Targets work with LSF vectors too: every star then carries its fixed ``Inst_R`` vector
        and none has an ``Inst_R`` column.

        ``binary``: every spectrum is a double-lined binary, read from ``fitpars_i`` / ``fixedpars`` under the names
        ``Teff_sec``, ``log(g)_sec``, ``[Fe/H]_sec``, ``[a/Fe]_sec``, ``Vmic_sec``, ``Vrad_sec``, ``Vrot_sec`` and
        ``Rratio`` (see ``set_binary``).

        ``cont_box``: a single-star engine's ``'cont_box'``."""
        if stars is None:
            stars = [{'wave': obs_wave, 'flux': obs_flux, 'eflux': obs_eflux, 'phot': obs_phot, 'cont_box': cont_box}]
        elif cont_box is not None:
            raise ValueError("with stars=[...], give every star its own 'cont_box'")
        elif any(v is not None for v in (obs_wave, obs_flux, obs_eflux, obs_phot)):
            raise ValueError('give either stars=[...] or obs_wave / obs_flux / obs_eflux / obs_phot, not both')
        stars = list(stars)
        if not stars:
            raise ValueError('stars is empty')
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.PayneError('no CUDA device: thepayne_b200 has no CPU fallback')
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.fitpars_i = list(fitpars_i)
        self.fixedpars = dict(fixedpars or {})
        keep = []   # numpy buffers referenced by the structs until create returns
        # every star's layout: its own free parameters and run booleans or the shared ones; a star of a photometry
        # engine without 'phot' has none
        self.star_fitpars_i = [list(st['fitpars_i']) if st.get('fitpars_i') is not None else self.fitpars_i
                               for st in stars]
        star_rb = [[bool(b) for b in (st['runbools'] if st.get('runbools') is not None else runbools)[:4]]
                   for st in stars]
        for rb, st in zip(star_rb, stars):
            rb[1] = rb[1] and st.get('phot') is not None
        self.star_ndim = [len(f) for f in self.star_fitpars_i]
        self.ndim = max(self.star_ndim)
        own_layouts = any(st.get('fitpars_i') is not None or st.get('runbools') is not None for st in stars) or \
            any(rb != star_rb[0] for rb in star_rb)
        spec_bool, phot_bool, modpoly_bool, photscale_bool = [bool(b) for b in runbools[:4]]
        if own_layouts:
            # the context layout is star 0's; its phot_bool says whether the engine has a photometry net
            spec_bool, modpoly_bool, photscale_bool = star_rb[0][0], star_rb[0][2], star_rb[0][3]
            phot_bool = any(rb[1] for rb in star_rb)
        elif phot_bool and any(st.get('phot') is None for st in stars):
            raise ValueError('phot_bool set but no photometry emulator / observation given')
        shared_vals, shared_lsf = _split_fixed(self.fixedpars)
        lay = _layout(self.star_fitpars_i[0] if own_layouts else self.fitpars_i, shared_vals,
                      [spec_bool, phot_bool, modpoly_bool, photscale_bool], precision)

        sp = None
        if spec_bool:
            if spec is None:
                raise ValueError('spec_bool set but no spectrum emulator given')
            sp = _specnet_struct(spec, keep)
            self.D_in, self.D_out = int(sp.D_in), int(sp.D_out)
        self.n_stars = len(stars)
        obs = (_lib.PayneObs * self.n_stars)()
        opts = (_lib.PayneStarOpts * self.n_stars)()      # all fields NULL: the star has no option
        self.star_fixedpars = [dict(st['fixedpars']) if st.get('fixedpars') is not None else self.fixedpars
                               for st in stars]
        for k, st in enumerate(stars):
            vals, lsf = (shared_vals, shared_lsf) if st.get('fixedpars') is None else _split_fixed(st['fixedpars'])
            if own_layouts:
                sl = _layout(self.star_fitpars_i[k], vals, star_rb[k], precision)
                keep.append(sl)
                opts[k].layout = C.pointer(sl)
            elif st.get('fixedpars') is not None:
                keep.append(vals)
                opts[k].fixed = _pd(vals)
            if lsf is not None:
                if not spec_bool:
                    raise ValueError('an LSF vector (fixed Inst_R array) needs the spectrum emulator (star %d)' % k)
                if len(lsf) != len(st['wave']):
                    raise ValueError('star %d: the LSF vector needs one dispersion per observed pixel (%d, got %d)'
                                     % (k, len(st['wave']), len(lsf)))
                keep.append(lsf)
                opts[k].lsf = _pd(lsf)
        self.n_obs_star = [0] * self.n_stars
        if spec_bool:
            for k, st in enumerate(stars):
                ow, of, oe = _f64(st['wave']), _f64(st['flux']), _f64(st['eflux'])
                if not (len(ow) == len(of) == len(oe)):
                    raise ValueError('observed wave/flux/eflux lengths differ (star %d)' % k)
                keep += [ow, of, oe]
                obs[k].n_obs, obs[k].wave, obs[k].flux, obs[k].eflux = len(ow), _pd(ow), _pd(of), _pd(oe)
                self.n_obs_star[k] = len(ow)
        self.n_obs = max(self.n_obs_star)          # the largest star's
        ph = None
        self.bands = []
        self.star_bands = [[] for _ in stars]
        if phot_bool:
            if phot is None:
                raise ValueError('phot_bool set but no photometry emulator / observation given')
            self.bands = list(phot.bands)
            ph = _lib.PaynePhotNet()
            arrs = [_f32(phot.w1), _f32(phot.b1), _f32(phot.w2), _f32(phot.b2),
                    _f32(np.asarray(phot.w3).reshape(len(self.bands), -1)), _f32(np.asarray(phot.b3).reshape(-1))]
            keep += arrs
            ph.nb, ph.H = arrs[0].shape[0], arrs[0].shape[1]
            ph.w1, ph.b1, ph.w2, ph.b2, ph.w3, ph.b3 = [_pf(a) for a in arrs]
            pxmin, pxmax, hiav = _f64(phot.xmin), _f64(phot.xmax), _f64(phot.hiav)
            keep += [pxmin, pxmax, hiav]
            ph.xmin, ph.xmax, ph.hiav = _pd(pxmin), _pd(pxmax), _pd(hiav)
            for k, st in enumerate(stars):
                if not star_rb[k][1]:
                    continue                                # a star without photometry: nb = 0
                bands = list(st['bands']) if st.get('bands') is not None else \
                    [b for b in self.bands if b in st['phot']]
                unknown = [b for b in list(st['phot']) + bands if b not in self.bands]
                if unknown:
                    raise ValueError('star %d: bands %s are not in the photometry net' % (k, sorted(set(unknown))))
                if sorted(bands) != sorted(st['phot']) or len(set(bands)) != len(bands):
                    raise ValueError("star %d: 'bands' must list each of its 'phot' keys once" % k)
                self.star_bands[k] = bands
                mag = _f64([st['phot'][b][0] for b in bands])
                err = _f64([st['phot'][b][1] for b in bands])
                keep += [mag, err]
                obs[k].nb, obs[k].phot_mag, obs[k].phot_err = len(bands), _pd(mag), _pd(err)
                if bands != self.bands:
                    idx = np.array([self.bands.index(b) for b in bands], dtype=np.int32)
                    keep.append(idx)
                    opts[k].band = idx.ctypes.data_as(C.POINTER(C.c_int32))
        self.nb = len(self.bands)

        ctx = C.c_void_p()
        _lib.check(self.lib.payne_ctx_create_stars_opts(C.byref(sp) if sp is not None else None,
                                                         C.byref(ph) if ph is not None else None,
                                                         obs, opts, self.n_stars, C.byref(lay), self.device,
                                                         C.byref(ctx)))
        self._ctx = ctx
        del keep
        self.n_targets = 0
        if targets is not None:
            self.set_targets(targets)
        self.binary = False
        if binary:
            self.set_binary()
        self.cont_k = None
        boxes = [st.get('cont_box') for st in stars]
        if any(b is not None for b in boxes):
            self.set_cont_marg(boxes)

    # ------------------------------------------------------------------ lifecycle
    def close(self):
        if getattr(self, '_ctx', None):
            self.lib.payne_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def query(self, key):
        return int(self.lib.payne_ctx_query(self._ctx, key.encode()))

    def set(self, key, value):
        if key == 'precision' and isinstance(value, str):
            value = PREC[value]
        _lib.check(self.lib.payne_ctx_set(self._ctx, key.encode(), int(value)))

    def attach_continuum(self, cont):
        """Continuum emulator of ``PayneSpecPredict(Cnnpath=...)`` (predictspec.py:96-102): every model
        spectrum is multiplied by the normalised F_lambda continuum interpolated onto the emulator grid
        (predictspec.py:208-226)."""
        keep = []
        sp = _specnet_struct(cont, keep)
        _lib.check(self.lib.payne_ctx_attach_continuum(self._ctx, C.byref(sp)))

    def set_lsf(self, lsf):
        """LSF vector: the dispersion (AA) at every observed pixel (predictspec.py:265-286); None switches
        back to the scalar ``Inst_R`` stage."""
        if lsf is None:
            _lib.check(self.lib.payne_ctx_set_lsf(self._ctx, None, 0))
            return
        v = _f64(lsf)
        if v.ndim != 1 or len(v) != self.n_obs:
            raise ValueError('the LSF vector needs one dispersion per observed pixel (%d)' % self.n_obs)
        _lib.check(self.lib.payne_ctx_set_lsf(self._ctx, v.ctypes.data, len(v)))

    def set_targets(self, counts):
        """Group the stars into targets: target t is the next ``counts[t]`` stars, its members, which share the
        emulator labels and ``Vrot`` (same columns or fixed values) and may differ in ``Vrad``, ``Inst_R``, pixels and
        continuum order; only the first member may have photometry.  With LSF vectors each member is broadened by its
        own vector, on any emulator grid the LSF tail takes, and a member with an ``Inst_R`` column is refused (nothing
        would read it).  Without them the emulator grid must be uniform in ln wavelength.  None removes the targets."""
        if counts is None:
            _lib.check(self.lib.payne_ctx_set_targets(self._ctx, None, 0))
            self.n_targets = 0
            return
        counts = [int(n) for n in counts]
        if not counts or min(counts) < 1 or sum(counts) != self.n_stars:
            raise ValueError('targets: member counts >= 1 that sum to the number of stars (%d)' % self.n_stars)
        first = np.ascontiguousarray(np.concatenate([[0], np.cumsum(counts)]), dtype=np.int32)
        _lib.check(self.lib.payne_ctx_set_targets(self._ctx, first.ctypes.data, len(counts)))
        self.n_targets = len(counts)
        self.target_first = first
        self.target_members = [list(range(first[t], first[t + 1])) for t in range(len(counts))]
        # a target's model row: its members' pixels back to back
        self.target_n_obs = [sum(self.n_obs_star[k] for k in m) for m in self.target_members]
        self.target_kmax = max(counts)

    def set_binary(self, on=True, fitpars_i=None, fixedpars=None):
        """Model every spectrum as a double-lined binary: (a_1 + k a_2) / (1 + k) times the continuum, a_c the
        spectrum of component c before the continuum and k = Rratio^2 B(lambda, Teff_1) / B(lambda, Teff_2) the
        blackbody flux ratio (include/payne_b200.h, PayneBinary).  The secondary's parameters and ``Rratio`` come from
        ``fitpars_i`` / ``fixedpars`` (default: the engine's) under the names of ``BINARY_PARS`` and ``Rratio``; a
        secondary parameter in neither is the primary's.  ``Inst_R`` and the continuum are shared.  ``on=False``
        removes it.  Photometry, LSF vectors, targets, per-star layouts and grids without the fast tail are refused."""
        if not on:
            _lib.check(self.lib.payne_ctx_set_binary(self._ctx, None))
            self.binary = False
            return
        b = _binary(list(self.fitpars_i if fitpars_i is None else fitpars_i),
                    dict(self.fixedpars if fixedpars is None else fixedpars))
        _lib.check(self.lib.payne_ctx_set_binary(self._ctx, C.byref(b)))
        self.binary = True

    def set_cont_marg(self, boxes):
        """Integrate every star's continuum polynomial out (include/payne_b200.h, PayneContMarg): ``boxes[k]`` is star
        k's [(lo, hi), ...], one pair per coefficient, whose widths normalise the flat prior of the integral; None for
        every star removes the setting.  lnL is then -0.5 (Q + chi2_sed) + M, Q the chi2 at the best-fitting
        coefficients and M the log of the Gaussian integral over them, and the model rows are at those coefficients.
        A star with the setting has no ``pc_k`` among its free parameters."""
        if boxes is None or all(b is None for b in boxes):
            _lib.check(self.lib.payne_ctx_set_cont_marg(self._ctx, None))
            self.cont_k = None
            return
        if len(boxes) != self.n_stars:
            raise ValueError('set_cont_marg: one box list per star (%d)' % self.n_stars)
        arr = (_lib.PayneContMarg * self.n_stars)()
        for k, b in enumerate(boxes):
            b = [] if b is None else [tuple(map(float, lh)) for lh in b]
            if len(b) > _lib.MAX_POLY:
                raise ValueError('star %d: at most %d continuum coefficients' % (k, _lib.MAX_POLY))
            arr[k].n_coef = len(b)
            for i, (lo, hi) in enumerate(b):
                arr[k].lo[i], arr[k].hi[i] = lo, hi
        _lib.check(self.lib.payne_ctx_set_cont_marg(self._ctx, arr))
        self.cont_k = [int(arr[k].n_coef) for k in range(self.n_stars)]

    def cont_batch(self, theta, star=None):
        """With the continuum integrated out: the best-fitting coefficients [B, K] (K the largest star's; a row's
        columns beyond its star's K stay NaN), the Cholesky factor L of G = L L^T as packed lower triangles
        [B, K(K+1)/2] (row by row), Q (the chi2 at those coefficients) [B] and lnL [B], as CUDA float64 tensors.  A
        draw of the coefficients' conditional posterior is coef + L^-T z, z ~ N(0, I)."""
        if self.cont_k is None:
            raise ValueError('no continuum marginalisation: set_cont_marg first')
        th, sv, lnl, st = self._dev_args(theta, star, copy=True)
        B, dev = th.shape[0], th.device
        kc = max(self.cont_k)
        coef, chol, chi2 = _nan(True, (B, kc), dev), _nan(True, (B, kc * (kc + 1) // 2), dev), _nan(True, (B,), dev)
        _lib.check(self.lib.payne_cont_batch_stars(
            self._ctx, th.data_ptr(), _ptr(sv), B, th.shape[1],
            coef.data_ptr(), coef.shape[1], chol.data_ptr(), chol.shape[1], chi2.data_ptr(), lnl.data_ptr(), st))
        return coef, chol, chi2, lnl

    def cont_batch_targets(self, theta, target):
        """``cont_batch`` for targets: the members' coefficients and Cholesky factors back to back in member order,
        and Q [B, target_kmax] per member."""
        if self.cont_k is None:
            raise ValueError('no continuum marginalisation: set_cont_marg first')
        if not self.n_targets:
            raise ValueError('no targets: set_targets first')
        th, tv, lnl, st = self._dev_args(theta, target, copy=True)
        B, dev = th.shape[0], th.device
        kc = max(sum(self.cont_k[k] for k in m) for m in self.target_members)
        kl = max(sum(self.cont_k[k] * (self.cont_k[k] + 1) // 2 for k in m) for m in self.target_members)
        coef, chol, chi2 = _nan(True, (B, kc), dev), _nan(True, (B, kl), dev), _nan(True, (B, self.target_kmax), dev)
        _lib.check(self.lib.payne_cont_batch_targets(
            self._ctx, th.data_ptr(), _ptr(tv), B, th.shape[1], coef.data_ptr(), kc, chol.data_ptr(), kl,
            chi2.data_ptr(), self.target_kmax, lnl.data_ptr(), st))
        return coef, chol, chi2, lnl

    def lnlike_batch_binary(self, theta, star=None):
        """lnL of every row as a binary, ``theta`` and ``star`` as in ``lnlike_batch`` (None: star 0)."""
        return self._lnlike(self.lib.payne_lnlike_batch_binary, self.lib.payne_lnlike_batch_binary_host, theta, star,
                            'star')

    def model_batch_binary(self, theta, star=None, want_flux=True, want_comp=True):
        """Model spectra [B, n_obs], the components' spectra before the continuum [B, 2, n_obs] and lnL [B] of every
        row as a binary, as CUDA float64 tensors (the pixels beyond a row's star stay NaN)."""
        th, sv, lnl, st = self._dev_args(theta, star, copy=True)
        B, dev = th.shape[0], th.device
        flux = _nan(want_flux, (B, self.n_obs), dev)
        comp = _nan(want_comp, (B, 2, self.n_obs), dev)
        _lib.check(self.lib.payne_model_batch_binary(
            self._ctx, th.data_ptr(), _ptr(sv), B, th.shape[1], _ptr(flux), self.n_obs, _ptr(comp), lnl.data_ptr(), st))
        return flux, comp, lnl

    def lnlike_batch_targets(self, theta, target):
        """lnL of every row against its target: ``target`` [B], as ``star`` in ``lnlike_batch`` (int32 CUDA tensor
        with a CUDA theta: stream-ordered, an index outside [0, n_targets) gives NaN and status bit 2; else numpy
        through the host entry, which refuses such an index)."""
        if not self.n_targets:
            raise ValueError('no targets: set_targets first')
        return self._lnlike(self.lib.payne_lnlike_batch_targets, self.lib.payne_lnlike_batch_targets_host, theta,
                            target, 'target')

    def model_batch_targets(self, theta, target, want_flux=True, want_chi2=True, want_mags=True):
        """Model spectra [B, max target_n_obs] (row p: its members' spectra back to back in member order, the rest
        NaN), chi2 [B, target_kmax] (chi2[p, m] of member m, the rest NaN), the first member's magnitudes [B, nb] and
        lnL [B], as CUDA float64 tensors."""
        if not self.n_targets:
            raise ValueError('no targets: set_targets first')
        th, tv, lnl, st = self._dev_args(theta, target, copy=True)
        B, dev = th.shape[0], th.device
        nf = max(self.target_n_obs)
        flux = _nan(want_flux, (B, nf), dev)
        chi2 = _nan(want_chi2, (B, self.target_kmax), dev)
        mags = _nan(want_mags and self.nb, (B, self.nb), dev)
        _lib.check(self.lib.payne_model_batch_targets(
            self._ctx, th.data_ptr(), _ptr(tv), B, th.shape[1], _ptr(flux), nf, _ptr(chi2), self.target_kmax,
            _ptr(mags), lnl.data_ptr(), st))
        return flux, chi2, mags, lnl

    def last_ms(self, which):
        return float(self.lib.payne_ctx_last_ms(self._ctx, {'mlp': 0, 'tail': 1, 'phot': 2}[which]))

    # ------------------------------------------------------------------ compute
    def _theta_dev(self, theta):   # [B, ndim]: row p's star reads its first star_ndim columns
        if not (theta.is_cuda and theta.dtype == torch.float64 and theta.dim() == 2):
            raise ValueError('theta must be a 2-D float64 CUDA tensor')
        if theta.shape[1] != self.ndim:
            raise ValueError('theta has %d columns, layout expects %d' % (theta.shape[1], self.ndim))
        return theta.contiguous()

    def _dev_args(self, theta, idx, copy):
        """A device entry's inputs: theta [B, ndim] and idx [B] (every row's star or target; None: star 0) as CUDA
        tensors, an empty float64 lnL [B] on their device and that device's current stream.  ``copy``: numpy and CPU
        inputs are copied to the engine's device first; else theta must be a CUDA tensor and idx an int32 CUDA
        tensor on its device."""
        if copy:
            theta = theta if isinstance(theta, torch.Tensor) else torch.from_numpy(_f64(theta))
            theta = theta.to(torch.device('cuda', self.device))
        th = self._theta_dev(theta)
        B, dev = th.shape[0], th.device
        if idx is not None:
            if copy:
                idx = (idx if isinstance(idx, torch.Tensor) else torch.from_numpy(_i32(idx))).to(dev)
            if not (isinstance(idx, torch.Tensor) and idx.is_cuda and idx.dtype == torch.int32):
                raise ValueError('with a CUDA theta, star must be an int32 CUDA tensor')
            if idx.shape != (B,) or idx.device != dev:
                raise ValueError('star must be [%d] on %s' % (B, dev))
            idx = idx.contiguous()
        return th, idx, torch.empty(B, dtype=torch.float64, device=dev), torch.cuda.current_stream(dev).cuda_stream

    def _lnlike(self, dev_entry, host_entry, theta, idx, what):
        """lnL [B] of theta [B, ndim] and idx [B] (every row's star or target, ``what``; None: star 0): with a CUDA
        theta a CUDA tensor from the device entry ``dev_entry``, else numpy from the host-buffer entry ``host_entry``,
        theta and idx then as anything numpy takes."""
        if isinstance(theta, torch.Tensor) and theta.is_cuda:
            th, iv, lnl, st = self._dev_args(theta, idx, copy=False)
            _lib.check(dev_entry(self._ctx, th.data_ptr(), _ptr(iv), th.shape[0], th.shape[1], lnl.data_ptr(), st))
            return lnl
        th = _f64(theta)
        if th.ndim != 2 or th.shape[1] != self.ndim:
            raise ValueError('theta must be [B, %d]' % self.ndim)
        iv = None
        if idx is not None:
            iv = _i32(idx.cpu().numpy() if isinstance(idx, torch.Tensor) else idx)
            if iv.shape != (th.shape[0],):
                raise ValueError('%s must be [%d]' % (what, th.shape[0]))
        out = np.empty(th.shape[0], dtype=np.float64)
        _lib.check(host_entry(self._ctx, th.ctypes.data, iv.ctypes.data if iv is not None else None, th.shape[0],
                              th.shape[1], out.ctypes.data))
        return out

    def lnlike_batch(self, theta, star=None):
        """theta: [B, ndim] float64.  CUDA tensor -> CUDA tensor [B] (stream-ordered, no sync);
        numpy / CPU tensor -> numpy [B] through the host-buffer entry point.  ``star``: [B] star index of
        every row, an int32 CUDA tensor with a CUDA theta, anything numpy takes otherwise (None: star 0,
        which only a single-star engine accepts).  On the device a row with an index outside
        [0, n_stars) gets NaN and sets status bit 2; the host path refuses such an index."""
        return self._lnlike(self.lib.payne_lnlike_batch_stars, self.lib.payne_lnlike_batch_stars_host, theta, star,
                            'star')

    def model_batch(self, theta, star=None, want_flux=True, want_mags=True):
        """Model spectra [B, n_obs], magnitudes [B, nb] and lnL [B] as CUDA float64 tensors.  With several
        stars, n_obs is the largest star's: row p holds the first ``n_obs_star[star[p]]`` pixels, the rest
        stay NaN; likewise row p of the magnitudes holds its star's ``star_bands[star[p]]``, the rest NaN.  ``star`` as in ``lnlike_batch`` (numpy is copied to the device)."""
        th, sv, lnl, st = self._dev_args(theta, star, copy=True)
        B, dev = th.shape[0], th.device
        flux = _nan(want_flux and self.n_obs, (B, self.n_obs), dev)
        mags = _nan(want_mags and self.nb, (B, self.nb), dev)
        _lib.check(self.lib.payne_model_batch_stars(
            self._ctx, th.data_ptr(), _ptr(sv), B, th.shape[1], _ptr(flux), self.n_obs, _ptr(mags), lnl.data_ptr(), st))
        return flux, mags, lnl

    def ann_eval(self, x):
        """Emulator forward pass: labels [B, D_in] -> flux [B, D_out] float32 (CUDA tensor)."""
        dev = torch.device('cuda', self.device)
        if not isinstance(x, torch.Tensor):
            x = torch.from_numpy(np.ascontiguousarray(np.atleast_2d(np.asarray(x, dtype=np.float64))))
        x = x.to(dev, dtype=torch.float64).contiguous()
        if x.shape[1] != self.D_in:
            raise ValueError('labels have %d columns, emulator expects %d' % (x.shape[1], self.D_in))
        ldy = (self.D_out + 3) // 4 * 4
        y = torch.empty((x.shape[0], ldy), dtype=torch.float32, device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(self.lib.payne_ann_eval(self._ctx, x.data_ptr(), x.shape[0], y.data_ptr(), ldy, st))
        return y[:, :self.D_out]


def engine_from_config(cfg, precision='parity', device=None):
    """Engine for a ``thepayne_b200.synth.SynthConfig``."""
    return Engine(spec=cfg.spec if cfg.runbools[0] else None, phot=cfg.phot if cfg.runbools[1] else None,
                  obs_wave=cfg.obs_wave, obs_flux=cfg.obs_flux, obs_eflux=cfg.obs_eflux,
                  obs_phot=cfg.obs_phot, fitpars_i=cfg.fitpars_i, fixedpars=cfg.fixedpars,
                  runbools=cfg.runbools, precision=precision, device=device)
