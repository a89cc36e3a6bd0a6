"""Drop-in ``likelihood`` class: same constructor and ``lnlikefn`` / ``lnlike`` signatures as
``Payne/fitting/likelihood.py:5-117`` plus ``lnlike_batch`` for a whole set of live points.

The caller (dynesty through ``fitstar.lnprobfn``, fitstar.py:647-659) reads ``parsdict`` after
``lnlikefn``; after a batched call it holds the LAST row, which is what the reference's logging
expects (fitstar.py:342-348).

A fixed ``Inst_R`` that is a 1-D array is the LSF vector of the observation (one dispersion per observed
pixel), as in the reference: lnlikefn passes it on to genspec, which hands a non-float ``inst_R`` to getspec's
LSF branch (genmod.py:82-85, predictspec.py:265-286).

``fitargs['cont_box']`` (``FitPayne`` with ``spec['modpoly_marginal']``) integrates the continuum coefficients out
(``Engine.set_cont_marg``); ``cont_batch`` gives their best-fitting values and Cholesky factors.
"""
from __future__ import annotations

import numpy as np

from ..engine import Engine
from .genmod import GenMod

_SPEC = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Vmic', 'Inst_R']


def free_parameters(fitpars):
    """Names of the sampled parameters in sampler order (likelihood.py:35-40)."""
    return [pp for pp in fitpars[0] if fitpars[1][pp]]


def _genmod(fitargs, runbools, precision, bands=None):
    """The run booleans (spec, phot, modpoly, photscale, carbon) and the emulators (``GenMod``) of a fit: the spectrum
    net of ``specANNpath`` / ``NNtype`` with spectra, the photometry net of ``photANNpath`` for ``bands`` (default:
    the ``obs_phot`` bands) with photometry."""
    runbools = tuple(runbools[:5])
    if runbools[4]:
        raise NotImplementedError('carbon_bool is hard-wired off in the reference (fitstar.py:150-154)')
    GM = GenMod(precision=precision)
    if runbools[0]:
        GM._initspecnn(nnpath=fitargs['specANNpath'], NNtype=fitargs.get('NNtype', 'LinNet'))
    if runbools[1]:
        GM._initphotnn(fitargs['obs_phot'].keys() if bands is None else bands, nnpath=fitargs['photANNpath'])
    return runbools, GM


class _Likelihood(object):
    """The interface every kind of fit gives its sampler: ``fitpars_i`` (the sampled parameters in theta order),
    ``ndim``, ``fixedpars``, ``parsdict`` (the last row evaluated, fixed values included), ``lnlikefn`` for one row
    and ``lnlike_batch`` for many.  A kind of fit supplies ``_lnlike(theta)``: lnL of rows [B, ndim] (CUDA float64
    tensor, or numpy) of the same kind; ``_lnlike_batch`` may route the batched calls elsewhere.  With continuum
    marginalisation it supplies ``_cont(theta)`` too: ``Engine.cont_batch``'s outputs for the rows."""

    def __init__(self, fitpars_i, fixedpars):
        self.fitpars_i = fitpars_i
        self.ndim = len(fitpars_i)
        self.fixedpars = fixedpars
        self.parsdict = {}

    def _set_parsdict(self, pars):
        self.parsdict = {pp: vv for pp, vv in zip(self.fitpars_i, pars)}
        for kk in self.fixedpars.keys():
            self.parsdict[kk] = self.fixedpars[kk]

    def lnlikefn(self, pars):
        """One parameter vector -> float (likelihood.py:42-82)."""
        self._set_parsdict(pars)
        th = np.asarray(pars, dtype=np.float64).reshape(1, self.ndim)
        return float(self._lnlike(th)[0])

    def lnlike_batch(self, theta):
        """theta [B, ndim] (CUDA float64 tensor, or numpy) -> lnL [B] of the same kind."""
        out = self._lnlike_batch(theta)
        last = theta[-1]
        self._set_parsdict([float(v) for v in (last.tolist() if hasattr(last, 'tolist') else last)])
        return out

    def _lnlike_batch(self, theta):
        return self._lnlike(theta)

    def cont_batch(self, theta):
        """Marginalised continuum: c-hat [B, K] and the packed Cholesky factors [B, K(K+1)/2] (numpy)."""
        coef, chol, _, _ = self._cont(theta)
        return coef.cpu().numpy(), chol.cpu().numpy()

    def _cont(self, theta):
        raise NotImplementedError('%s integrates no continuum out' % type(self).__name__)


class likelihood(_Likelihood):
    def __init__(self, fitargs, fitpars, runbools, **kwargs):
        self.verbose = kwargs.get('verbose', True)
        self.fitargs = fitargs
        self.precision = kwargs.get('precision', 'parity')
        (self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool, self.carbon_bool), self.GM = \
            _genmod(fitargs, runbools, self.precision)
        super().__init__(free_parameters(fitpars), fitargs['fixedpars'])
        self.engine = self._engine(self.fitpars_i, self.fixedpars, device=kwargs.get('device'),
                                   cont_box=fitargs.get('cont_box'))
        self._explicit = None

    def _engine(self, fitpars_i, fixedpars, **kwargs):
        """An engine on this fit's observation and emulators for the layout ``fitpars_i`` / ``fixedpars``."""
        fa = self.fitargs
        return Engine(spec=self.GM.PP.anns.model if self.spec_bool else None,
                      phot=self.GM.fppsed.net if self.phot_bool else None,
                      obs_wave=fa.get('obs_wave_fit'), obs_flux=fa.get('obs_flux_fit'),
                      obs_eflux=fa.get('obs_eflux_fit'), obs_phot=fa.get('obs_phot'),
                      fitpars_i=fitpars_i, fixedpars=fixedpars,
                      runbools=[self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool, False],
                      precision=self.precision, **kwargs)

    def _lnlike(self, theta):
        return self.engine.lnlike_batch(theta)

    def _cont(self, theta):
        return self.engine.cont_batch(theta)

    def lnlike(self, specpars=None, photpars=None):
        """Explicit ``specpars`` / ``photpars`` lists as built by lnlikefn (likelihood.py:84-117)."""
        names, vals = [], []
        lsf = None
        if self.spec_bool:
            sp = list(specpars)
            if np.ndim(sp[7]) == 1:                     # an LSF vector in place of Inst_R (genmod.py:82-85)
                lsf = np.ascontiguousarray(sp[7], dtype=np.float64)
                names += [n for n in _SPEC if n != 'Inst_R'] + ['pc_%d' % k for k in range(len(sp) - 8)]
                vals += [float(v) for v in sp[:7] + sp[8:]]
            else:
                names += _SPEC + ['pc_%d' % k for k in range(len(sp) - 8)]
                vals += [float(v) for v in sp]
        if self.phot_bool:
            pp = list(photpars)
            pn = ['log(A)', 'Av'] if self.photscale_bool else ['log(R)', 'Dist', 'Av']
            for n, v in zip(['Teff', 'log(g)', '[Fe/H]', '[a/Fe]'] + pn, pp):
                if n in names:
                    continue
                names.append(n)
                vals.append(float(v))
        key = (tuple(names), None if lsf is None else lsf.tobytes())
        if self._explicit is None or self._explicit[0] != key:
            if self._explicit is not None:
                self._explicit[1].close()
            self._explicit = (key, self._engine(names, None if lsf is None else {'Inst_R': lsf}))
        return float(self._explicit[1].lnlike_batch(np.array([vals], dtype=np.float64))[0])
