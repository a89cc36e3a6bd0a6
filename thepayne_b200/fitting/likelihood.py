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


class likelihood(object):
    def __init__(self, fitargs, fitpars, runbools, **kwargs):
        self.verbose = kwargs.get('verbose', True)
        self.fitargs = fitargs
        self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool, self.carbon_bool = runbools[:5]
        if self.carbon_bool:
            raise NotImplementedError('carbon_bool is hard-wired off in the reference (fitstar.py:150-154)')
        self.fixedpars = self.fitargs['fixedpars']
        self.precision = kwargs.get('precision', 'parity')
        self.GM = GenMod(precision=self.precision)
        if self.spec_bool:
            self.GM._initspecnn(nnpath=fitargs['specANNpath'], NNtype=self.fitargs.get('NNtype', 'LinNet'),
                                carbon_bool=self.carbon_bool)
        if self.phot_bool:
            self.GM._initphotnn(self.fitargs['obs_phot'].keys(), nnpath=fitargs['photANNpath'])
        self.fitpars_i = free_parameters(fitpars)
        self.ndim = len(self.fitpars_i)
        self.parsdict = {}
        self.engine = Engine(
            spec=self.GM.PP.anns.model if self.spec_bool else None,
            phot=self.GM.fppsed.net if self.phot_bool else None,
            obs_wave=fitargs.get('obs_wave_fit'), obs_flux=fitargs.get('obs_flux_fit'),
            obs_eflux=fitargs.get('obs_eflux_fit'), obs_phot=fitargs.get('obs_phot'),
            fitpars_i=self.fitpars_i, fixedpars=self.fixedpars,
            runbools=[self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool, False],
            precision=self.precision, device=kwargs.get('device'), cont_box=fitargs.get('cont_box'))
        self._explicit = None

    # ------------------------------------------------------------------ reference entry points
    def _set_parsdict(self, pars):
        self.parsdict = {pp: vv for pp, vv in zip(self.fitpars_i, pars)}
        for kk in self.fixedpars.keys():
            self.parsdict[kk] = self.fixedpars[kk]

    def lnlikefn(self, pars):
        """One parameter vector -> float (likelihood.py:42-82)."""
        self._set_parsdict(pars)
        th = np.asarray(pars, dtype=np.float64).reshape(1, self.ndim)
        return float(self.engine.lnlike_batch(th)[0])

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
            fa = self.fitargs
            eng = Engine(spec=self.GM.PP.anns.model if self.spec_bool else None,
                         phot=self.GM.fppsed.net if self.phot_bool else None,
                         obs_wave=fa.get('obs_wave_fit'), obs_flux=fa.get('obs_flux_fit'),
                         obs_eflux=fa.get('obs_eflux_fit'), obs_phot=fa.get('obs_phot'), fitpars_i=names,
                         fixedpars=None if lsf is None else {'Inst_R': lsf},
                         runbools=[self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool, False],
                         precision=self.precision)
            self._explicit = (key, eng)
        return float(self._explicit[1].lnlike_batch(np.array([vals], dtype=np.float64))[0])

    def cont_batch(self, theta):
        """Marginalised continuum: c-hat [B, K] and the packed Cholesky factors [B, K(K+1)/2] (numpy)."""
        coef, chol, _, _ = self.engine.cont_batch(theta)
        return coef.cpu().numpy(), chol.cpu().numpy()

    # ------------------------------------------------------------------ batched entry point
    def lnlike_batch(self, theta):
        """theta [B, ndim] (CUDA float64 tensor, or numpy) -> lnL [B] of the same kind."""
        out = self.engine.lnlike_batch(theta)
        last = theta[-1]
        self._set_parsdict([float(v) for v in (last.tolist() if hasattr(last, 'tolist') else last)])
        return out
