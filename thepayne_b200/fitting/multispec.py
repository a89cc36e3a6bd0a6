"""``MultiSpecLikelihood``: one star observed in several spectra (echelle orders, spectrograph arms).

The spectra are the members of one target of an observation set (``Engine(stars=[...], targets=[S])``): the labels,
``Vrad`` and ``Vrot`` are shared, spectrum s has its own resolving power ``Inst_R_<s>`` and continuum coefficients
``pc_<s>_<k>``, and the photometry belongs to the first spectrum.  A sampler row holds every free parameter once; each
spectrum's layout reads its own columns under the reference's names (``Inst_R_<s>`` as ``Inst_R``, ``pc_<s>_<k>`` as
``pc_k``), so lnL = -0.5 (chi2_0 + ... + chi2_{S-1} + chi2_sed) with each chi2_s what a single-spectrum ``likelihood``
of spectrum s gives.  ``fitargs['spectra']`` is the list of ``{'obs_wave_fit', 'obs_flux_fit', 'obs_eflux_fit'}``
(``FitPayne`` builds it from a list-valued ``inputdict['spec']``).

``fitargs['spectra'][s]['cont_box']`` (``FitPayne`` with ``modpoly_marginal``) integrates spectrum s's continuum
coefficients out (``Engine.set_cont_marg``); ``cont_batch`` gives every spectrum's best-fitting values back to back.

A fixed ``Inst_R_<s>`` that is a 1-D array is spectrum s's LSF vector, one dispersion (AA) per fitted pixel of that
spectrum, as a fixed ``Inst_R`` array is in the single-spectrum ``likelihood``.  Every spectrum has one or none does.
"""
from __future__ import annotations

import re

import numpy as np
import torch

from ..engine import Engine
from .likelihood import _genmod, _Likelihood, free_parameters

_PHOT = ['log(R)', 'Dist', 'log(A)', 'Av', 'Rv']


def spectrum_name(name, s):
    """The reference name under which spectrum s reads sampler parameter ``name``; None: not spectrum s's."""
    m = re.fullmatch(r'Inst_R_(\d+)', name)
    if m:
        return 'Inst_R' if int(m.group(1)) == s else None
    m = re.fullmatch(r'pc_(\d+)_(\d+)', name)
    if m:
        return 'pc_%s' % m.group(2) if int(m.group(1)) == s else None
    return name


class MultiSpecLikelihood(_Likelihood):
    def __init__(self, fitargs, fitpars, runbools, **kwargs):
        self.fitargs = fitargs
        if not runbools[0]:
            raise ValueError('MultiSpecLikelihood needs spectra')
        fixedpars = fitargs['fixedpars']
        spectra = fitargs['spectra']
        lsf = [np.ndim(fixedpars.get('Inst_R_%d' % s, 0.0)) == 1 for s in range(len(spectra))]
        if any(lsf) and not all(lsf):
            raise ValueError('spectra %s have an LSF vector (a fixed Inst_R_<s> array) and spectra %s do not: every '
                             'spectrum has one or none does' % ([s for s, v in enumerate(lsf) if v],
                                                                [s for s, v in enumerate(lsf) if not v]))
        self.precision = kwargs.get('precision', 'parity')
        (self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool, self.carbon_bool), self.GM = \
            _genmod(fitargs, runbools, self.precision)
        super().__init__(free_parameters(fitpars), fixedpars)
        stars = []
        for s, sp in enumerate(spectra):
            fit = [spectrum_name(p, s) for p in self.fitpars_i]
            if s > 0:                                        # the photometry is the first spectrum's
                fit = [None if p in _PHOT else p for p in fit]
            fit = [p if p is not None else 'pad' for p in fit]
            fixed = {}
            for kk, v in self.fixedpars.items():
                name = spectrum_name(kk, s)
                if name is not None and not (s > 0 and name in _PHOT):
                    fixed[name] = v
            poly = any(p.startswith('pc_') for p in fit)
            st = {'wave': sp['obs_wave_fit'], 'flux': sp['obs_flux_fit'], 'eflux': sp['obs_eflux_fit'],
                  'fitpars_i': fit, 'fixedpars': fixed,
                  'runbools': [True, bool(self.phot_bool) and s == 0, poly, bool(self.photscale_bool)],
                  'cont_box': sp.get('cont_box')}
            if self.phot_bool and s == 0:
                st['phot'] = fitargs['obs_phot']
            stars.append(st)
        if len({s['runbools'][2] for s in stars}) > 1:
            raise ValueError('every spectrum has a continuum polynomial (modpoly) or none does')
        self.engine = Engine(spec=self.GM.PP.anns.model, phot=self.GM.fppsed.net if self.phot_bool else None,
                             stars=stars, targets=[len(stars)],
                             runbools=[True, self.phot_bool, self.modpoly_bool, self.photscale_bool, False],
                             precision=self.precision, device=kwargs.get('device'))

    def _lnlike(self, theta):
        if isinstance(theta, torch.Tensor) and theta.is_cuda:
            target = torch.zeros(theta.shape[0], dtype=torch.int32, device=theta.device)
        else:
            target = np.zeros(len(theta), np.int32)
        return self.engine.lnlike_batch_targets(theta, target)

    def _cont(self, theta):
        return self.engine.cont_batch_targets(theta, np.zeros(len(theta), np.int32))
