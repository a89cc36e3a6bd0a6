"""``BinaryLikelihood``: a double-lined binary (SB2), one observed spectrum that is the flux-weighted sum of two stars.

The primary's parameters have the reference's names.  The secondary's are ``Teff_sec``, ``log(g)_sec``, ``[Fe/H]_sec``,
``[a/Fe]_sec``, ``Vmic_sec``, ``Vrad_sec`` and ``Vrot_sec``; one that is neither sampled nor fixed is the primary's.
``Rratio`` = R_sec / R_pri weights the secondary's blackbody flux.  ``Inst_R`` and the continuum polynomial are shared
(``Engine(binary=True)``, include/payne_b200.h ``PayneBinary``).
"""
from __future__ import annotations

from ..engine import Engine
from .likelihood import _genmod, _Likelihood, free_parameters


class BinaryLikelihood(_Likelihood):
    def __init__(self, fitargs, fitpars, runbools, **kwargs):
        self.fitargs = fitargs
        if not runbools[0]:
            raise ValueError('BinaryLikelihood needs a spectrum')
        if runbools[1]:
            raise NotImplementedError('binaries with photometry: the SED of two stars is not modelled')
        self.precision = kwargs.get('precision', 'parity')
        (self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool, self.carbon_bool), self.GM = \
            _genmod(fitargs, runbools, self.precision)
        super().__init__(free_parameters(fitpars), fitargs['fixedpars'])
        self.engine = Engine(spec=self.GM.PP.anns.model, obs_wave=fitargs['obs_wave_fit'],
                             obs_flux=fitargs['obs_flux_fit'], obs_eflux=fitargs['obs_eflux_fit'],
                             fitpars_i=self.fitpars_i, fixedpars=self.fixedpars,
                             runbools=[True, False, self.modpoly_bool, False, False], precision=self.precision,
                             device=kwargs.get('device'), binary=True)

    def _lnlike(self, theta):
        return self.engine.lnlike_batch_binary(theta)
