"""``BinaryLikelihood``: a double-lined binary (SB2), one observed spectrum that is the flux-weighted sum of two stars,
with the ``likelihood`` interface (``lnlikefn``, ``lnlike_batch``, ``parsdict``, ``fitpars_i``, ``ndim``, ``fixedpars``).

The primary's parameters have the reference's names.  The secondary's are ``Teff_sec``, ``log(g)_sec``, ``[Fe/H]_sec``,
``[a/Fe]_sec``, ``Vmic_sec``, ``Vrad_sec`` and ``Vrot_sec``; one that is neither sampled nor fixed is the primary's.
``Rratio`` = R_sec / R_pri weights the secondary's blackbody flux.  ``Inst_R`` and the continuum polynomial are shared
(``Engine(binary=True)``, include/payne_b200.h ``PayneBinary``).
"""
from __future__ import annotations

import numpy as np

from ..engine import Engine
from .genmod import GenMod
from .likelihood import free_parameters


class BinaryLikelihood(object):
    def __init__(self, fitargs, fitpars, runbools, **kwargs):
        self.fitargs = fitargs
        self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool, self.carbon_bool = runbools[:5]
        if not self.spec_bool:
            raise ValueError('BinaryLikelihood needs a spectrum')
        if self.phot_bool:
            raise NotImplementedError('binaries with photometry: the SED of two stars is not modelled')
        if self.carbon_bool:
            raise NotImplementedError('carbon_bool is hard-wired off in the reference (fitstar.py:150-154)')
        self.fixedpars = fitargs['fixedpars']
        self.precision = kwargs.get('precision', 'parity')
        self.GM = GenMod(precision=self.precision)
        self.GM._initspecnn(nnpath=fitargs['specANNpath'], NNtype=fitargs.get('NNtype', 'LinNet'))
        self.fitpars_i = free_parameters(fitpars)
        self.ndim = len(self.fitpars_i)
        self.parsdict = {}
        self.engine = Engine(spec=self.GM.PP.anns.model, obs_wave=fitargs['obs_wave_fit'],
                             obs_flux=fitargs['obs_flux_fit'], obs_eflux=fitargs['obs_eflux_fit'],
                             fitpars_i=self.fitpars_i, fixedpars=self.fixedpars,
                             runbools=[True, False, self.modpoly_bool, False, False], precision=self.precision,
                             device=kwargs.get('device'), binary=True)

    def _set_parsdict(self, pars):
        self.parsdict = {pp: vv for pp, vv in zip(self.fitpars_i, pars)}
        for kk in self.fixedpars.keys():
            self.parsdict[kk] = self.fixedpars[kk]

    def lnlikefn(self, pars):
        """One parameter vector -> float."""
        self._set_parsdict(pars)
        th = np.asarray(pars, dtype=np.float64).reshape(1, self.ndim)
        return float(self.engine.lnlike_batch_binary(th)[0])

    def lnlike_batch(self, theta):
        """theta [B, ndim] (CUDA float64 tensor, or numpy) -> lnL [B] of the same kind."""
        out = self.engine.lnlike_batch_binary(theta)
        last = theta[-1]
        self._set_parsdict([float(v) for v in (last.tolist() if hasattr(last, 'tolist') else last)])
        return out
