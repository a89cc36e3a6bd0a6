"""Model generation with the reference's ``GenMod`` interface (Payne/fitting/genmod.py)."""
from __future__ import annotations

import numpy as np

from ..predict.predictsed import FastPayneSEDPredict
from ..predict.predictspec import PayneSpecPredict


class GenMod(object):
    def __init__(self, *arg, **kwargs):
        self.verbose = kwargs.get('verbose', False)
        self.precision = kwargs.get('precision', 'parity')

    def _initspecnn(self, nnpath=None, **kwargs):          # genmod.py:15-32
        # the reference's own default here is 'YST1', but fitstar always passes NNtype and defaults
        # it to 'LinNet' (fitstar.py:81); an in-memory network brings its own type
        NNtype = kwargs.get('NNtype', getattr(nnpath, 'nntype', 'LinNet'))
        if NNtype == 'YST1':                                # genmod.py:20-21
            from ..predict.ystpred import PayneSpecPredict as YstPredict
            self.PP = YstPredict(nnpath=nnpath, NNtype=NNtype, precision=self.precision)
        else:
            self.PP = PayneSpecPredict(nnpath=nnpath, NNtype=NNtype, precision=self.precision)

    def _initphotnn(self, filterarray, nnpath=None):       # genmod.py:35-43
        self.filterarray = None if filterarray is None else list(filterarray)
        self.fppsed = FastPayneSEDPredict(usebands=self.filterarray, nnpath=nnpath, precision=self.precision)
        if self.filterarray is None:
            self.filterarray = self.fppsed.filternames

    def genspec(self, pars, outwave=None, verbose=False, modpoly=False, carbon_bool=False):
        """genmod.py:58-108: pars = [Teff, logg, FeH, aFe, Vrad, Vrot, Vmic, Inst_R, pc_0...].  An Inst_R that is a
        1-D array is the LSF vector on ``outwave`` (genmod.py:82-85 -> predictspec.py:265-286)."""
        if carbon_bool:
            raise NotImplementedError('carbon_bool is hard-wired off in the reference (fitstar.py:150-154)')
        pars = list(pars)
        lsf = None
        if np.ndim(pars[7]) == 1:
            if outwave is None:
                raise ValueError('an LSF vector Inst_R gives the dispersion at the pixels of outwave: give outwave')
            lsf = np.ascontiguousarray(pars[7], dtype=np.float64)
            pars[7] = np.nan                               # the vector replaces the scalar-R stage
        pars = [float(p) for p in pars]
        polycoef = pars[8:] if modpoly else []
        if outwave is None:
            # genmod.py:87-100 + predictspec.py:243-294: the Doppler-shifted native grid, flux not resampled
            inst = pars[7] * 2.355 if np.isfinite(pars[7]) else pars[7]
            wave, flux = self.PP.getspec(Teff=pars[0], logg=pars[1], feh=pars[2], afe=pars[3], rad_vel=pars[4],
                                         rot_vel=pars[5], vmic=pars[6], inst_R=inst, outwave=None)
            if modpoly:
                from .fitutils import polycalc
                flux = flux * polycalc(polycoef, wave)
            return wave, flux
        eng = self.PP.anns.engine_for(outwave, npoly=len(polycoef), lsf=lsf)
        row = np.array([pars[:8] + list(polycoef)], dtype=np.float64)
        flux, _, _ = eng.model_batch(row, want_mags=False)
        return outwave, flux[0].cpu().numpy()

    def genphot(self, pars, rvfree=False, verbose=False):   # genmod.py:110-155
        if rvfree:
            raise NotImplementedError('rvfree is never set by the likelihood (likelihood.py:103-106)')
        teff, logg, feh, afe, logR, dist, av = [float(p) for p in pars[:7]]
        logt = np.log10(teff)
        logl = 2.0 * logR + 4.0 * (logt - np.log10(5770.0))
        sed = self.fppsed.sed(logt=logt, logg=logg, feh=feh, afe=afe, logl=logl, dist=dist, av=av, rv=3.1)
        return {ff: s for s, ff in zip(sed, self.filterarray)}

    def genphot_scaled(self, pars, rvfree=False, verbose=False):   # genmod.py:157-187
        if rvfree:
            raise NotImplementedError('rvfree is never set by the likelihood (likelihood.py:103-106)')
        teff, logg, feh, afe, logA, av = [float(p) for p in pars[:6]]
        sed = self.fppsed.sed(logt=np.log10(teff), logg=logg, feh=feh, afe=afe, logA=logA, av=av, rv=3.1)
        return {ff: s for s, ff in zip(sed, self.filterarray)}
