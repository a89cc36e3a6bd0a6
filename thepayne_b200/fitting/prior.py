"""Prior transform / ln-prior with the reference's ``prior`` interface plus batched forms.

Mirror of ``Payne/fitting/prior.py``: constructor ``prior(fitargs, inpriordict, fitpars, runbools)``
(:6-124), ``priortrans(upars)`` (:126-142; unit cube -> parameters: pv_uniform / pv_gaussian /
pv_tgaussian / pv_exp / pv_texp, reference defaults otherwise, ``pc_0`` in [0.75, 1.25] and
``pc_k`` within +-5 sigma of ``blaze_coeff``, :187-197) and ``lnpriorfn(pars)`` (:274-377; additive
'gaussian' / 'uniform' priors of :379-465, incl. the derived ``Parallax = 1000/Dist``).

``priortrans_batch(U[B, ndim])`` and ``lnprior_batch(theta[B, ndim])`` do the same for a whole
proposal queue (scipy's ppf functions are vectorised), so the sampler side keeps up with
``likelihood.lnlike_batch``.  The brutus-derived IMF / Galactic / Vrot / Vtot priors
(``advancedpriors.py``, astropy-based) are outside the accelerated path and raise.

Several spectra (``FitPayne`` with a list-valued ``spec``): ``Inst_R_<s>`` takes the priors and default range of
``Inst_R``, and ``pc_<s>_<k>`` those of ``pc_k`` with ``blaze_coeff_<s>`` in place of ``blaze_coeff``.

Binaries (``FitPayne`` with ``'binary': True``): ``<name>_sec`` takes the default range of ``<name>`` (``Vmic_sec``: none,
like ``Vmic``), and ``Rratio`` defaults to uniform [0, 1].
"""
from __future__ import annotations

import re

import numpy as np
from scipy.stats import expon, norm, truncexpon, truncnorm

_SPEC = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Inst_R', 'CarbonScale']
_BINARY = [p + '_sec' for p in _SPEC[:6]] + ['Vmic_sec', 'Rratio']
_ISO = ['log(A)', 'log(R)', 'Av', 'Rv', 'Dist']
_SPECTRUM = re.compile(r'(Inst_R|pc)_(\d+)(?:_(\d+))?$')     # Inst_R_<s>, pc_<s>_<k>
_PV = {'pv_uniform': 'uniform', 'pv_gaussian': 'gaussian', 'pv_tgaussian': 'tgaussian', 'pv_exp': 'exp',
       'pv_texp': 'texp'}


class prior(object):
    def __init__(self, fitargs, inpriordict, fitpars, runbools):
        self.fitargs = fitargs
        self.fixedpars = self.fitargs['fixedpars']
        self.fitpars_i = [pp for pp in fitpars[0] if fitpars[1][pp]]
        self.ndim = len(self.fitpars_i)
        self.priordict = {k: {} for k in ['uniform', 'gaussian', 'tgaussian', 'exp', 'texp']}
        self.additionalpriors = {}
        self.polycoefarr = None
        self.spectrum_polycoef = {}                            # s -> blaze_coeff_<s>
        for kk in inpriordict.keys():
            if kk == 'blaze_coeff':
                self.polycoefarr = inpriordict['blaze_coeff']
            elif kk.startswith('blaze_coeff_'):
                self.spectrum_polycoef[int(kk[len('blaze_coeff_'):])] = inpriordict[kk]
            elif kk in ('IMF', 'GAL', 'VROT', 'VTOT', 'AngDia'):
                raise NotImplementedError('%s prior (advancedpriors.py) is outside the accelerated path' % kk)
            else:
                for ii in inpriordict[kk].keys():
                    if ii in _PV:
                        self.priordict[_PV[ii]][kk] = inpriordict[kk][ii]
                    elif ii == 'pv_loguniform':
                        raise NotImplementedError('pv_loguniform is broken in the reference (prior.py:266)')
                    elif ii != 'fixed':
                        self.additionalpriors.setdefault(kk, {})[ii] = inpriordict[kk][ii]
        self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool = runbools[:4]
        self.defaultpars = {                                   # prior.py:100-113
            'Teff': [3000.0, 17000.0], 'log(g)': [-1.0, 5.5], '[Fe/H]': [-4.0, 0.5], '[a/Fe]': [-0.2, 0.6],
            'Vrad': [-700.0, 700.0], 'Vrot': [0, 300.0], 'Inst_R': [10000.0, 60000.0], 'log(A)': [-3.0, 7.0],
            'log(R)': [-2.0, 3.0], 'Dist': [0.0, 100000.0], 'Av': [0.0, 5.0], 'Rv': [2.0, 5.0],
            'CarbonScale': [0.0, 2.0], 'Rratio': [0.0, 1.0]}
        self.defaultpars.update({p + '_sec': self.defaultpars[p] for p in _SPEC[:6]})

    # ------------------------------------------------------------------ unit cube -> parameters
    @staticmethod
    def pc_box(k, polycoefarr):
        """(lo, hi) of continuum coefficient k (prior.py:187-197): [0.75, 1.25] for k = 0, blaze_coeff[k]'s mean +- 5
        sigma otherwise.  The uniform prior of a sampled ``pc_k`` and the box of a marginalised one."""
        if k == 0:
            return 0.75, 1.25
        return polycoefarr[k][0] - 5.0 * polycoefarr[k][1], polycoefarr[k][0] + 5.0 * polycoefarr[k][1]

    def _transform(self, name, u, iso):
        """One named parameter, scalar or array ``u`` (prior.py:150-176 / :226-268)."""
        pd = self.priordict
        if name in pd['uniform']:
            lo, hi = min(pd['uniform'][name]), max(pd['uniform'][name])
            return (hi - lo) * u + lo
        if name in pd['gaussian']:
            return norm.ppf(u, loc=pd['gaussian'][name][0], scale=pd['gaussian'][name][1])
        if name in pd['tgaussian']:
            lo, hi, mu, sig = pd['tgaussian'][name]
            a, b = (lo - mu) / sig, (hi - mu) / sig
            x = truncnorm.ppf(u, a, b, loc=mu, scale=sig)
            return np.where(x == np.inf, hi, x) if np.ndim(x) else (hi if x == np.inf else x)
        if name in pd['exp']:
            return expon.ppf(u, loc=pd['exp'][name][0], scale=pd['exp'][name][1])
        if name in pd['texp']:
            if iso:
                raise NotImplementedError('pv_texp for photometric parameters has an inconsistent '
                                          'signature in the reference (prior.py:257-262)')
            lo, hi, sc = pd['texp'][name]
            x = truncexpon.ppf(u, (hi - lo) / sc, loc=lo, scale=sc)
            return np.where(x == np.inf, hi, x) if np.ndim(x) else (hi if x == np.inf else x)
        lo, hi = self.defaultpars['Inst_R' if _SPECTRUM.match(name) else name]
        return (hi - lo) * u + lo

    def _column(self, name, u):
        m = _SPECTRUM.match(name)
        if m and self.spec_bool:                               # Inst_R_<s>, pc_<s>_<k>
            if m.group(1) == 'Inst_R' and m.group(3) is None:
                return self._transform(name, u, iso=False)
            if m.group(1) == 'pc' and m.group(3) is not None:
                pcmin, pcmax = self.pc_box(int(m.group(3)), self.spectrum_polycoef[int(m.group(2))])
                return (pcmax - pcmin) * u + pcmin
        if 'pc' in name:
            if not self.spec_bool:
                raise KeyError(name)
            pcmin, pcmax = self.pc_box(int(name.split('_')[-1]), self.polycoefarr)
            return (pcmax - pcmin) * u + pcmin
        if self.spec_bool and (name in _SPEC or name in _BINARY):
            return self._transform(name, u, iso=False)
        if self.phot_bool and (name in _ISO or (not self.spec_bool and name in _SPEC[:4])):
            return self._transform(name, u, iso=name in _ISO)
        raise KeyError('no prior transform for %s' % name)     # reference: KeyError on outputPT[pp]

    def priortrans(self, upars):
        return [self._column(pp, uu) for pp, uu in zip(self.fitpars_i, upars)]

    def priortrans_batch(self, U):
        U = np.asarray(U, dtype=np.float64)
        return np.stack([np.asarray(self._column(pp, U[:, i]), dtype=np.float64)
                         for i, pp in enumerate(self.fitpars_i)], axis=1)

    # ------------------------------------------------------------------ additive ln-priors
    def _lnprior_cols(self, get, n):
        """``get(name)`` -> value(s); returns ln-prior (scalar or [n]) per prior.py:379-465."""
        out = np.zeros(n) if n else 0.0
        if len(self.additionalpriors) == 0:
            return out
        groups = []
        if self.spec_bool:
            groups.append(_SPEC + _BINARY + [p for p in self.fitpars_i if p.startswith('Inst_R_')])
        if self.phot_bool:
            g = [] if self.spec_bool else ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]']
            g += [p for p in ['log(R)', 'Dist', 'log(A)', 'Av'] if p in self.fitpars_i]
            if 'Dist' in self.fitpars_i:
                g.append('Parallax')
            groups.append(g)
        for names in groups:
            for kk, pri in self.additionalpriors.items():
                if kk not in names:
                    continue
                v = 1000.0 / get('Dist') if kk == 'Parallax' else get(kk)
                if 'gaussian' in pri:
                    out = out + -0.5 * (((v - pri['gaussian'][0]) ** 2.0) / (pri['gaussian'][1] ** 2.0))
                if 'uniform' in pri:
                    bad = (v < pri['uniform'][0]) | (v > pri['uniform'][1])
                    out = np.where(bad, -np.inf, out) if n else (-np.inf if bad else out)
                if 'beta' in pri or 'log-normal' in pri:
                    raise IOError('Beta / Log-Normal priors are not implemented in the reference either')
        return out

    def lnpriorfn(self, pars):
        parsdict = {pp: vv for pp, vv in zip(self.fitpars_i, pars)} if isinstance(pars, list) else pars
        for kk in self.fixedpars.keys():
            parsdict[kk] = self.fixedpars[kk]
        return float(self._lnprior_cols(lambda k: parsdict[k], 0))

    def lnprior_batch(self, theta):
        theta = np.asarray(theta, dtype=np.float64)
        ix = {p: i for i, p in enumerate(self.fitpars_i)}

        def get(k):
            return theta[:, ix[k]] if k in ix else np.full(theta.shape[0], float(self.fixedpars[k]))
        return np.asarray(self._lnprior_cols(get, theta.shape[0]), dtype=np.float64)
