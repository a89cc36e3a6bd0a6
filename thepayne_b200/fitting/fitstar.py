"""``FitPayne`` with the reference's input dictionary and output file, driving the lock-step batched
nested sampler instead of dynesty (SURVEY.md §8f-1).

Mirror of ``Payne/fitting/fitstar.py``: ``run(inputdict=...)`` (:19-217) turns the user dictionary
(``spec`` / ``phot`` / ``priordict`` / ``sampler`` / ``output`` / ``specANNpath`` / ``photANNpath`` /
``NNtype`` / ``photscale``) into ``fitargs``, the ordered parameter list with its on/off switches and
the run booleans; ``run_dynesty`` (:236-258) builds the prior and likelihood objects;
``_runsampler`` (:260-463) samples and writes one line per dead point -- iteration, the parameters,
``log(lk) log(vol) log(wt) h nc log(z) delta(log(z))`` -- then the final live points.

What differs, on purpose:
  * the sampler is ``nested.BatchedNestedSampler``: every likelihood evaluation is part of one
    ``likelihood.lnlike_batch`` call of ``queue_size`` (default ``npoints``) proposals.  The sampler keys
    of the reference keep their meaning (``npoints``, ``walks``, ``delta_logz_final``, ``flushnum``,
    ``maxiter``, ``maxcall``, ``reflective``); ``samplemethod`` must be 'rwalk' (the demo's choice,
    demo/runPayne.py:112), ``samplerbounds`` is a single ellipsoid, ``samplertype`` 'Static';
  * the parameters written for a dead point are that point's own (the reference writes
    ``likeobj.parsdict``, i.e. whatever vector the likelihood saw last, fitstar.py:347);
  * ``inputdict['precision']`` / ``['device']`` select the CUDA precision mode and device;
  * ``inputdict['spec']`` may be a list of spectrum dictionaries (echelle orders, spectrograph arms), each with the
    keys of the single one.  The labels, ``Vrad`` and ``Vrot`` are shared; spectrum s has its own ``Inst_R_<s>`` and
    continuum coefficients ``pc_<s>_<k>``, whose priors come from ``priordict['Inst_R_<s>']`` and
    ``priordict['blaze_coeff_<s>']`` (``multispec.MultiSpecLikelihood``).  ``priordict['Inst_R_<s>'] = {'fixed': lsf}``
    with a 1-D ``lsf`` (one dispersion per fitted pixel of spectrum s, for every s) fits with LSF vectors; the output
    file then has no column for them;
  * ``inputdict['binary'] = True`` with a single ``spec`` fits a double-lined binary (``binary.BinaryLikelihood``): the
    secondary's ``Teff_sec``, ``log(g)_sec``, ``Vrad_sec`` and ``Vrot_sec`` and the radius ratio ``Rratio`` follow the
    reference parameters (before ``pc_k``); ``[Fe/H]_sec``, ``[a/Fe]_sec`` and ``Vmic_sec`` get a column only when
    ``priordict`` names them, and are the primary's otherwise.  ``{'fixed': v}`` fixes any of them;
  * ``spec['modpoly_marginal'] = True`` (beside ``modpoly``; with a list-valued ``spec`` in every spectrum or in none)
    integrates the continuum coefficients out per likelihood call instead of sampling them (``Engine.set_cont_marg``):
    the sampler has K fewer dimensions per spectrum, and the coefficients' flat prior boxes are the ones a sampled
    ``pc_k`` would get (``prior.pc_box``).  The output file keeps its ``pc`` columns: every written row holds a draw
    c-hat + L^-T z, z ~ N(0, I), of the coefficients' conditional posterior at that row's parameters, seeded from the
    sampler seed.
"""
from __future__ import annotations

import sys
from datetime import datetime

import numpy as np

from .batching import BatchedLnProb
from .fitutils import airtovacuum
from .nested import BatchedNestedSampler

_ALLPARS = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Vmic', 'Inst_R', 'log(R)', 'Dist', 'log(A)',
            'Av', 'Rv', 'CarbonScale']
# a binary's own parameters in sampler order; those outside _BINARY_ON only when priordict names them
_BINARY = ['Teff_sec', 'log(g)_sec', '[Fe/H]_sec', '[a/Fe]_sec', 'Vrad_sec', 'Vrot_sec', 'Vmic_sec', 'Rratio']
_BINARY_ON = ['Teff_sec', 'log(g)_sec', 'Vrad_sec', 'Vrot_sec', 'Rratio']


def _fitted(sp, sel):
    """A spectrum dictionary's fitted observation: wave, flux and eflux at ``sel`` as float64, the wavelengths in
    vacuum unless ``convertair`` is False."""
    fit = {'obs_%s_fit' % k: np.asarray(sp['obs_' + k], dtype=np.float64)[sel] for k in ['wave', 'flux', 'eflux']}
    if sp.get('convertair', True):
        fit['obs_wave_fit'] = airtovacuum(fit['obs_wave_fit'])
    return fit


class FitPayne(object):
    def __init__(self, **kwargs):
        from .likelihood import likelihood
        from .prior import prior
        self.prior = prior
        self.likelihood = likelihood

    # ------------------------------------------------------------------ input dictionary -> fit setup
    def run(self, *args, **kwargs):
        return self(self._setup(*args, **kwargs))

    def _setup(self, *args, **kwargs):
        """The user dictionary -> ``indicts`` (fitargs, fitpars, sampler, priordict, runbools)."""
        self.verbose = kwargs.get('verbose', True)
        if 'inputdict' not in kwargs:
            print('NO USER DEFINED INPUT DICT, NOTHING TO FIT!')
            raise IOError
        inputdict = kwargs['inputdict']
        self.priordict = inputdict.get('priordict', {})
        self.output = inputdict.get('output', 'Test.dat')
        self.samplerdict = inputdict.get('sampler', {})
        self.precision = inputdict.get('precision', 'parity')
        self.device = inputdict.get('device', None)
        fa = self.fitargs = {}
        self.spec_bool = self.phot_bool = self.modpoly_bool = self.photscale_bool = self.carbon_bool = False
        self.fitpars = list(_ALLPARS)
        self.fitpars_bool = {pp: False for pp in self.fitpars}

        self.binary_bool = bool(inputdict.get('binary', False))
        if self.binary_bool and isinstance(inputdict.get('spec'), (list, tuple)):
            raise NotImplementedError('binary with several spectra (a list-valued spec)')
        if self.binary_bool and 'phot' in inputdict:
            raise NotImplementedError('binary with photometry: the SED of two stars is not modelled')
        if 'spec' in inputdict:                                            # fitstar.py:70-154
            self.spec_bool = True
            fa['specANNpath'] = inputdict.get('specANNpath', None)
            fa['NNtype'] = inputdict.get('NNtype', 'LinNet')
            for pp in ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Inst_R'] + \
                    (['Vmic'] if fa['NNtype'] == 'YST2' else []):
                self.fitpars_bool[pp] = True
        if isinstance(inputdict.get('spec'), (list, tuple)):
            self._setup_spectra(inputdict)
        elif 'spec' in inputdict:
            sp = inputdict['spec']
            fa['obs_wave'], fa['obs_flux'], fa['obs_eflux'] = sp['obs_wave'], sp['obs_flux'], sp['obs_eflux']
            sel = slice(None)
            if 'wave_minmax' in sp:                    # the wavelengths as given: float32 ones compare in float32
                fa['wave_minmax'] = sp['wave_minmax']
                sel = (np.asarray(fa['obs_wave']) >= sp['wave_minmax'][0]) & (np.asarray(fa['obs_wave']) <= sp['wave_minmax'][1])
            fa.update(_fitted(sp, sel))
            coef, box = self._setup_continuum(sp, 'blaze_coeff', 'pc_{}')
            if coef is not None:
                self.polycoefarr, self.polyorder = coef, len(coef)
                fa['norm_polyorder'] = self.polyorder
                if box is not None:
                    fa['cont_box'] = box

        if 'phot' in inputdict:                                            # fitstar.py:157-190
            self.phot_bool = True
            fa['photANNpath'] = inputdict.get('photANNpath', None)
            for pp in ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Av']:
                self.fitpars_bool[pp] = True
            fa['obs_phot'] = {kk: inputdict['phot'][kk] for kk in inputdict['phot'].keys()}
            self.photscale_bool = inputdict.get('photscale', False)
            if self.photscale_bool:
                self.fitpars_bool['log(A)'] = True
            else:
                self.fitpars_bool['log(R)'] = True
                self.fitpars_bool['Dist'] = True
            if inputdict.get('Rvfree', False):
                raise NotImplementedError('Rvfree: the likelihood never forwards Rv (likelihood.py:103-106)')

        if self.binary_bool:
            if not self.spec_bool:
                raise ValueError("binary needs inputdict['spec']")
            names = [pp for pp in _BINARY if pp in _BINARY_ON or pp in self.priordict]
            at = next((i for i, pp in enumerate(self.fitpars) if pp.startswith('pc_')), len(self.fitpars))
            self.fitpars[at:at] = names
            for pp in names:
                self.fitpars_bool[pp] = True
            fa['binary'] = True

        fa['fixedpars'] = {}                                               # fitstar.py:193-198
        for kk in self.priordict.keys():
            if isinstance(self.priordict[kk], dict) and 'fixed' in self.priordict[kk]:
                fa['fixedpars'][kk] = self.priordict[kk]['fixed']
                self.fitpars_bool[kk] = False
        return {'fitargs': fa, 'fitpars': [self.fitpars, self.fitpars_bool], 'sampler': self.samplerdict,
                'priordict': self.priordict,
                'runbools': [self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool, self.carbon_bool]}

    def _setup_spectra(self, inputdict):
        """A list-valued ``spec``: every spectrum's observation as the single one's (wave_minmax, convertair), and
        ``Inst_R_<s>`` in place of ``Inst_R`` and ``pc_<s>_<k>`` per spectrum."""
        specs = list(inputdict['spec'])
        if not specs:
            raise ValueError("inputdict['spec'] is an empty list")
        if any('Vrad' in sp for sp in specs) or any(k.startswith('Vrad_') for k in self.priordict):
            raise NotImplementedError('a Vrad per spectrum: FitPayne fits one Vrad shared by every spectrum')
        fa = self.fitargs
        fa['spectra'] = []
        for sp in specs:
            w = np.asarray(sp['obs_wave'], dtype=np.float64)
            sel = slice(None)
            if 'wave_minmax' in sp:
                sel = (w >= sp['wave_minmax'][0]) & (w <= sp['wave_minmax'][1])
            fa['spectra'].append(_fitted(sp, sel))
        self.fitpars.remove('Inst_R')
        self.fitpars_bool.pop('Inst_R')
        for s in range(len(specs)):
            self.fitpars.append('Inst_R_%d' % s)
            self.fitpars_bool['Inst_R_%d' % s] = True
        if len({bool(sp.get('modpoly', False)) for sp in specs}) > 1:
            raise ValueError('every spectrum has a continuum polynomial (modpoly) or none does')
        if len({bool(sp.get('modpoly_marginal', False)) for sp in specs}) > 1:
            raise ValueError('every spectrum sets modpoly_marginal or none does')
        for s, sp in enumerate(specs):                                     # as fitstar.py:110-147 per spectrum
            box = self._setup_continuum(sp, 'blaze_coeff_%d' % s, 'pc_%d_{}' % s)[1]
            if box is not None:
                fa['spectra'][s]['cont_box'] = box

    def _setup_continuum(self, sp, key, name):
        """The continuum polynomial of a spectrum dictionary with ``modpoly`` (fitstar.py:110-147): the prior
        ``priordict[key]`` of its coefficients (default: ``polyorder`` + 1 of width ``polysigma``, else three of width
        1), named ``name.format(k)``.  Sampled, they join the free parameters; with ``modpoly_marginal`` they join
        ``cont_names`` and get the boxes of a sampled ``pc_k``.  Returns the prior and the boxes (None when sampled);
        (None, None) without ``modpoly``."""
        if sp.get('modpoly_marginal', False) and not sp.get('modpoly', False):
            raise ValueError("spec['modpoly_marginal'] needs spec['modpoly']")
        if not sp.get('modpoly', False):
            return None, None
        self.modpoly_bool = True
        if key not in self.priordict:
            if 'polyorder' in sp:
                self.priordict[key] = [[0.0, sp.get('polysigma', 1.0)] for _ in range(sp['polyorder'] + 1)]
            else:
                self.priordict[key] = [[0.0, 1.0] for _ in range(3)]
        coef = self.priordict[key]
        names = [name.format(k) for k in range(len(coef))]
        if not sp.get('modpoly_marginal', False):
            for pp in names:
                self.fitpars.append(pp)
                self.fitpars_bool[pp] = True
            return coef, None
        self.fitargs.setdefault('cont_names', []).extend(names)
        return coef, [self.prior.pc_box(k, coef) for k in range(len(coef))]

    def __call__(self, indicts):
        return self.run_dynesty(indicts)

    def run_dynesty(self, indicts):
        """Name kept from the reference (fitstar.py:236-258); the sampler is the batched one."""
        fitargs, fitpars, runbools = indicts['fitargs'], indicts['fitpars'], indicts['runbools']
        self._prepare(indicts)
        like = self.likelihood
        if 'spectra' in fitargs:
            from .multispec import MultiSpecLikelihood as like
        elif fitargs.get('binary', False):
            from .binary import BinaryLikelihood as like
        self.likeobj = like(fitargs, fitpars, runbools, verbose=False, precision=getattr(self, 'precision', 'parity'),
                            device=getattr(self, 'device', None))
        self._check_sampler(indicts)
        return self._runsampler(indicts['sampler'])

    def _prepare(self, indicts):
        """Dimension and prior object of the fit (everything but the likelihood)."""
        fitpars = indicts['fitpars']
        self.ndim = sum(1 for pp in fitpars[0] if fitpars[1][pp])
        self.priorobj = self.prior(indicts['fitargs'], indicts['priordict'], fitpars, indicts['runbools'])

    @staticmethod
    def _check_sampler(indicts):
        kind = indicts['sampler'].get('samplertype', 'Static')
        if kind != 'Static':
            raise NotImplementedError("samplertype %r: only the static sampler is batched" % kind)

    # ------------------------------------------------------------------ output file (fitstar.py:219-227)
    def _initoutput(self, parnames):
        self.outff = open(self.output, 'w')
        self.outff.write('Iter ')
        for pp in parnames:
            self.outff.write('{} '.format(pp))
        self.outff.write('log(lk) log(vol) log(wt) h nc log(z) delta(log(z))')
        self.outff.write('\n')

    def _writerow(self, it, vstar, parnames, tail, cont=None):
        pd = {pp: vv for pp, vv in zip(self.likeobj.fitpars_i, vstar)}
        if cont is not None:
            pd.update(zip(self.fitargs['cont_names'], cont))
        pd.update(self.likeobj.fixedpars)
        self.outff.write('{0} '.format(it))
        self.outff.write(' '.join([str(pd[q]) for q in parnames]))
        self.outff.write(' {0} {1} {2} {3} {4} {5} {6} '.format(*tail))
        self.outff.write('\n')

    def _cont_boxes(self):
        """The boxes of the marginalised coefficients in ``cont_names`` order, and every spectrum's count."""
        fa = self.fitargs
        per = [sp['cont_box'] for sp in fa['spectra']] if 'spectra' in fa else [fa['cont_box']]
        return [b for p in per for b in p], [len(p) for p in per]

    def _cont_draws(self, V):
        """A draw c-hat + L^-T z, z ~ N(0, I), of the marginalised coefficients at every row of V (one batched call);
        counts the rows whose c-hat leaves its box."""
        coef, chol = self.likeobj.cont_batch(V)
        boxes, orders = self._cont_boxes()
        lo, hi = np.array([b[0] for b in boxes]), np.array([b[1] for b in boxes])
        self._cont_outside += int(np.sum(np.any((coef[:, :len(boxes)] < lo) | (coef[:, :len(boxes)] > hi), axis=1)))
        out = np.empty((len(V), len(boxes)))
        c0 = l0 = 0
        for K in orders:
            L = np.zeros((len(V), K, K))
            i, j = np.tril_indices(K)
            L[:, i, j] = chol[:, l0:l0 + K * (K + 1) // 2]
            z = self._cont_rng.standard_normal((len(V), K, 1))
            out[:, c0:c0 + K] = coef[:, c0:c0 + K] + np.linalg.solve(np.transpose(L, (0, 2, 1)), z)[..., 0]
            c0 += K
            l0 += K * (K + 1) // 2
        return out

    def _runsampler(self, samplerdict):
        npoints = samplerdict.get('npoints', 200)
        samplemethod = samplerdict.get('samplemethod', 'rwalk')
        if samplemethod != 'rwalk':
            raise NotImplementedError("samplemethod %r: the batched sampler implements 'rwalk'" % samplemethod)
        delta_logz_final = samplerdict.get('delta_logz_final', 0.01)
        flushnum = samplerdict.get('flushnum', 10)
        numwalks = samplerdict.get('walks', 25)
        maxiter = samplerdict.get('maxiter', sys.maxsize)
        maxcall = samplerdict.get('maxcall', sys.maxsize)
        reflective = [ii for ii, par in enumerate(self.likeobj.fitpars_i) if par in samplerdict.get('reflective', [])]
        starttime = datetime.now()
        if self.verbose:
            print('Batched static nested sampler w/ rwalk, {0} walks, {1} live points, queue of {2}, Ndim = {3}, '
                  'dlog(z) = {4}: {5}'.format(numwalks, npoints, samplerdict.get('queue_size', npoints), self.ndim,
                                              delta_logz_final, starttime))
        lnprob = BatchedLnProb(self.likeobj, self.priorobj)
        sampler = BatchedNestedSampler(lnprob.batch, self.priorobj.priortrans_batch, self.ndim, nlive=npoints,
                                       walks=numwalks, queue_size=samplerdict.get('queue_size', None),
                                       reflective=reflective, seed=samplerdict.get('seed', None))
        # several spectra: an LSF vector (one value per pixel, the same in every row) gets no column
        multi = 'spectra' in self.fitargs
        cont_names = self.fitargs.get('cont_names')
        parnames = list(self.likeobj.fitpars_i) + list(cont_names or []) + \
            [kk for kk, vv in self.likeobj.fixedpars.items() if not (multi and np.ndim(vv) > 0)]
        self._initoutput(parnames)
        # marginalised continuum: rows wait for one batched call per flush that draws their coefficients
        pending = []
        self._cont_rng = np.random.default_rng(samplerdict.get('seed', None))
        self._cont_outside = 0

        def write(it, vstar, tail):
            if cont_names is None:
                self._writerow(it, vstar, parnames, tail)
            else:
                pending.append((it, vstar, tail))

        def flush():
            if pending:
                draws = self._cont_draws(np.array([r[1] for r in pending], dtype=np.float64))
                for (it, vstar, tail), c in zip(pending, draws):
                    self._writerow(it, vstar, parnames, tail, c)
                del pending[:]
            self.outff.flush()

        ncall, nit = 0, 0
        for it, res in enumerate(sampler.sample(dlogz=delta_logz_final, maxiter=maxiter, maxcall=maxcall)):
            (worst, ustar, vstar, loglstar, logvol, logwt, logz, logzvar, h, nc, worst_it, propidx, propiter, eff,
             delta_logz) = res
            write(it, vstar, (loglstar, logvol, logwt, h, nc, logz, delta_logz))
            ncall += nc
            nit = it
            if (it % flushnum) == 0 or it == maxiter:
                flush()
                if self.verbose and (it % (50 * flushnum)) == 0:
                    logzerr = np.sqrt(logzvar) if logzvar > 0.0 else np.nan
                    sys.stdout.write('iter: {0:d} | nc: {1:d} | ncall: {2:d} | eff(%): {3:6.3f} | logz: {4:6.3f} +/- '
                                     '{5:6.3f} | loglk: {6:6.3f} | dlogz: {7:6.3f} > {8:6.3f}\n'.format(
                                         nit, nc, sampler.ncall, eff, logz, logzerr, loglstar, delta_logz,
                                         delta_logz_final))
                    sys.stdout.flush()
            if it == maxiter:
                break
        for it2, res in enumerate(sampler.add_live_points()):
            (worst, ustar, vstar, loglstar, logvol, logwt, logz, logzvar, h, nc, worst_it, boundidx, bounditer, eff,
             delta_logz) = res
            write(nit + it2, vstar, (loglstar, logvol, logwt, h, nc, logz, delta_logz))
        flush()
        self.outff.close()
        if self.verbose and cont_names is not None:
            print('{0} written rows have a best-fitting continuum coefficient outside its box'.format(
                self._cont_outside))
        if self.verbose:
            print('RUN TIME: {0}  ({1} likelihood evaluations in {2} batched calls)'.format(
                datetime.now() - starttime, sampler.ncall, len(sampler.batch_sizes)))
        self.likeobj._set_parsdict([float(v) for v in vstar])
        return sampler
