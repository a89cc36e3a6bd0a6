"""Fitting many stars at once: one engine for all their observations, and their samplers in lock-step.

A survey fits thousands of stars with the same emulator.  Between two stars the observation changes
(wavelengths, fluxes, errors, which magnitudes and in what order), and so may the values of the fixed parameters
(an instrumental resolution or LSF vector, a catalogue distance or extinction, an asteroseismic log(g)) and, given
one ``fitpars`` per star, the parameter layout itself (which parameters are free, the continuum order, photometry
or not, ``log(A)`` or ``log(R)`` + ``Dist``); the emulator weights and every table built from the emulator grid
stay the same.  A single star's sampler hands over a few hundred points per call, which
leaves the GPU latency-bound; the points of many stars together make one full-size batch.

``StarSetLikelihood`` builds one ``Engine`` holding every star's observation.  ``star(k)`` is a view with the
interface of ``likelihood.likelihood`` for star k, so ``BatchedLnProb`` and ``BatchedNestedSampler`` work on it
unchanged.

``FitPayneMany().run(inputdicts=[...])`` is ``FitPayne.run`` for a list of input dictionaries: each star gets its
fitargs, prior, sampler and output file exactly as ``FitPayne.run`` makes them, and the samplers run in their own
threads.  Every sampler's likelihood call goes to a ``LockstepBatcher``; once every unfinished sampler has posted
its points, the batcher makes ONE ``lnlike_batch(theta, star)`` call, concatenated in star order, and hands back
the slices.  A sampler that finishes or raises leaves the barrier.  Each sampler sees exactly the values a
separate ``FitPayne`` run would give it, so its output file is the same byte for byte.
"""
from __future__ import annotations

import threading

import numpy as np

from ..engine import Engine
from .fitstar import FitPayne
from .likelihood import _genmod, _Likelihood, free_parameters


def _same(a, b):
    if a is b:
        return True
    if isinstance(a, (str, int, float)) and isinstance(b, (str, int, float)):
        return a == b
    return False


class StarSetLikelihood(object):
    """The likelihoods of several stars that share emulators.

    ``fitargs_list``: one ``fitargs`` per star (as ``FitPayne.run`` builds them).  ``fitpars`` / ``runbools``:
    one value for every star, or a list with one per star.  Each star keeps its own fixed values (a vector
    ``Inst_R`` is its LSF) and its own photometric bands: the photometry net covers the union of the bands of the
    stars that have photometry, in order of first appearance, and each star's SED chi2 is summed in its
    ``obs_phot`` order, as a separate ``likelihood`` of that star sums it.

    With one shared ``fitpars`` the stars share one layout, and the names of the fixed parameters must agree
    (they are the columns of every star's output file).  With one ``fitpars`` per star each star has its own
    layout: its free parameters, photometry, photscale, continuum order and fixed parameter names may differ;
    the emulator paths, ``NNtype``, ``spec_bool`` and ``modpoly_bool`` must agree."""

    def __init__(self, fitargs_list, fitpars, runbools, precision='parity', device=None):
        fitargs_list = list(fitargs_list)
        if not fitargs_list:
            raise ValueError('no stars')
        S = len(fitargs_list)
        per_star = _is_per_star(fitpars, S)
        fp_list = list(fitpars) if per_star else [fitpars] * S
        rb_list = list(runbools) if isinstance(runbools[0], (list, tuple)) else [runbools] * S
        if len(rb_list) != S:
            raise ValueError('runbools: one list for all stars or one per star')
        rb_list = [[bool(b) for b in rb[:5]] for rb in rb_list]
        free_list = [free_parameters(fp) for fp in fp_list]
        fa0, free0, rb0 = fitargs_list[0], free_list[0], rb_list[0]
        phot_stars = [k for k in range(S) if rb_list[k][1]]
        for k in range(1, S):
            fa = fitargs_list[k]
            if per_star:
                for i, name in ((0, 'spec_bool'), (2, 'modpoly_bool')):
                    if rb_list[k][i] != rb0[i]:
                        raise ValueError('star %d: %s differs from star 0' % (k, name))
            else:
                if rb_list[k] != rb0:
                    raise ValueError('star %d: runbools differ from star 0' % k)
                if free_list[k] != free0:
                    raise ValueError('star %d: free parameters differ from star 0' % k)
            if not _same(fa.get('specANNpath'), fa0.get('specANNpath')):
                raise ValueError('star %d: specANNpath differs from star 0' % k)
            if fa.get('NNtype', 'LinNet') != fa0.get('NNtype', 'LinNet'):
                raise ValueError('star %d: NNtype differs from star 0' % k)
            if not per_star and set(fa.get('fixedpars', {})) != set(fa0.get('fixedpars', {})):
                raise ValueError('star %d: fixedpars names differ from star 0' % k)
        for k in phot_stars[1:]:
            if not _same(fitargs_list[k].get('photANNpath'), fitargs_list[phot_stars[0]].get('photANNpath')):
                raise ValueError('star %d: photANNpath differs from star %d' % (k, phot_stars[0]))
        self.bands = []
        for k in phot_stars:
            self.bands += [b for b in fitargs_list[k]['obs_phot'].keys() if b not in self.bands]
        # star 0's spectrum net (every star names the same), the photometry net of the first star with photometry
        nets = dict(fa0, photANNpath=fitargs_list[phot_stars[0]]['photANNpath']) if phot_stars else fa0
        (self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool, self.carbon_bool), self.GM = _genmod(
            nets, [rb0[0], bool(phot_stars), rb0[2], rb0[3], any(rb[4] for rb in rb_list)], precision, self.bands)
        self.n_stars = S
        self.fitargs_list = fitargs_list
        self.fixedpars = fa0['fixedpars']
        self.precision = precision
        stars = [{'wave': fa.get('obs_wave_fit'), 'flux': fa.get('obs_flux_fit'), 'eflux': fa.get('obs_eflux_fit'),
                  'phot': fa.get('obs_phot') if rb[1] else None,
                  'bands': list(fa['obs_phot'].keys()) if rb[1] else None,
                  'fixedpars': dict(fa.get('fixedpars', {})), 'cont_box': fa.get('cont_box')}
                 for fa, rb in zip(fitargs_list, rb_list)]
        if any(free != free0 for free in free_list) or any(rb != rb0 for rb in rb_list):
            for st, free, rb in zip(stars, free_list, rb_list):     # each star's own layout
                st['fitpars_i'], st['runbools'] = free, rb
        self.engine = Engine(spec=self.GM.PP.anns.model if self.spec_bool else None,
                             phot=self.GM.fppsed.net if self.phot_bool else None, stars=stars,
                             fitpars_i=free0, fixedpars=self.fixedpars,
                             runbools=[self.spec_bool, self.phot_bool, self.modpoly_bool, self.photscale_bool, False],
                             precision=precision, device=device)
        self.fitpars_i = free0
        self.star_fitpars_i, self.star_ndim = self.engine.star_fitpars_i, self.engine.star_ndim
        self.ndim = self.engine.ndim                      # the largest star's: the width of a batch row
        self.ncalls = 0                                   # lnlike_batch calls made on the engine
        self._lock = threading.Lock()                     # the samplers' threads share the engine

    def lnlike_batch(self, theta, star):
        """theta [B, ndim] and star [B] (CUDA tensors or numpy, as ``Engine.lnlike_batch``) -> lnL [B]."""
        with self._lock:
            self.ncalls += 1
            return self.engine.lnlike_batch(theta, star)

    def cont_batch(self, theta, star):
        """Marginalised continua (a star's ``cont_box``): c-hat and packed Cholesky factors of every row (numpy)."""
        coef, chol, _, _ = self._cont(theta, star)
        return coef.cpu().numpy(), chol.cpu().numpy()

    def _cont(self, theta, star):
        with self._lock:
            return self.engine.cont_batch(theta, star)

    def star(self, k):
        """Star k with the interface of ``likelihood.likelihood``."""
        if not 0 <= k < self.n_stars:
            raise IndexError('star %d of %d' % (k, self.n_stars))
        return StarView(self, k)


def _is_per_star(fitpars, S):
    # [names, flags] for all stars vs a list of S such pairs
    return len(fitpars) == S and all(isinstance(f, (list, tuple)) and len(f) == 2 and isinstance(f[1], dict)
                                     for f in fitpars)


class StarView(_Likelihood):
    """One star of a ``StarSetLikelihood`` with the interface of ``likelihood.likelihood`` and the star's own
    ``fixedpars``.  Its rows [B, ndim] are padded to the engine's width before they are posted."""

    def __init__(self, owner, k):
        self.owner, self.k = owner, int(k)
        own = getattr(owner, 'star_fitpars_i', None)        # an owner without it has one layout for all stars
        self.fitargs = owner.fitargs_list[self.k]
        super().__init__(own[self.k] if own is not None else owner.fitpars_i, self.fitargs.get('fixedpars', {}))

    def _pad(self, theta):
        # columns beyond the star's ndim are never read (NaN keeps a wrong read visible)
        w = self.owner.ndim - self.ndim
        if w == 0:
            return theta
        if hasattr(theta, 'is_cuda'):
            import torch
            return torch.nn.functional.pad(theta, (0, w), value=float('nan'))
        theta = np.asarray(theta, dtype=np.float64)
        return np.concatenate([theta, np.full((len(theta), w), np.nan)], axis=1)

    def _lnlike(self, theta):
        theta = self._pad(theta)
        if hasattr(theta, 'is_cuda') and theta.is_cuda:
            import torch
            star = torch.full((theta.shape[0],), self.k, dtype=torch.int32, device=theta.device)
        else:
            star = np.full(len(theta), self.k, dtype=np.int32)
        return self.owner.lnlike_batch(theta, star)

    def _cont(self, theta):
        theta = self._pad(np.asarray(theta, dtype=np.float64))
        return self.owner._cont(theta, np.full(len(theta), self.k, dtype=np.int32))


class _Released(Exception):
    """The batcher stopped (its likelihood raised) while this participant waited."""


class LockstepBatcher(object):
    """Barrier that turns the likelihood calls of n participants into one call.

    ``fn(theta_cat, star_cat) -> values`` with ``theta_cat`` the posted arrays concatenated in participant order
    and ``star_cat`` the participant index of every row.  ``call(k, theta)`` posts and blocks until every
    participant that has not left has posted too, then returns participant k's slice.  ``leave(k)``: k makes no
    more calls.  If ``fn`` raises, every waiting participant raises that exception."""

    def __init__(self, fn, n):
        self.fn = fn
        self.cv = threading.Condition()
        self.active = set(range(n))
        self.pending = {}
        self.results = {}
        self.error = None
        self.ncalls = 0
        self.batch_sizes = []

    def call(self, k, theta):
        theta = np.ascontiguousarray(np.asarray(theta, dtype=np.float64))
        with self.cv:
            if self.error is not None:
                raise _Released() from self.error
            if k not in self.active or k in self.pending:
                raise RuntimeError('participant %d cannot post now' % k)
            self.pending[k] = theta
            self._run_if_complete()
            while k not in self.results:
                if self.error is not None:
                    raise _Released() from self.error
                self.cv.wait()
            return self.results.pop(k)

    def leave(self, k):
        with self.cv:
            self.active.discard(k)
            self._run_if_complete()

    def _run_if_complete(self):
        # (lock held) every participant still active has posted: one call for all of them
        if not self.pending or not self.active.issubset(self.pending.keys()):
            return
        ks = sorted(self.pending)
        theta = np.concatenate([self.pending[k] for k in ks], axis=0)
        star = np.concatenate([np.full(len(self.pending[k]), k, dtype=np.int32) for k in ks])
        try:
            out = np.asarray(self.fn(theta, star))
        except BaseException as e:                      # noqa: B036 -- handed to every waiting thread
            self.error = e
            self.pending.clear()
            self.cv.notify_all()
            return
        self.ncalls += 1
        self.batch_sizes.append(len(theta))
        o = 0
        for k in ks:
            n = len(self.pending[k])
            self.results[k] = out[o:o + n]
            o += n
        self.pending.clear()
        self.cv.notify_all()


class _BatchedStarView(StarView):
    """A star's view whose batched calls go through the lock-step batcher.  ``lnlikefn`` goes straight to the owner:
    one row through the barrier would wait for every other sampler."""

    def __init__(self, owner, k, batcher):
        super().__init__(owner, k)
        self.batcher = batcher

    def _lnlike_batch(self, theta):
        return self.batcher.call(self.k, self._pad(theta))


class FitPayneMany(object):
    """``FitPayne`` for many stars sharing one emulator: one engine, samplers in lock-step (module docstring)."""

    def run(self, *args, **kwargs):
        """``inputdicts=[inputdict, ...]``, each as ``FitPayne.run(inputdict=...)`` takes it (its own ``output``
        file and ``sampler`` settings).  Returns the list of samplers in star order.  ``precision`` and
        ``device`` come from the first dictionary."""
        if 'inputdicts' not in kwargs:
            raise IOError('NO USER DEFINED INPUT DICTS, NOTHING TO FIT!')
        inputdicts = list(kwargs['inputdicts'])
        verbose = kwargs.get('verbose', True)
        fits, indicts = [], []
        for d in inputdicts:
            if isinstance(d.get('spec'), (list, tuple)):
                raise NotImplementedError('FitPayneMany with several spectra per star (a list-valued spec)')
            if d.get('binary', False):
                raise NotImplementedError('FitPayneMany with binaries: fit each binary with FitPayne')
            f = FitPayne()
            ind = f._setup(inputdict=d, verbose=verbose)
            f._prepare(ind)
            f._check_sampler(ind)
            fits.append(f)
            indicts.append(ind)
        self.fits = fits
        self.likeobj = StarSetLikelihood([ind['fitargs'] for ind in indicts], [ind['fitpars'] for ind in indicts],
                                         [ind['runbools'] for ind in indicts], precision=fits[0].precision,
                                         device=fits[0].device)
        self.batcher = LockstepBatcher(self.likeobj.lnlike_batch, len(fits))
        for k, f in enumerate(fits):
            f.likeobj = _BatchedStarView(self.likeobj, k, self.batcher)
        samplers, errors = run_lockstep([lambda f=f, ind=ind: f._runsampler(ind['sampler'])
                                         for f, ind in zip(fits, indicts)], self.batcher)
        for e in errors:
            if e is not None:
                raise e
        return samplers


def run_lockstep(jobs, batcher):
    """Run ``jobs[k]()`` in thread k; job k's batched calls go through ``batcher`` as participant k.  Returns
    (results, exceptions) in job order once every thread has ended.  A job that returns or raises leaves the
    barrier, so the others never wait for it."""
    results, errors = [None] * len(jobs), [None] * len(jobs)

    def body(k):
        try:
            results[k] = jobs[k]()
        except _Released as e:
            errors[k] = e.__cause__ if e.__cause__ is not None else e
        except BaseException as e:                      # noqa: B036 -- re-raised by the caller
            errors[k] = e
        finally:
            batcher.leave(k)

    threads = [threading.Thread(target=body, args=(k,), name='lockstep-%d' % k, daemon=True)
               for k in range(len(jobs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    return results, errors
