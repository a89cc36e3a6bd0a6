"""CPU: the lock-step batcher of fitting/multistar.py with a fake numpy likelihood.

Several participants (threads) post their points; one call per round covers every participant still running,
concatenated in participant order, and each gets back exactly its slice.  Participants finish at different
times; one that raises leaves the barrier and the others run on; a likelihood that raises reaches every waiting
participant.  Nothing may hang: every run has a watchdog."""
import threading

import numpy as np
import pytest

from thepayne_b200.fitting.multistar import LockstepBatcher, run_lockstep


def fake_lnlike(theta, star):
    return -0.5 * np.sum(theta ** 2, axis=1) + 1000.0 * star


def _run(jobs, batcher, timeout=30.0):
    box = {}
    t = threading.Thread(target=lambda: box.setdefault('r', run_lockstep(jobs, batcher)), daemon=True)
    t.start()
    t.join(timeout)
    assert not t.is_alive(), 'lock-step run hung'
    return box['r']


def _job(batcher, k, sizes, seed, log, fail_at=None):
    def run():
        rng = np.random.default_rng(seed)
        got = []
        for i, n in enumerate(sizes):
            if fail_at == i:
                raise KeyError('sampler %d failed' % k)
            th = rng.standard_normal((n, 3))
            out = batcher.call(k, th)
            assert out.shape == (n,)
            np.testing.assert_array_equal(out, fake_lnlike(th, np.full(n, k)))
            got.append(out)
        log[k] = got
        return len(sizes)
    return run


def test_slices_are_each_participants_own_rows():
    calls = []

    def fn(theta, star):
        calls.append(star.copy())
        return fake_lnlike(theta, star)

    b = LockstepBatcher(fn, 3)
    log = {}
    sizes = [[5, 7, 1], [64, 3, 9], [2, 2, 2]]
    res, err = _run([_job(b, k, sizes[k], 10 + k, log) for k in range(3)], b)
    assert err == [None, None, None] and res == [3, 3, 3]
    assert b.ncalls == 3 and len(calls) == 3
    for i, st in enumerate(calls):             # concatenated in participant order
        assert np.array_equal(st, np.repeat([0, 1, 2], [sizes[0][i], sizes[1][i], sizes[2][i]]))
    assert b.batch_sizes == [71, 12, 12]


def test_participants_finishing_at_different_times():
    b = LockstepBatcher(fake_lnlike, 4)
    log = {}
    sizes = [[4] * 2, [3] * 7, [5] * 1, [6] * 4]
    res, err = _run([_job(b, k, sizes[k], k, log) for k in range(4)], b)
    assert err == [None] * 4 and res == [2, 7, 1, 4]
    assert b.ncalls == 7                        # the longest participant's count, not the sum
    assert b.batch_sizes == [18, 13, 9, 9, 3, 3, 3]


def test_exception_in_one_participant_is_returned_and_the_others_finish():
    b = LockstepBatcher(fake_lnlike, 3)
    log = {}
    jobs = [_job(b, 0, [3] * 5, 0, log), _job(b, 1, [2] * 5, 1, log, fail_at=2), _job(b, 2, [4] * 5, 2, log)]
    res, err = _run(jobs, b)
    assert isinstance(err[1], KeyError) and err[0] is None and err[2] is None
    assert res[0] == 5 and res[2] == 5 and sorted(log) == [0, 2]
    assert b.ncalls == 5


def test_likelihood_exception_reaches_every_waiting_participant():
    n = {'calls': 0}

    def fn(theta, star):
        n['calls'] += 1
        if n['calls'] == 3:
            raise FloatingPointError('device said no')
        return fake_lnlike(theta, star)

    b = LockstepBatcher(fn, 3)
    res, err = _run([_job(b, k, [2] * 6, k, {}) for k in range(3)], b)
    assert all(isinstance(e, FloatingPointError) for e in err), err
    with pytest.raises(Exception):
        b.call(0, np.zeros((1, 3)))              # the batcher stays stopped


def test_fitpaynemany_reraises_a_sampler_exception(monkeypatch):
    """FitPayneMany.run re-raises the first sampler exception after every thread has ended (stand-in stars: the
    engine is replaced by the fake likelihood, so no GPU is involved)."""
    from thepayne_b200.fitting import multistar

    class FakeSet(object):
        def __init__(self, fitargs_list, fitpars, runbools, precision='parity', device=None):
            self.n_stars, self.ncalls = len(fitargs_list), 0
            self.fitpars_i = [p for p in fitpars[0][0] if fitpars[0][1][p]]
            self.ndim, self.fixedpars, self.fitargs_list = len(self.fitpars_i), {}, fitargs_list

        def lnlike_batch(self, theta, star):
            self.ncalls += 1
            return fake_lnlike(theta, star)

    ran = []

    def fake_runsampler(self, samplerdict):
        ran.append(samplerdict['seed'])
        for _ in range(3):
            self.likeobj.lnlike_batch(np.zeros((4, self.likeobj.ndim)))
        if samplerdict['seed'] == 1:
            raise ValueError('star 1 diverged')
        return samplerdict['seed']

    monkeypatch.setattr(multistar, 'StarSetLikelihood', FakeSet)
    monkeypatch.setattr(multistar.FitPayne, '_runsampler', fake_runsampler)
    box = {'Teff': {'pv_uniform': [4000.0, 6000.0]}, 'log(g)': {'pv_uniform': [4.0, 5.0]},
           'Av': {'pv_uniform': [0.0, 1.0]}, 'log(A)': {'pv_uniform': [0.0, 1.0]},
           '[Fe/H]': {'pv_uniform': [-0.1, 0.1]}, '[a/Fe]': {'pv_uniform': [-0.1, 0.1]}}
    dicts = [{'phot': {'Bessell_V': [5.0, 0.05]}, 'photANNpath': None, 'photscale': True, 'priordict': dict(box),
              'sampler': {'seed': k}, 'output': 'unused'} for k in range(3)]
    many = multistar.FitPayneMany()
    with pytest.raises(ValueError, match='star 1 diverged'):
        many.run(inputdicts=dicts, verbose=False)
    assert sorted(ran) == [0, 1, 2] and many.batcher.ncalls == 3
