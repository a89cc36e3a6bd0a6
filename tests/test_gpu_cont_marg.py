"""Continuum marginalisation (payne_ctx_set_cont_marg, Engine(cont_box=...)): the Chebyshev continuum integrated out
per point instead of sampled.

The anchor is bit-identity: Q (the chi2 at the best-fitting coefficients c-hat) and the model rows equal, NaN patterns
included, what a context that samples pc_0 .. pc_{K-1} gives when fed theta with c-hat appended.  Then an fp64 numpy
oracle of G, L, c-hat and lnL; the normalisation by quadrature over the coefficients; observation sets, targets,
determinism, the failure cases and refusals; and FitPayne with sampled against marginal coefficients.
"""
import numpy as np
import pytest
import torch
from scipy.integrate import simpson

from thepayne_b200 import _lib, synth
from thepayne_b200.engine import Engine
from test_gpu_targets import _emulator, _targets, _theta

pytestmark = pytest.mark.gpu
_INVALID, _UNSUPPORTED = -1, -4
LABELS = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]']
LN2PI = np.log(2.0 * np.pi)


def _box(K):
    return [(0.75, 1.25)] + [(-0.5, 0.5)] * (K - 1)


def _obs(spec, n=1500, f=(0.1, 0.9), seed=0):
    w = spec.wavelength
    a, b = w[0], w[-1]
    rng = np.random.default_rng(seed)
    g = np.linspace(a + f[0] * (b - a), a + f[1] * (b - a), n)
    x = 2.0 * (g - g[0]) / (g[-1] - g[0]) - 1.0
    cont = 1.02 + 0.03 * x - 0.01 * x * x
    return g, cont * (1.0 + 0.02 * rng.standard_normal(n)), 0.02 + 0.005 * rng.random(n)


def _pair(spec, K, instr, obs, phot=None, obs_phot=None):
    """(marginal engine, sampled engine) of one star; instr 'free', a fixed value, or 0 (no instrumental stage)"""
    fit = LABELS + ['Vrad', 'Vrot'] + (['Inst_R'] if instr == 'free' else [])
    fixed = {} if instr == 'free' else {'Inst_R': float(instr)}
    pfit = ['log(R)', 'Dist', 'Av'] if phot is not None else []
    rb = [True, phot is not None, False, False, False]
    kw = dict(spec=spec, phot=phot, obs_wave=obs[0], obs_flux=obs[1], obs_eflux=obs[2], obs_phot=obs_phot,
              fixedpars=fixed)
    marg = Engine(fitpars_i=fit + pfit, runbools=rb, cont_box=_box(K), **kw)
    samp = Engine(fitpars_i=fit + pfit + ['pc_%d' % k for k in range(K)], runbools=[True, rb[1], True, False, False],
                  **kw)
    samp.set('tail_cluster', 0)                             # 65536 samples: the single-CTA kernel, as the marginal path
    return marg, samp


def _rows(B, ncol, seed, instr_col=True):
    rng = np.random.default_rng(seed)
    box = dict(synth._BOX, Vrad=(-30.0, 30.0), Vrot=(0.5, 12.0), Inst_R=(25000.0, 40000.0))
    names = LABELS + ['Vrad', 'Vrot'] + (['Inst_R'] if instr_col else [])
    th = np.stack([box[p][0] + (box[p][1] - box[p][0]) * rng.random(B) for p in names], axis=1)
    th[rng.random(B) < 0.25, 5] = 0.0                       # Vrot = 0: no rotation stage
    return np.hstack([th, np.zeros((B, ncol - th.shape[1]))]) if ncol > th.shape[1] else th


def _np(t):
    return t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def _unpack(chol, K):
    L = np.zeros((len(chol), K, K))
    i, j = np.tril_indices(K)
    L[:, i, j] = chol[:, :K * (K + 1) // 2]
    return L


def _anchor(marg, samp, th, K):
    coef, chol, q, lnl = [_np(v) for v in marg.cont_batch(th)]
    fm, _, lm = marg.model_batch(th, want_mags=False)
    ths = np.hstack([th, coef[:, :K]])
    fs, _, ls = samp.model_batch(ths, want_mags=False)
    assert np.array_equal(q, -2.0 * _np(ls), equal_nan=True)
    assert np.array_equal(_np(fm), _np(fs), equal_nan=True)
    assert np.array_equal(_np(lm), lnl, equal_nan=True)
    assert np.array_equal(marg.lnlike_batch(th), lnl, equal_nan=True)
    return coef, chol, q, lnl


def _oracle(marg, samp, obs, th, K, coef, lnl):
    """G, L, c-hat and lnL in fp64 from a_j (the sampled context's model at c = e_0, bit-exact)"""
    e0 = np.zeros((len(th), K))
    e0[:, 0] = 1.0
    a, _, _ = samp.model_batch(np.hstack([th, e0]), want_mags=False)
    a = _np(a)
    w, o, s = obs
    x = 2.0 * ((w - w.min()) / (w.max() - w.min())) - 1.0
    V = np.polynomial.chebyshev.chebvander(x, K - 1)
    C = sum(0.5 * LN2PI - np.log(hi - lo) for lo, hi in _box(K))
    n_ok = 0
    for p in range(len(th)):
        if not np.all(np.isfinite(a[p])):
            assert np.isnan(lnl[p])
            continue
        b = a[p][:, None] * V / s[:, None]
        G, h = b.T @ b, b.T @ (o / s)
        L = np.linalg.cholesky(G)
        c = np.linalg.solve(G, h)
        Q = np.sum((b @ c - o / s) ** 2)
        ref = -0.5 * Q - np.sum(np.log(np.diag(L))) + C
        assert np.allclose(coef[p, :K], c, rtol=1e-9, atol=1e-9 * np.abs(c).max())
        assert abs(lnl[p] - ref) <= 1e-8 * abs(ref)
        n_ok += 1
    assert n_ok > 0


SIZES = [(10, 1, 'free'), (11, 2, 31000.0), (12, 5, 0.0), (13, 16, 'free'), (14, 2, 0.0), (15, 5, 'free'),
         (16, 1, 28000.0)]


@pytest.mark.parametrize('l2,K,instr', SIZES)
def test_anchor_and_oracle_every_size(l2, K, instr):
    spec = _emulator(l2)
    obs = _obs(spec, n=900 if l2 <= 11 else 2500, seed=l2)
    marg, samp = _pair(spec, K, instr, obs)
    assert marg.query('nfft1') == 1 << l2 and marg.query('cont_marg') == 1
    th = _rows(24, marg.ndim, seed=l2, instr_col=instr == 'free')
    coef, chol, q, lnl = _anchor(marg, samp, th, K)
    assert np.isfinite(lnl).sum() >= 20
    _oracle(marg, samp, obs, th, K, coef, lnl)


@pytest.mark.parametrize('K', [1, 2, 5, 16])
@pytest.mark.parametrize('instr', ['free', 33000.0, 0.0])
def test_anchor_orders_and_stages(K, instr):
    spec = _emulator(13)
    obs = _obs(spec, n=3000, seed=K)
    marg, samp = _pair(spec, K, instr, obs)
    th = _rows(64, marg.ndim, seed=K + 7, instr_col=instr == 'free')
    th[::9, 4] = 1500.0                                     # shifted off the grid: NaN pixels
    coef, chol, q, lnl = _anchor(marg, samp, th, K)
    assert np.isnan(lnl[::9]).all() and np.isfinite(lnl[1:9]).all()
    assert (marg.query('status') & 8) == 0


def _sampled_grid_lnz(samp, th_row, c, L, K, n):
    """ln of the integral of exp(lnL(c)) over c-hat +- 8 sd (Simpson's rule, one batch)"""
    cov = np.linalg.inv(L @ L.T)
    axes = [c[k] + 8.0 * np.sqrt(cov[k, k]) * np.linspace(-1.0, 1.0, n) for k in range(K)]
    mesh = np.stack(np.meshgrid(*axes, indexing='ij'), axis=-1).reshape(-1, K)
    l = samp.lnlike_batch(np.hstack([np.repeat(th_row[None], len(mesh), 0), mesh])).reshape((n,) * K)
    m = l.max()
    f = np.exp(l - m)
    for k in reversed(range(K)):
        f = simpson(f, x=axes[k], axis=k)
    return m + np.log(f)


@pytest.mark.parametrize('K,n', [(1, 401), (2, 161)])
def test_quadrature_normalisation(K, n):
    spec = _emulator(12)
    obs = _obs(spec, n=1200, seed=5)
    marg, samp = _pair(spec, K, 'free', obs)
    th = _rows(3, marg.ndim, seed=11)
    th[:, 5] = 4.0
    coef, chol, q, lnl = [_np(v) for v in marg.cont_batch(th)]
    L = _unpack(chol, K)
    logw = sum(np.log(hi - lo) for lo, hi in _box(K))
    for p in range(len(th)):
        lnz = _sampled_grid_lnz(samp, th[p], coef[p, :K], L[p], K, n) - logw
        assert abs(lnz - lnl[p]) < 1e-6


def test_optimality():
    spec = _emulator(12)
    obs = _obs(spec, n=1500, seed=9)
    K = 4
    marg, samp = _pair(spec, K, 'free', obs)
    th = _rows(8, marg.ndim, seed=13)
    coef, chol, q, lnl = [_np(v) for v in marg.cont_batch(th)]
    L = _unpack(chol, K)
    rng = np.random.default_rng(1)
    at = samp.lnlike_batch(np.hstack([th, coef]))
    for _ in range(4):
        d = np.stack([np.linalg.solve(L[p].T, 0.1 * rng.standard_normal(K)) for p in range(len(th))])
        assert np.all(samp.lnlike_batch(np.hstack([th, coef + d])) < at)


def _set_stars(spec, phot):
    """per-star layouts with different K, photometry on stars 0 and 2 only"""
    Ks = [3, 1, 6, 2]
    stars = []
    for k, K in enumerate(Ks):
        w, f, e = _obs(spec, n=800 + 300 * k, f=(0.05 + 0.05 * k, 0.8 + 0.04 * k), seed=20 + k)
        fit = LABELS + ['Vrad', 'Vrot', 'Inst_R'] + (['log(R)', 'Dist', 'Av'] if k % 2 == 0 else [])
        st = {'wave': w, 'flux': f, 'eflux': e, 'fitpars_i': fit, 'runbools': [True, k % 2 == 0, False, False],
              'cont_box': [(0.8, 1.2)] + [(-0.3 - 0.1 * i, 0.2 + 0.1 * i) for i in range(K - 1)]}
        if k % 2 == 0:
            st['phot'] = {b: (5.0 + 0.3 * i + 0.1 * k, 0.02) for i, b in enumerate(BANDS)}
        stars.append(st)
    return stars


BANDS = synth.PROCYON_BANDS[:4]


def test_observation_set_layouts_and_photometry():
    spec = _emulator(13)
    phot = synth.make_photnet(BANDS, H=16)
    stars = _set_stars(spec, phot)
    eng = Engine(spec=spec, phot=phot, stars=stars)
    B = 64
    th = _rows(B, eng.ndim, seed=3)
    rng = np.random.default_rng(4)
    th[:, 7] = rng.uniform(-0.05, 0.05, B)
    th[:, 8] = rng.uniform(5.0, 50.0, B)
    th[:, 9] = rng.uniform(0.0, 0.5, B)
    star = rng.integers(0, len(stars), B).astype(np.int32)
    coef, chol, q, lnl = [_np(v) for v in eng.cont_batch(th, star)]
    assert np.array_equal(eng.lnlike_batch(th, star), lnl, equal_nan=True)
    for k, st in enumerate(stars):
        rows = np.nonzero(star == k)[0]
        K = len(st['cont_box'])
        hasp = 'phot' in st
        one = Engine(spec=spec, phot=phot if hasp else None, obs_wave=st['wave'], obs_flux=st['flux'],
                     obs_eflux=st['eflux'], obs_phot=st.get('phot'),
                     fitpars_i=st['fitpars_i'] + ['pc_%d' % i for i in range(K)],
                     runbools=[True, hasp, True, False, False])
        ths = np.hstack([th[rows][:, :len(st['fitpars_i'])], coef[rows][:, :K]])
        ls = one.lnlike_batch(ths)
        C = sum(0.5 * LN2PI - np.log(hi - lo) for lo, hi in st['cont_box'])
        M = -np.log(np.diagonal(_unpack(chol[rows], K), axis1=1, axis2=2)).sum(axis=1) + C
        # lnL = -0.5 (Q + chi2_sed) + M, and -0.5 (Q + chi2_sed) is the sampled context's lnL at c-hat
        assert np.allclose(lnl[rows], ls + M, rtol=1e-12, atol=0)
        if not hasp:
            assert np.array_equal(q[rows], -2.0 * ls, equal_nan=True)
        assert np.isnan(coef[rows][:, K:]).all()
        one.close()


def test_targets_members_differ_in_k():
    spec = _emulator(13)
    stars, counts = _targets(spec)
    Ks = [2, 4, 1, 3, 5, 2, 1, 3]
    for st, K in zip(stars, Ks):
        st['cont_box'] = _box(K)
    eng = Engine(spec=spec, stars=stars, targets=counts)
    th, tgt = _theta(stars, counts, 96, seed=5)
    coef, chol, q, lnl = [_np(v) for v in eng.cont_batch_targets(th, tgt)]
    assert np.array_equal(eng.lnlike_batch_targets(th, tgt), lnl, equal_nan=True)
    first = np.concatenate([[0], np.cumsum(counts)])
    Mall = np.full(q.shape, np.nan)
    for t in range(len(counts)):
        rows = np.nonzero(tgt == t)[0]
        co = lo = 0
        for m, k in enumerate(range(first[t], first[t + 1])):
            st, K = stars[k], Ks[k]
            one = Engine(spec=spec, obs_wave=st['wave'], obs_flux=st['flux'], obs_eflux=st['eflux'],
                         fitpars_i=st['fitpars_i'] + ['pc_%d' % i for i in range(K)], fixedpars=st['fixedpars'],
                         runbools=[True, False, True, False, False])
            ths = np.hstack([th[rows][:, :len(st['fitpars_i'])], coef[rows][:, co:co + K]])
            assert np.array_equal(q[rows, m], -2.0 * one.lnlike_batch(ths), equal_nan=True)
            # the member's c-hat and L are those of a single-star marginal context of that member
            solo = Engine(spec=spec, obs_wave=st['wave'], obs_flux=st['flux'], obs_eflux=st['eflux'],
                          fitpars_i=st['fitpars_i'], fixedpars=st['fixedpars'], cont_box=_box(K))
            sc, sl, sq, _ = [_np(v) for v in solo.cont_batch(np.ascontiguousarray(th[rows][:, :len(st['fitpars_i'])]))]
            assert np.array_equal(coef[rows][:, co:co + K], sc[:, :K], equal_nan=True)
            assert np.array_equal(chol[rows][:, lo:lo + K * (K + 1) // 2], sl, equal_nan=True)
            assert np.array_equal(q[rows, m], sq, equal_nan=True)
            solo.close()
            C = sum(0.5 * LN2PI - np.log(hi - lo_) for lo_, hi in _box(K))
            Lm = _unpack(chol[rows][:, lo:lo + K * (K + 1) // 2], K)
            Mall[rows, m] = -np.log(np.diagonal(Lm, axis1=1, axis2=2)).sum(axis=1) + C
            co += K
            lo += K * (K + 1) // 2
            one.close()
    for p in range(len(th)):
        n = counts[tgt[p]]
        Q, M = q[p, 0], Mall[p, 0]
        for m in range(1, n):
            Q, M = Q + q[p, m], M + Mall[p, m]
        ref = -0.5 * Q + M
        if np.isnan(ref):
            assert np.isnan(lnl[p])
        else:
            assert abs(lnl[p] - ref) <= 1e-12 * abs(ref)
    assert np.isnan(lnl[tgt == 3]).all()                    # target 3's second member is bad by itself
    assert np.isfinite(q[tgt == 3, 0]).all()


def test_determinism_grid_caps():
    spec = _emulator(14)
    obs = _obs(spec, n=4000, seed=2)
    marg, _ = _pair(spec, 5, 'free', obs)
    th = _rows(300, marg.ndim, seed=17)
    ref = marg.lnlike_batch(th)
    for cap in (1, 2, 3, 0):
        marg.set('tail_grid_cap', cap)
        assert np.array_equal(marg.lnlike_batch(th), ref, equal_nan=True)
    assert np.array_equal(marg.lnlike_batch(th), ref, equal_nan=True)


def test_failures_and_refusals():
    spec = _emulator(12)
    w, f, e = _obs(spec, n=900, seed=1)
    # fewer pixels than K: a non-positive pivot, NaN and status bit 3
    few = Engine(spec=spec, obs_wave=w[400:403], obs_flux=f[400:403], obs_eflux=e[400:403],
                 fitpars_i=LABELS + ['Vrad', 'Vrot', 'Inst_R'], cont_box=_box(5))
    th = _rows(4, few.ndim, seed=1)
    th[:, 4] = 0.0
    assert np.isnan(few.lnlike_batch(th)).all()
    assert few.query('status') & 8
    # pixels beyond the coverage: NaN as in the sampled path, bit 3 clear
    marg, samp = _pair(spec, 3, 'free', (w, f, e))
    th = _rows(4, marg.ndim, seed=2)
    th[:, 4] = 500.0
    assert np.isnan(marg.lnlike_batch(th)).all() and not (marg.query('status') & 8)
    # removing the setting gives a fresh context's bits
    th = _rows(16, marg.ndim, seed=3)
    marg.set_cont_marg(None)
    fresh = Engine(spec=spec, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=LABELS + ['Vrad', 'Vrot', 'Inst_R'])
    assert np.array_equal(marg.lnlike_batch(th), fresh.lnlike_batch(th), equal_nan=True)
    marg.set_cont_marg([_box(3)])

    def code(fn):
        with pytest.raises(_lib.PayneError) as ei:
            fn()
        return int(str(ei.value).split()[2].rstrip(':'))
    assert code(lambda: samp.set_cont_marg([_box(3)])) == _INVALID                   # pc_k sampled too
    arr = (_lib.PayneContMarg * 1)()
    arr[0].n_coef = 17
    assert fresh.lib.payne_ctx_set_cont_marg(fresh._ctx, arr) == _INVALID
    arr[0].n_coef = 0
    assert fresh.lib.payne_ctx_set_cont_marg(fresh._ctx, arr) == _INVALID
    assert code(lambda: fresh.set_cont_marg([[(1.0, 1.0)]])) == _INVALID
    assert code(lambda: fresh.set_cont_marg([[(0.0, np.inf)]])) == _INVALID
    two = Engine(spec=spec, stars=[{'wave': w, 'flux': f, 'eflux': e}, {'wave': w[:500], 'flux': f[:500],
                                                                        'eflux': e[:500]}],
                 fitpars_i=LABELS + ['Vrad', 'Vrot', 'Inst_R'])
    assert code(lambda: two.set_cont_marg([_box(2), []])) == _UNSUPPORTED           # mixed set
    fresh.set_lsf(np.full(len(w), 0.05))
    assert code(lambda: fresh.set_cont_marg([_box(2)])) == _UNSUPPORTED               # LSF vector
    fresh.set_lsf(None)
    fresh.set_cont_marg([_box(2)])
    fresh.set_lsf(np.full(len(w), 0.05))
    assert code(lambda: fresh.lnlike_batch(th)) == _UNSUPPORTED                        # checked again in the entries
    fresh.set_lsf(None)
    fresh.set('fast_tail', 0)
    assert code(lambda: fresh.lnlike_batch(th)) == _UNSUPPORTED                        # no fast tail
    fresh.set('fast_tail', 1)
    assert np.isfinite(fresh.lnlike_batch(th)).any()
    fresh.set_cont_marg(None)
    fresh.attach_continuum(_emulator(12))
    assert code(lambda: fresh.set_cont_marg([_box(2)])) == _UNSUPPORTED               # continuum emulator
    bfit = LABELS + ['Vrad', 'Vrot', 'Inst_R', 'Teff_sec', 'Rratio']
    binary = Engine(spec=spec, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=bfit, binary=True)
    assert code(lambda: binary.set_cont_marg([_box(2)])) == _UNSUPPORTED              # binary
    odd = synth.make_specnet(4, 64, np.linspace(5140.0, 5190.0, 3000), _emulator(12).resolution, seed=0)
    nonlog = Engine(spec=odd, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=LABELS + ['Vrad', 'Vrot', 'Inst_R'])
    assert nonlog.query('fast_tail') == 0
    assert code(lambda: nonlog.set_cont_marg([_box(2)])) == _UNSUPPORTED              # grid without the fast tail


def test_removing_binaries_keeps_marginalisation():
    """binaries and continuum marginalisation share the per-CTA a_j scratch: clearing the one that is off keeps it"""
    spec = _emulator(13)
    marg, samp = _pair(spec, 3, 'free', _obs(spec, seed=4))
    th = _rows(300, marg.ndim, seed=4)
    lnl = marg.lnlike_batch(th)
    cont = [_np(t) for t in marg.cont_batch(th)]
    marg.set_binary(False)
    assert np.array_equal(marg.lnlike_batch(th), lnl, equal_nan=True) and np.isfinite(lnl).any()
    for a, b in zip(marg.cont_batch(th), cont):
        assert np.array_equal(_np(a), b, equal_nan=True)
    marg.close()
    samp.close()


# ------------------------------------------------------------------ FitPayne, sampled against marginal coefficients

TRUTH = {'Teff': 5770.0, 'log(g)': 4.44, '[Fe/H]': 0.0, '[a/Fe]': 0.0, 'Vrad': 0.5, 'Vrot': 3.0, 'Inst_R': 32000.0}


def _fit(spec, tmp_path, marginal):
    from thepayne_b200.fitting.fitstar import FitPayne
    rng = np.random.default_rng(12)
    w = np.linspace(5150.0, 5180.0, 900)
    one = Engine(spec=spec, obs_wave=w, obs_flux=np.ones(len(w)), obs_eflux=np.ones(len(w)),
                 fitpars_i=LABELS + ['Vrad', 'Vrot', 'Inst_R'])
    f = one.model_batch(np.array([[TRUTH[p] for p in LABELS + ['Vrad', 'Vrot', 'Inst_R']]]),
                        want_mags=False)[0].cpu().numpy()[0]
    one.close()
    x = 2.0 * (w - w[0]) / (w[-1] - w[0]) - 1.0
    f = f * np.polynomial.chebyshev.chebval(x, [1.0, 0.02, -0.01])
    e = np.abs(f) / 40.0
    sp = {'obs_wave': w, 'obs_flux': f + e * rng.standard_normal(len(w)), 'obs_eflux': e, 'convertair': False,
          'modpoly': True, 'polyorder': 2, 'polysigma': 0.1, 'modpoly_marginal': marginal}
    pri = {'Teff': {'pv_uniform': [5400.0, 6100.0]}, 'log(g)': {'pv_uniform': [4.0, 4.8]},
           '[Fe/H]': {'pv_uniform': [-0.1, 0.1]}, '[a/Fe]': {'pv_uniform': [-0.1, 0.1]},
           'Vrad': {'pv_uniform': [-3.0, 3.0]}, 'Vrot': {'fixed': 3.0}, 'Inst_R': {'pv_uniform': [24000.0, 40000.0]}}
    out = str(tmp_path / ('marg.dat' if marginal else 'samp.dat'))
    fp = FitPayne()
    sampler = fp.run(inputdict={'spec': sp, 'specANNpath': spec, 'NNtype': 'LinNet', 'priordict': pri, 'output': out,
                                'sampler': {'samplertype': 'Static', 'samplemethod': 'rwalk', 'npoints': 60,
                                            'walks': 12, 'delta_logz_final': 0.2, 'seed': 5, 'maxiter': 20000}},
                     verbose=False)
    return fp, sampler, out


def _posterior(out, names):
    head = open(out).readline().split()
    d = np.loadtxt(out, skiprows=1)
    lw = d[:, head.index('log(wt)')] - d[:, head.index('log(z)')][-1]
    w = np.exp(lw - lw.max())
    w /= w.sum()
    res = {}
    for p in names:
        v = d[:, head.index(p)]
        m = np.sum(w * v)
        res[p] = (m, np.sqrt(np.sum(w * (v - m) ** 2)))
    return head, res


def test_fitpayne_marginal_matches_sampled(tmp_path):
    spec = _emulator(12)
    fs, ss, out_s = _fit(spec, tmp_path, False)
    fm, sm, out_m = _fit(spec, tmp_path, True)
    assert fm.ndim == fs.ndim - 3
    err = 3.0 * np.sqrt(ss.logzvar + sm.logzvar)
    assert abs(ss.logz - sm.logz) <= err, (ss.logz, sm.logz, err)
    names = LABELS[:3] + ['Vrad', 'Inst_R', 'pc_0', 'pc_1', 'pc_2']
    hs, ps = _posterior(out_s, names)
    hm, pm = _posterior(out_m, names)
    assert hs == hm                                        # the marginal file keeps the pc columns
    for p in names:
        (a, sa), (b, sb) = ps[p], pm[p]
        assert abs(a - b) <= 3.0 * np.hypot(sa, sb) + 1e-12, (p, a, b, sa, sb)
