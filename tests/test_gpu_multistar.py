"""Observation sets: one context holding several stars (payne_ctx_create_stars), every point naming its star.

The core check is bit-identity: a single-star context is already pinned to the reference goldens, so every star's
rows of an interleaved multi-star batch must give exactly (np.array_equal, NaN patterns included) what a single-star
engine gives on those rows -- lnL of the device and host entries, model flux, magnitudes and lnL of model_batch.
The stars share one emulator and differ in observed range and n_obs, sort order, coverage (NaN pixels), mask width
(a different second transform) and magnitudes.  Setups reach the single-CTA fast tail with and without the
continuum polynomial at two transform sizes, the cluster tail (sorted and unsorted grids), the general-grid tail,
photometry-only and joint contexts, both precisions, a slab boundary inside a star's rows and dynamic point
scheduling that hands one CTA points of several stars.

Then: invalid star indices, the refusals on several stars, and FitPayneMany against separate FitPayne runs.
"""
import ctypes

import numpy as np
import pytest
import torch

from thepayne_b200 import _lib, synth
from thepayne_b200.engine import Engine, _specnet_struct

pytestmark = pytest.mark.gpu

BANDS = synth.PROCYON_BANDS[:4]
RANGES = {'mini': (5140.0, 5190.0),       # 3403 pixels -> 4096-sample transforms
          'c2': (5130.0, 5340.0),         # 14172 -> 16384
          'mid': (5000.0, 5280.0),        # 32768
          'wide': (4800.0, 5300.0)}       # 65536


_SPEC_CACHE = {}


def _spec(rng_name):
    if rng_name not in _SPEC_CACHE:
        wave, rsig = synth.ann_wavegrid(*RANGES[rng_name], 50000.0)
        _SPEC_CACHE[rng_name] = synth.make_specnet(4, 64, wave, rsig, seed=0)
    return _SPEC_CACHE[rng_name]


def _stars(spec, nb, seed=5):
    """Six observations inside (and one partly beyond) the emulator's coverage."""
    w = spec.wavelength
    a, b = w[0], w[-1]
    span = b - a
    rng = np.random.default_rng(seed)
    grids = [
        np.linspace(a + 0.10 * span, b - 0.10 * span, 1500),
        np.linspace(a + 0.25 * span, b - 0.05 * span, 2311),
        rng.permutation(np.linspace(a + 0.15 * span, b - 0.20 * span, 977)),          # unsorted
        np.linspace(a - 0.02 * span, b - 0.30 * span, 1201),                          # beyond the coverage: NaN pixels
        np.linspace(a + 0.50 * span, a + 0.53 * span, 257),                           # narrow mask: small N2
        np.linspace(a + 0.05 * span, b - 0.05 * span, 3050),
    ]
    out = []
    for k, g in enumerate(grids):
        flux = 1.0 + 0.05 * rng.standard_normal(len(g))
        eflux = 0.02 + 0.01 * rng.random(len(g))
        phot = {bd: (float(5.0 + k + 0.1 * i), 0.05 + 0.01 * k) for i, bd in enumerate(BANDS[:nb])}
        out.append({'wave': g, 'flux': flux, 'eflux': eflux, 'phot': phot})
    return out


def _layout(spec_on, npoly, bands):
    fit = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]']
    if spec_on:
        fit += ['Vrad', 'Vrot', 'Inst_R']
    if bands:
        fit += ['log(A)', 'Av']
    fit += ['pc_%d' % k for k in range(npoly)]
    box = dict(synth._BOX)
    for k in range(npoly):
        box['pc_%d' % k] = (0.75, 1.25) if k == 0 else (-0.1, 0.1)
    runbools = [spec_on, bool(bands), npoly > 0, bool(bands), False]
    return fit, box, runbools


def _thetas(fit, box, B, seed):
    rng = np.random.default_rng(seed)
    lo = np.array([box[p][0] for p in fit])
    hi = np.array([box[p][1] for p in fit])
    th = lo + (hi - lo) * rng.random((B, len(fit)))
    if 'Inst_R' in fit:
        th[rng.random(B) < 0.1, fit.index('Inst_R')] = 0.0           # no instrumental profile: plain np.interp
        th[rng.random(B) < 0.1, fit.index('Vrot')] = 0.0             # no rotation stage
    return th


SETUPS = {
    # name: (emulator, npoly, bands, precision, settings)
    'fast12': ('mini', 0, 0, 'parity', {}),
    'fast12_poly': ('mini', 3, 0, 'parity', {}),
    'fast14': ('c2', 0, 0, 'parity', {}),
    'fast14_poly': ('c2', 4, 0, 'parity', {}),
    'cluster15': ('mid', 0, 0, 'parity', {'tail_cluster': 1}),
    'cluster16_poly': ('wide', 3, 0, 'parity', {}),
    'general': ('mini', 2, 0, 'parity', {'fast_tail': 0}),
    'phot_only': (None, 0, 4, 'parity', {}),
    'joint': ('mini', 2, 3, 'parity', {}),
    'simt': ('mini', 2, 0, 'simt', {}),
    'slab200': ('mini', 0, 0, 'parity', {'max_batch': 200}),
    'slab200_cluster': ('wide', 0, 0, 'parity', {'max_batch': 200}),
    'cap1': ('mini', 0, 0, 'parity', {'tail_grid_cap': 1}),
    'cap3_poly': ('c2', 2, 0, 'parity', {'tail_grid_cap': 3}),
    'cap2_cluster': ('mid', 2, 0, 'parity', {'tail_cluster': 1, 'tail_grid_cap': 2}),
}


def _build(name, n_stars=None):
    emu, npoly, nb, prec, settings = SETUPS[name]
    spec = _spec(emu) if emu else _spec('mini')
    phot = synth.make_photnet(BANDS[:nb], H=16) if nb else None
    fit, box, runbools = _layout(emu is not None, npoly, BANDS[:nb])
    stars = _stars(spec, nb)[:n_stars]
    kw = dict(spec=spec if emu else None, phot=phot, fitpars_i=fit, fixedpars={}, runbools=runbools, precision=prec)
    return kw, stars, fit, box, settings


def _apply(eng, settings):
    for k, v in settings.items():
        eng.set(k, v)


@pytest.mark.parametrize('name', list(SETUPS))
def test_stars_bit_identical_to_single_star_engines(name):
    kw, stars, fit, box, settings = _build(name)
    S = len(stars)
    multi = Engine(stars=stars, **kw)
    _apply(multi, settings)
    assert multi.query('n_stars') == S
    if kw['spec'] is not None:
        assert multi.query('n_obs') == max(len(s['wave']) for s in stars)
        assert multi.query('n_obs_total') == sum(len(s['wave']) for s in stars)
    if name.startswith('cluster') or name.endswith('_cluster'):
        assert multi.query('tail_cluster') == 1
    if name == 'general':
        assert multi.query('fast_tail') == 0
    B = 520
    th = _thetas(fit, box, B, seed=sum(map(ord, name)))
    rng = np.random.default_rng(17)
    star = rng.integers(0, S, B).astype(np.int32)
    star[:250] = 1                      # a run of one star's rows across the 200-point slab boundary
    tht = torch.from_numpy(np.ascontiguousarray(th)).cuda()
    stt = torch.from_numpy(star).cuda()
    lnl_d = multi.lnlike_batch(tht, stt).cpu().numpy()
    flux, mags, lnl_m = multi.model_batch(tht, stt)
    lnl_h = multi.lnlike_batch(th, star)
    torch.cuda.synchronize()
    flux = flux.cpu().numpy() if flux is not None else None
    mags = mags.cpu().numpy() if mags is not None else None
    lnl_m = lnl_m.cpu().numpy()
    assert multi.query('status') == 0
    n_finite = 0
    for k in range(S):
        idx = np.flatnonzero(star == k)
        one = Engine(obs_wave=stars[k]['wave'] if kw['spec'] is not None else None,
                     obs_flux=stars[k]['flux'] if kw['spec'] is not None else None,
                     obs_eflux=stars[k]['eflux'] if kw['spec'] is not None else None,
                     obs_phot=stars[k]['phot'] if kw['phot'] is not None else None, **kw)
        _apply(one, settings)
        t1 = torch.from_numpy(np.ascontiguousarray(th[idx])).cuda()
        ref_d = one.lnlike_batch(t1).cpu().numpy()
        rf, rm, rl = one.model_batch(t1)
        ref_h = one.lnlike_batch(th[idx])
        torch.cuda.synchronize()
        assert np.array_equal(lnl_d[idx], ref_d, equal_nan=True), (name, k)
        assert np.array_equal(lnl_h[idx], ref_h, equal_nan=True), (name, k)
        assert np.array_equal(lnl_m[idx], rl.cpu().numpy(), equal_nan=True), (name, k)
        if flux is not None:
            n = len(stars[k]['wave'])
            assert np.array_equal(flux[idx, :n], rf.cpu().numpy(), equal_nan=True), (name, k)
            assert np.isnan(flux[idx, n:]).all()                         # beyond the star's pixels: not written
        if mags is not None:
            assert np.array_equal(mags[idx], rm.cpu().numpy(), equal_nan=True), (name, k)
        n_finite += int(np.isfinite(ref_d).sum())
        one.close()
    assert n_finite > B // 4                 # the comparison is not between NaN vectors
    if kw['spec'] is not None:
        assert np.isnan(flux[star == 3]).any()           # star 3 reaches beyond the emulator's coverage
    multi.close()


def _raw_ctx(lib, kw, star, n_stars=1, use_create=False):
    """A context made through the C ABI directly (payne_ctx_create or payne_ctx_create_stars)."""
    keep = []
    sp = _specnet_struct(kw['spec'], keep)
    lay = _lib.PayneLayout()
    fit = kw['fitpars_i']
    lay.ndim = len(fit)
    for nm, k in _lib.PAR_INDEX.items():
        lay.col[k] = fit.index(nm) if nm in fit else -1
        lay.fixed[k] = float('nan')
    pcs = [i for i, p in enumerate(fit) if 'pc' in p]
    lay.n_poly = len(pcs)
    for i, c in enumerate(pcs):
        lay.poly_col[i] = c
    rb = kw['runbools']
    lay.spec_bool, lay.phot_bool, lay.modpoly_bool, lay.photscale_bool = [int(bool(b)) for b in rb[:4]]
    lay.precision = _lib.PREC[kw['precision']]
    obs = (_lib.PayneObs * n_stars)()
    for k in range(n_stars):
        ow, of, oe = [np.ascontiguousarray(star[k][x], dtype=np.float64) for x in ('wave', 'flux', 'eflux')]
        keep += [ow, of, oe]
        obs[k].n_obs = len(ow)
        obs[k].wave, obs[k].flux, obs[k].eflux = [a.ctypes.data_as(ctypes.POINTER(ctypes.c_double)) for a in (ow, of, oe)]
    ctx = ctypes.c_void_p()
    if use_create:
        rc = lib.payne_ctx_create(ctypes.byref(sp), None, obs, ctypes.byref(lay), 0, ctypes.byref(ctx))
    else:
        rc = lib.payne_ctx_create_stars(ctypes.byref(sp), None, obs, n_stars, ctypes.byref(lay), 0, ctypes.byref(ctx))
    assert rc == 0, lib.payne_last_error()
    return ctx


def test_create_stars_of_one_star_matches_create():
    lib = _lib.load()
    kw, stars, fit, box, _ = _build('fast12_poly')
    th = torch.from_numpy(_thetas(fit, box, 300, seed=4)).cuda()
    outs = []
    for use_create in (True, False):
        ctx = _raw_ctx(lib, kw, stars[:1], 1, use_create)
        lnl = torch.empty(300, dtype=torch.float64, device='cuda')
        flux = torch.empty((300, len(stars[0]['wave'])), dtype=torch.float64, device='cuda')
        st = torch.cuda.current_stream().cuda_stream
        assert lib.payne_lnlike_batch(ctx, th.data_ptr(), 300, th.shape[1], lnl.data_ptr(), st) == 0
        assert lib.payne_model_batch(ctx, th.data_ptr(), 300, th.shape[1], flux.data_ptr(), None, None, st) == 0
        torch.cuda.synchronize()
        outs.append((lnl.cpu().numpy(), flux.cpu().numpy()))
        lib.payne_ctx_destroy(ctx)
    assert np.array_equal(outs[0][0], outs[1][0], equal_nan=True)
    assert np.array_equal(outs[0][1], outs[1][1], equal_nan=True)
    assert np.isfinite(outs[0][0]).sum() > 100


@pytest.mark.parametrize('name', ['fast12_poly', 'joint', 'phot_only', 'cluster16_poly', 'general'])
def test_invalid_star_index(name):
    lib = _lib.load()
    kw, stars, fit, box, settings = _build(name, n_stars=3)
    eng = Engine(stars=stars, **kw)
    _apply(eng, settings)
    B = 300
    th = _thetas(fit, box, B, seed=8)
    rng = np.random.default_rng(2)
    star = rng.integers(0, 3, B).astype(np.int32)
    bad = np.zeros(B, dtype=bool)
    bad[[0, 7, 150, 299]] = True
    star[bad] = np.array([-1, 3, 1000, -7], dtype=np.int32)
    tht = torch.from_numpy(np.ascontiguousarray(th)).cuda()
    stt = torch.from_numpy(star).cuda()
    good = np.flatnonzero(~bad)
    ref = eng.lnlike_batch(tht[good], stt[good]).cpu().numpy()
    assert eng.query('status') == 0
    lnl = eng.lnlike_batch(tht, stt).cpu().numpy()
    assert np.isnan(lnl[bad]).all()
    assert np.array_equal(lnl[good], ref, equal_nan=True)
    assert eng.query('status') & 4
    # model_batch: no flux or magnitudes row for an invalid star (sentinel survives), the rest bit-identical
    n = eng.n_obs
    flux = torch.full((B, max(n, 1)), 7.0, dtype=torch.float64, device='cuda')
    mags = torch.full((B, max(eng.nb, 1)), 7.0, dtype=torch.float64, device='cuda')
    lm = torch.empty(B, dtype=torch.float64, device='cuda')
    st = torch.cuda.current_stream().cuda_stream
    rc = lib.payne_model_batch_stars(eng._ctx, tht.data_ptr(), stt.data_ptr(), B, th.shape[1],
                                     flux.data_ptr() if n else None, max(n, 1),
                                     mags.data_ptr() if eng.nb else None, lm.data_ptr(), st)
    assert rc == 0
    torch.cuda.synchronize()
    lm = lm.cpu().numpy()
    assert np.isnan(lm[bad]).all() and np.array_equal(lm[good], ref, equal_nan=True)
    if n:
        assert (flux.cpu().numpy()[bad] == 7.0).all()
    if eng.nb:
        assert (mags.cpu().numpy()[bad] == 7.0).all()
        assert np.isfinite(mags.cpu().numpy()[good]).all()
    # host entry: refused before anything is launched or written
    out = np.full(B, 7.0)
    rc = lib.payne_lnlike_batch_stars_host(eng._ctx, np.ascontiguousarray(th).ctypes.data, star.ctypes.data, B,
                                           th.shape[1], out.ctypes.data)
    assert rc == _INVALID and b'outside' in lib.payne_last_error()
    assert (out == 7.0).all()
    with pytest.raises(_lib.PayneError):
        eng.lnlike_batch(th, star)
    # no star array on several stars: refused, naming the entry that takes one
    with pytest.raises(_lib.PayneError, match='payne_lnlike_batch_stars'):
        eng.lnlike_batch(tht)
    with pytest.raises(_lib.PayneError, match='payne_lnlike_batch_stars_host'):
        eng.lnlike_batch(th)
    with pytest.raises(_lib.PayneError, match='payne_model_batch_stars'):
        eng.model_batch(tht)
    eng.close()


_INVALID, _UNSUPPORTED = -1, -4


def test_lsf_and_gather_refused_on_several_stars_continuum_kept():
    lib = _lib.load()
    kw, stars, fit, box, _ = _build('fast12', n_stars=2)
    eng = Engine(stars=stars, **kw)
    lsf = np.full(len(stars[0]['wave']), 0.05)
    assert lib.payne_ctx_set_lsf(eng._ctx, lsf.ctypes.data, len(lsf)) == _UNSUPPORTED
    assert b'LSF' in lib.payne_last_error()
    handles = ctypes.create_string_buffer(_lib.GATHER_HANDLE_BYTES)
    assert lib.payne_gather_create(eng._ctx, 1, 0, 16, handles) == _UNSUPPORTED
    # the continuum multiply does not touch the observation: attached to a context of several stars it gives, for
    # every star, what it gives on a single-star context
    cont = _spec('mini')
    eng.attach_continuum(cont)
    th = _thetas(fit, box, 200, seed=9)
    star = (np.arange(200) % 2).astype(np.int32)
    lnl = eng.lnlike_batch(th, star)
    for k in range(2):
        one = Engine(obs_wave=stars[k]['wave'], obs_flux=stars[k]['flux'], obs_eflux=stars[k]['eflux'], **kw)
        one.attach_continuum(cont)
        ref = one.lnlike_batch(th[star == k])
        assert np.array_equal(lnl[star == k], ref, equal_nan=True)
        one.close()
    eng.close()


def _fit_inputdict(cfg, wave_sel, seed, out, maxiter):
    return {
        'spec': {'obs_wave': cfg.obs_wave[wave_sel], 'obs_flux': cfg.obs_flux[wave_sel],
                 'obs_eflux': cfg.obs_eflux[wave_sel], 'convertair': False, 'modpoly': False},
        'specANNpath': cfg.spec, 'NNtype': 'LinNet',
        'sampler': {'samplertype': 'Static', 'samplemethod': 'rwalk', 'npoints': 32, 'walks': 10,
                    'delta_logz_final': 0.5, 'flushnum': 10, 'seed': seed, 'maxiter': maxiter},
        'priordict': {p: {'pv_uniform': list(cfg.box[p])} for p in cfg.fitpars_i},
        'output': out,
    }


def test_fitpaynemany_matches_separate_fits(tmp_path):
    from conftest import load_case
    from thepayne_b200.fitting.fitstar import FitPayne
    from thepayne_b200.fitting.multistar import FitPayneMany
    cfg, _ = load_case('mini_spec')
    n = len(cfg.obs_wave)
    sels = [slice(0, n), slice(n // 5, n - n // 7), slice(0, n // 2)]
    maxiters = [120, 60, 90]                                      # the samplers finish at different times
    single, calls = [], []
    for k, sel in enumerate(sels):
        d = _fit_inputdict(cfg, sel, 100 + k, str(tmp_path / ('one%d.dat' % k)), maxiters[k])
        s = FitPayne().run(inputdict=d, verbose=False)
        calls.append(len(s.batch_sizes))
        single.append(open(d['output'], 'rb').read())
    many = FitPayneMany()
    dicts = [_fit_inputdict(cfg, sel, 100 + k, str(tmp_path / ('many%d.dat' % k)), maxiters[k])
             for k, sel in enumerate(sels)]
    samplers = many.run(inputdicts=dicts, verbose=False)
    for k in range(3):
        assert open(dicts[k]['output'], 'rb').read() == single[k], k
        assert len(samplers[k].batch_sizes) == calls[k]
    assert many.batcher.ncalls == max(calls) == many.likeobj.ncalls
    assert len(set(calls)) > 1
    assert sum(many.batcher.batch_sizes) == sum(sum(s.batch_sizes) for s in samplers)


def test_starset_view_works_with_the_batched_nested_sampler():
    """StarSetLikelihood.star(k) in BatchedLnProb / BatchedNestedSampler: the same run as on star k's own
    likelihood object."""
    from conftest import load_case
    from thepayne_b200.fitting.batching import BatchedLnProb
    from thepayne_b200.fitting.likelihood import likelihood
    from thepayne_b200.fitting.multistar import StarSetLikelihood
    from thepayne_b200.fitting.nested import BatchedNestedSampler
    from thepayne_b200.fitting.prior import prior
    cfg, _ = load_case('mini_spec')
    names = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Vmic', 'Inst_R', 'log(R)', 'Dist', 'log(A)',
             'Av', 'Rv', 'CarbonScale']
    flags = {nm: nm in cfg.fitpars_i for nm in names}
    n = len(cfg.obs_wave)
    fas = [{'obs_wave_fit': cfg.obs_wave[a:b], 'obs_flux_fit': cfg.obs_flux[a:b], 'obs_eflux_fit': cfg.obs_eflux[a:b],
            'specANNpath': cfg.spec, 'NNtype': 'LinNet', 'fixedpars': {}} for a, b in [(0, n), (n // 3, n)]]
    pri = {p: {'pv_uniform': list(cfg.box[p])} for p in cfg.fitpars_i}
    S = StarSetLikelihood(fas, [names, flags], cfg.runbools)
    for k in range(2):
        P = prior(fas[k], pri, [names, flags], cfg.runbools)
        runs = []
        for L in (S.star(k), likelihood(fas[k], [names, flags], cfg.runbools, verbose=False)):
            smp = BatchedNestedSampler(BatchedLnProb(L, P).batch, P.priortrans_batch, L.ndim, nlive=24, walks=5, seed=3)
            for _ in smp.sample(dlogz=0.5, maxiter=40):
                pass
            runs.append(smp.results['logl'])
            assert L.fitpars_i == cfg.fitpars_i and L.ndim == len(cfg.fitpars_i)
        assert np.array_equal(runs[0], runs[1])
        v = S.star(k)
        assert v.lnlikefn(list(cfg.theta_true)) == float(v.lnlike_batch(cfg.theta_true[None, :])[0])
        assert v.parsdict['Teff'] == cfg.theta_true[0]
    bad = dict(fas[1], NNtype='SMLP')
    with pytest.raises(ValueError, match='star 1: NNtype'):
        StarSetLikelihood([fas[0], bad], [names, flags], cfg.runbools)
    bad = dict(fas[1], fixedpars={'Vmic': 1.0})
    with pytest.raises(ValueError, match='star 1: fixedpars'):
        StarSetLikelihood([fas[0], bad], [names, flags], cfg.runbools)
