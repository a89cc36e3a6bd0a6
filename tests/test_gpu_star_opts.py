"""Per-star options of an observation set (payne_ctx_create_stars_opts): each star's own fixed parameter values,
photometric bands and LSF vector, and a fixed LSF vector ``Inst_R`` through the likelihood interfaces.

The core check is bit-identity, as for observation sets without options: every star's rows of an interleaved batch
(with a run of one star's rows across a slab boundary) give exactly (np.array_equal, NaN patterns included) what a
single-star engine gives that holds the star's values as its shared ``fixedpars``, a photometry net made of the
same per-band weights in the star's band order, and the star's LSF through ``set_lsf``.  Then the oracle, the
refusals, contexts without options, and FitPayneMany against separate FitPayne runs.
"""
import ctypes
import types

import numpy as np
import pytest
import torch

from thepayne_b200 import _lib, synth
from thepayne_b200.engine import Engine, _specnet_struct

pytestmark = pytest.mark.gpu

BANDS = synth.PROCYON_BANDS[:4]
RANGES = {'mini': (5140.0, 5190.0),       # 3403 pixels -> 4096-sample transforms
          'c2': (5130.0, 5340.0),         # 16384
          'mid': (5000.0, 5280.0),        # 32768
          'wide': (4800.0, 5300.0)}       # 65536
_SPEC_CACHE = {}
_INVALID, _UNSUPPORTED = -1, -4


def _spec(rng_name, d_in=4):
    key = (rng_name, d_in)
    if key not in _SPEC_CACHE:
        wave, rsig = synth.ann_wavegrid(*RANGES[rng_name], 50000.0)
        _SPEC_CACHE[key] = synth.make_specnet(d_in, 64, wave, rsig, seed=0)
    return _SPEC_CACHE[key]


def _subnet(net, bands):
    """The photometry net of ``bands`` (in that order) made of ``net``'s per-band weights."""
    idx = [net.bands.index(b) for b in bands]
    return synth.PhotNet(list(bands), net.w1[idx], net.b1[idx], net.w2[idx], net.b2[idx], net.w3[idx], net.b3[idx],
                         net.xmin, net.xmax, net.hiav[idx])


# one band; all bands in another order; two disjoint pairs; the net's order; a pair
STAR_BANDS = [[BANDS[2]], [BANDS[3], BANDS[1], BANDS[0], BANDS[2]], [BANDS[0], BANDS[1]], [BANDS[2], BANDS[3]],
              None, [BANDS[3], BANDS[1]]]


def _stars(spec, with_bands, seed=5):
    """Six observations: different ranges and sizes, one unsorted, one partly beyond the emulator's coverage."""
    w = spec.wavelength
    a, b = w[0], w[-1]
    span = b - a
    rng = np.random.default_rng(seed)
    grids = [
        np.linspace(a + 0.10 * span, b - 0.10 * span, 1500),
        np.linspace(a + 0.25 * span, b - 0.05 * span, 2311),
        rng.permutation(np.linspace(a + 0.15 * span, b - 0.20 * span, 977)),          # unsorted
        np.linspace(a - 0.02 * span, b - 0.30 * span, 1201),                          # beyond the coverage
        np.linspace(a + 0.50 * span, a + 0.53 * span, 257),                           # narrow mask
        np.linspace(a + 0.05 * span, b - 0.05 * span, 3050),
    ]
    out = []
    for k, g in enumerate(grids):
        flux = 1.0 + 0.05 * rng.standard_normal(len(g))
        eflux = 0.02 + 0.01 * rng.random(len(g))
        st = {'wave': g, 'flux': flux, 'eflux': eflux}
        if with_bands:
            bands = STAR_BANDS[k] if STAR_BANDS[k] is not None else BANDS
            st['phot'] = {bd: (float(5.0 + k + 0.1 * BANDS.index(bd)), 0.05 + 0.01 * k) for bd in bands}
            if STAR_BANDS[k] is not None:
                st['bands'] = list(STAR_BANDS[k])
        out.append(st)
    return out


def _lsf(wave, k):
    return 0.035 + 0.004 * k + 0.01 * (wave - wave.min()) / (wave.max() - wave.min()) + 0.003 * np.sin(wave / 2.0)


# per-star fixed values, one list entry per star
FIXED = {
    'Inst_R': [32000.0, 0.0, float('nan'), 45000.0, 28000.0, 60000.0],
    'Vrot': [0.0, 3.0, 12.0, 1.5, 0.0, 25.0],
    'Vrad': [-20.0, 0.0, 35.0, 4.0, 80.0, -3.0],
    'log(g)': [4.0, 4.5, 3.9, 4.2, 4.4, 4.1],
    'Vmic': [0.8, 1.0, 2.5, 1.2, 1.9, 0.6],
    'Dist': [10.0, 150.0, 35.0, 5.0, 80.0, 420.0],
    'Av': [0.1, 0.0, 0.8, 0.35, 0.6, 0.05],
}

SETUPS = {
    # name: (emulator, D_in, npoly, phot mode (None / 'scaled' / 'dist'), fixed names, lsf, precision, settings)
    'fast_instr_vrot': ('mini', 4, 0, None, ['Inst_R', 'Vrot'], False, 'parity', {'max_batch': 200}),
    'fast_poly_vrad': ('mini', 4, 3, None, ['Vrad', 'Inst_R'], False, 'parity', {'max_batch': 200}),
    'fast14_logg': ('c2', 4, 2, None, ['log(g)', 'Inst_R'], False, 'parity', {'max_batch': 200}),
    'cluster_instr': ('mid', 4, 0, None, ['Inst_R', 'Vrot'], False, 'parity', {'tail_cluster': 1, 'max_batch': 200}),
    'general_vmic': ('mini', 5, 2, None, ['Vmic', 'Inst_R'], False, 'parity', {'fast_tail': 0, 'max_batch': 200}),
    'simt_logg': ('mini', 4, 2, None, ['log(g)', 'Vrot', 'Inst_R'], False, 'simt', {'max_batch': 200}),
    'phot_only_dist': (None, 4, 0, 'dist', ['Dist', 'Av'], False, 'parity', {'max_batch': 200}),
    'joint_dist': ('mini', 4, 2, 'dist', ['Dist', 'Inst_R'], False, 'parity', {'max_batch': 200}),
    'joint_scaled': ('mini', 4, 0, 'scaled', ['log(g)', 'Vrot', 'Inst_R'], False, 'parity', {'max_batch': 200}),
    'lsf_rot': ('mini', 4, 2, None, ['Vrad'], True, 'parity', {'max_batch': 200}),
    'lsf_norot_cont': ('mini', 4, 0, None, ['Vrot'], True, 'parity', {'max_batch': 200, 'continuum': 1}),
    'lsf_joint': ('mini', 4, 0, 'scaled', ['log(g)'], True, 'parity', {'max_batch': 200}),
}


def _build(name):
    emu, d_in, npoly, pmode, fixed, lsf, prec, settings = SETUPS[name]
    spec = _spec(emu or 'mini', d_in)
    phot = synth.make_photnet(BANDS, H=16) if pmode else None
    fit = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]']
    if d_in == 5:
        fit.append('Vmic')
    if emu:
        fit += ['Vrad', 'Vrot', 'Inst_R']
    if pmode == 'scaled':
        fit += ['log(A)', 'Av']
    elif pmode == 'dist':
        fit += ['log(R)', 'Dist', 'Av']
    fit += ['pc_%d' % k for k in range(npoly)]
    fit = [p for p in fit if p not in fixed and not (lsf and p == 'Inst_R')]
    box = dict(synth._BOX)
    for k in range(npoly):
        box['pc_%d' % k] = (0.75, 1.25) if k == 0 else (-0.1, 0.1)
    runbools = [emu is not None, pmode is not None, npoly > 0, pmode == 'scaled', False]
    stars = _stars(spec, pmode is not None)
    for k, st in enumerate(stars):
        st['fixedpars'] = {p: FIXED[p][k] for p in fixed}
        if lsf:
            st['fixedpars']['Inst_R'] = _lsf(st['wave'], k)
    kw = dict(spec=spec if emu else None, phot=phot, fitpars_i=fit, runbools=runbools, precision=prec)
    return kw, stars, fit, box, settings


def _apply(eng, settings):
    for k, v in settings.items():
        if k == 'continuum':
            eng.attach_continuum(_spec('mini'))
        else:
            eng.set(k, v)


def _thetas(fit, box, B, seed):
    rng = np.random.default_rng(seed)
    lo = np.array([box[p][0] for p in fit])
    hi = np.array([box[p][1] for p in fit])
    th = lo + (hi - lo) * rng.random((B, len(fit)))
    if 'Inst_R' in fit:
        th[rng.random(B) < 0.1, fit.index('Inst_R')] = 0.0
    if 'Vrot' in fit:
        th[rng.random(B) < 0.1, fit.index('Vrot')] = 0.0
    return th


def _single(kw, st):
    """The single-star engine of star ``st``: its values as the shared fixedpars, its bands' net, set_lsf."""
    fx = dict(st['fixedpars'])
    lsf = fx.pop('Inst_R') if np.ndim(fx.get('Inst_R', 0.0)) == 1 else None
    kws = dict(kw, fixedpars=fx)
    obs_phot = None
    if kw['phot'] is not None:
        bands = st.get('bands') or [b for b in kw['phot'].bands if b in st['phot']]
        kws['phot'] = _subnet(kw['phot'], bands)
        obs_phot = {b: st['phot'][b] for b in bands}
    spec_on = kw['spec'] is not None
    one = Engine(obs_wave=st['wave'] if spec_on else None, obs_flux=st['flux'] if spec_on else None,
                 obs_eflux=st['eflux'] if spec_on else None, obs_phot=obs_phot, **kws)
    if lsf is not None:
        one.set_lsf(lsf)
    return one


@pytest.mark.parametrize('name', list(SETUPS))
def test_star_options_bit_identical_to_single_star_engines(name):
    kw, stars, fit, box, settings = _build(name)
    S = len(stars)
    multi = Engine(stars=stars, fixedpars={}, **kw)
    _apply(multi, settings)
    lsf_on = SETUPS[name][5]
    assert multi.query('n_stars') == S and multi.query('lsf') == int(lsf_on)
    if name.startswith('cluster'):
        assert multi.query('tail_cluster') == 1
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
        one = _single(kw, stars[k])
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
            assert np.isnan(flux[idx, n:]).all()
        if mags is not None:
            nbk = len(multi.star_bands[k])
            assert multi.star_bands[k] == one.bands
            assert np.array_equal(mags[idx, :nbk], rm.cpu().numpy(), equal_nan=True), (name, k)
            assert np.isnan(mags[idx, nbk:]).all()                      # columns beyond the star's bands
        n_finite += int(np.isfinite(ref_d).sum())
        one.close()
    assert n_finite > B // 4
    multi.close()


def test_per_star_values_change_the_result():
    """The per-star values are really read: the same rows give other lnL on stars with other fixed values."""
    kw, stars, fit, box, _ = _build('fast_instr_vrot')
    same = [dict(st, fixedpars={'Inst_R': 32000.0, 'Vrot': 3.0}) for st in stars[:2]]
    diff = [dict(st) for st in stars[:2]]
    th = _thetas(fit, box, 64, seed=2)
    star = (np.arange(64) % 2).astype(np.int32)
    a = Engine(stars=same, **kw).lnlike_batch(th, star)
    b = Engine(stars=diff, **kw).lnlike_batch(th, star)
    ref = Engine(stars=[{k: v for k, v in st.items() if k != 'fixedpars'} for st in same],
                 fixedpars={'Inst_R': 32000.0, 'Vrot': 3.0}, **kw).lnlike_batch(th, star)
    assert np.array_equal(a, ref)
    assert np.isfinite(a).all() and not np.array_equal(a, b)


# ------------------------------------------------------------------ oracle

def test_likelihood_with_lsf_vector_vs_oracle():
    """likelihood(fixedpars={'Inst_R': lsf}) -- lnlikefn, lnlike_batch, lnlike(specpars) and GenMod.genspec --
    against OracleLikelihood, with the bars of the LSF tail in test_gpu_f3.py."""
    from oracle import goldens, payne_oracle as O
    from thepayne_b200.fitting.likelihood import likelihood
    spec, _, calls = goldens.getspec_case()
    outwave, lsf = calls[3]['outwave'], calls[3]['inst_R']
    rng = np.random.default_rng(4)
    oflux = 1.0 + 0.03 * rng.standard_normal(len(outwave))
    oeflux = 0.02 + 0.005 * rng.random(len(outwave))
    names = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Vmic', 'Inst_R', 'log(R)', 'Dist', 'log(A)',
             'Av', 'Rv', 'CarbonScale']
    free = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot']
    fa = {'obs_wave_fit': outwave, 'obs_flux_fit': oflux, 'obs_eflux_fit': oeflux, 'specANNpath': spec,
          'NNtype': 'LinNet', 'fixedpars': {'Inst_R': lsf}}
    runbools = [True, False, False, False, False]
    L = likelihood(fa, [names, {n: n in free for n in names}], runbools, verbose=False)
    cfg = types.SimpleNamespace(spec=spec, phot=None, runbools=runbools, fitpars_i=free, fixedpars={'Inst_R': lsf},
                                obs_wave=outwave, obs_flux=oflux, obs_eflux=oeflux)
    OL = O.OracleLikelihood(cfg)
    th = np.array([[5770.0, 4.44, 0.0, 0.0, 0.5, 3.0], [4600.0, 4.7, -0.08, 0.05, -25.0, 0.0],
                   [6300.0, 4.1, 0.05, -0.02, 60.0, 14.0], [5200.0, 4.6, -0.03, 0.04, 0.0, 1.2]])
    lo, fo, _ = OL.lnlike_batch(th, return_model=True)
    flux, _, lm = L.engine.model_batch(th, want_mags=False)
    flux = flux.cpu().numpy()
    assert np.array_equal(np.isnan(flux), np.isnan(fo))
    assert np.nanmax(np.abs(flux - fo) / np.abs(fo)) <= 5e-7
    lb = L.lnlike_batch(th)
    assert np.all(np.abs(lb - lo) <= np.maximum(1e-3, 1e-5 * np.abs(lo))), (lb, lo)
    assert np.array_equal(lb, lm.cpu().numpy())
    for i in range(len(th)):
        assert L.lnlikefn(list(th[i])) == lb[i]
        assert L.parsdict['Inst_R'] is lsf
        sp = list(th[i][:4]) + [th[i][4], th[i][5], np.nan, lsf]
        assert L.lnlike(specpars=sp) == lb[i]
    from thepayne_b200.fitting.genmod import GenMod
    G = GenMod()
    G._initspecnn(nnpath=spec, NNtype='LinNet')
    for i in range(len(th)):
        pars = list(th[i][:4]) + [th[i][4], th[i][5], np.nan, lsf]
        w, f = G.genspec(pars, outwave=outwave)
        assert np.array_equal(w, outwave) and np.array_equal(f, flux[i], equal_nan=True)
    with pytest.raises(ValueError):
        G.genspec(list(th[0][:6]) + [np.nan, lsf], outwave=None)


def test_band_subset_vs_oracle():
    """A star with a band subset in its own order against the oracle with that star's net."""
    from oracle import payne_oracle as O
    net = synth.make_photnet(synth.PROCYON_BANDS, H=32)
    bands = ['2MASS_J', 'Bessell_V', 'Bessell_I']
    obs_phot = {b: (6.0 + 0.2 * i, 0.03 + 0.01 * i) for i, b in enumerate(bands)}
    full = {b: (7.0, 0.05) for b in synth.PROCYON_BANDS}
    fit = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'log(R)', 'Dist', 'Av']
    kw = dict(phot=net, fitpars_i=fit, runbools=[False, True, False, False, False])
    eng = Engine(stars=[{'phot': full}, {'phot': obs_phot, 'bands': bands}], **kw)
    rng = np.random.default_rng(8)
    lo = np.array([synth._BOX[p][0] for p in fit])
    hi = np.array([synth._BOX[p][1] for p in fit])
    th = lo + (hi - lo) * rng.random((40, len(fit)))
    th[:5, fit.index('Av')] = 6.0                                     # the high-Av extension
    lnl = eng.lnlike_batch(th, np.ones(40, dtype=np.int32))
    _, mags, _ = eng.model_batch(th, np.ones(40, dtype=np.int32))
    cfg = types.SimpleNamespace(spec=None, phot=_subnet(net, bands), runbools=[False, True, False, False, False],
                                fitpars_i=fit, fixedpars={}, obs_phot=obs_phot)
    lo_, _, mo = O.OracleLikelihood(cfg).lnlike_batch(th, return_model=True)
    m = mags.cpu().numpy()
    assert np.isnan(m[:, 3:]).all()
    ok = np.isfinite(mo)
    assert np.array_equal(ok, np.isfinite(m[:, :3]))
    assert np.allclose(m[:, :3][ok], mo[ok], rtol=1e-12, atol=1e-12)
    fin = np.isfinite(lo_)
    assert fin.sum() >= 30 and np.array_equal(fin, np.isfinite(lnl))
    assert np.allclose(lnl[fin], lo_[fin], rtol=1e-10, atol=1e-9)


# ------------------------------------------------------------------ refusals and defaults

def _raw_create(spec, phot, stars, opts, fit, runbools, fixed=None):
    """payne_ctx_create_stars_opts (opts: list of dicts or None; 'none' = the NULL-opts call of create_stars)."""
    lib = _lib.load()
    keep = []
    sp = _specnet_struct(spec, keep) if spec is not None else None
    ph = None
    if phot is not None:
        ph = _lib.PaynePhotNet()
        arrs = [np.ascontiguousarray(a, dtype=np.float32) for a in
                (phot.w1, phot.b1, phot.w2, phot.b2, np.asarray(phot.w3).reshape(len(phot.bands), -1),
                 np.asarray(phot.b3).reshape(-1))]
        keep += arrs
        ph.nb, ph.H = arrs[0].shape[0], arrs[0].shape[1]
        ph.w1, ph.b1, ph.w2, ph.b2, ph.w3, ph.b3 = [a.ctypes.data_as(ctypes.POINTER(ctypes.c_float)) for a in arrs]
        d = [np.ascontiguousarray(a, dtype=np.float64) for a in (phot.xmin, phot.xmax, phot.hiav)]
        keep += d
        ph.xmin, ph.xmax, ph.hiav = [a.ctypes.data_as(ctypes.POINTER(ctypes.c_double)) for a in d]
    lay = _lib.PayneLayout()
    lay.ndim = len(fit)
    for nm, k in _lib.PAR_INDEX.items():
        lay.col[k] = fit.index(nm) if nm in fit else -1
        lay.fixed[k] = (fixed or {}).get(nm, float('nan'))
    pcs = [i for i, p in enumerate(fit) if 'pc' in p]
    lay.n_poly = len(pcs)
    for i, c in enumerate(pcs):
        lay.poly_col[i] = c
    lay.spec_bool, lay.phot_bool, lay.modpoly_bool, lay.photscale_bool = [int(bool(b)) for b in runbools[:4]]
    S = len(stars)
    obs = (_lib.PayneObs * S)()
    dp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))        # noqa: E731
    for k, st in enumerate(stars):
        if spec is not None:
            ow, of, oe = [np.ascontiguousarray(st[x], dtype=np.float64) for x in ('wave', 'flux', 'eflux')]
            keep += [ow, of, oe]
            obs[k].n_obs, obs[k].wave, obs[k].flux, obs[k].eflux = len(ow), dp(ow), dp(of), dp(oe)
        if phot is not None:
            mag = np.ascontiguousarray(st['mag'], dtype=np.float64)
            err = np.full(len(mag), 0.05)
            keep += [mag, err]
            obs[k].nb, obs[k].phot_mag, obs[k].phot_err = len(mag), dp(mag), dp(err)
    ctx = ctypes.c_void_p()
    if opts == 'none':
        rc = lib.payne_ctx_create_stars(ctypes.byref(sp) if sp else None, ctypes.byref(ph) if ph else None, obs, S,
                                        ctypes.byref(lay), 0, ctypes.byref(ctx))
        return rc, ctx
    o = None
    if opts is not None:
        o = (_lib.PayneStarOpts * S)()
        for k, d in enumerate(opts):
            if d.get('band') is not None:
                b = np.ascontiguousarray(d['band'], dtype=np.int32)
                keep.append(b)
                o[k].band = b.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
            if d.get('lsf') is not None:
                v = np.ascontiguousarray(d['lsf'], dtype=np.float64)
                keep.append(v)
                o[k].lsf = dp(v)
            if d.get('fixed') is not None:
                v = np.ascontiguousarray(d['fixed'], dtype=np.float64)
                keep.append(v)
                o[k].fixed = dp(v)
    rc = lib.payne_ctx_create_stars_opts(ctypes.byref(sp) if sp else None, ctypes.byref(ph) if ph else None, obs, o,
                                         S, ctypes.byref(lay), 0, ctypes.byref(ctx))
    return rc, ctx


def test_refusals():
    lib = _lib.load()
    spec = _spec('mini')
    net = synth.make_photnet(BANDS, H=16)
    stars = _stars(spec, False)[:2]
    fit = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot']
    rb = [True, False, False, False, False]
    lsfs = [_lsf(s['wave'], k) for k, s in enumerate(stars)]
    # a mix of LSF and scalar-R stars
    rc, _ = _raw_create(spec, None, stars, [{'lsf': lsfs[0]}, {}], fit, rb)
    assert rc == _UNSUPPORTED and b'LSF' in lib.payne_last_error()
    with pytest.raises(_lib.PayneError, match='-4'):
        Engine(stars=[dict(stars[0], fixedpars={'Inst_R': lsfs[0]}), stars[1]], spec=spec, fitpars_i=fit)
    # LSF length (checked by the engine: the C ABI takes n_obs values) and sign
    with pytest.raises(ValueError, match='one dispersion per observed pixel'):
        Engine(stars=[dict(stars[0], fixedpars={'Inst_R': lsfs[0][:-1]})], spec=spec, fitpars_i=fit)
    bad = lsfs[1].copy()
    bad[7] = -0.01
    rc, _ = _raw_create(spec, None, stars, [{'lsf': lsfs[0]}, {'lsf': bad}], fit, rb)
    assert rc == _INVALID and b'positive' in lib.payne_last_error()
    bad[7] = np.nan
    rc, _ = _raw_create(spec, None, stars, [{'lsf': lsfs[0]}, {'lsf': bad}], fit, rb)
    assert rc == _INVALID
    # LSF on a 65536-pixel emulator grid
    wide = _spec('wide')
    wst = _stars(wide, False)[:2]
    rc, _ = _raw_create(wide, None, wst, [{'lsf': _lsf(s['wave'], k)} for k, s in enumerate(wst)], fit, rb)
    assert rc == _UNSUPPORTED and b'32768' in lib.payne_last_error()
    # bad band lists
    pfit = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'log(A)', 'Av']
    prb = [False, True, False, True, False]
    two = [{'mag': [5.0, 6.0]}, {'mag': [5.0, 6.0, 7.0, 8.0]}]
    rc, ctx = _raw_create(None, net, two, [{'band': [2, 0]}, {}], pfit, prb)
    assert rc == 0
    lib.payne_ctx_destroy(ctx)
    for band, what in [([4, 0], b'outside'), ([-1, 0], b'outside'), ([1, 1], b'twice')]:
        rc, _ = _raw_create(None, net, two, [{'band': band}, {}], pfit, prb)
        assert rc == _INVALID and what in lib.payne_last_error(), band
    five = [{'mag': [5.0, 6.0, 7.0, 8.0, 9.0]}, two[1]]
    rc, _ = _raw_create(None, net, five, [{'band': [0, 1, 2, 3, 0]}, {}], pfit, prb)
    assert rc == _INVALID and b'magnitudes' in lib.payne_last_error()
    rc, _ = _raw_create(None, net, two, [{}, {}], pfit, prb)        # no band list: nb must be the net's
    assert rc == _INVALID and b'nb' in lib.payne_last_error()
    with pytest.raises(ValueError, match='not in the photometry net'):
        Engine(stars=[{'phot': {'Gaia_G': (5.0, 0.1)}}], phot=net, fitpars_i=pfit, runbools=prb)
    # unchanged: set_lsf still refuses several stars, also on a context made with LSF vectors
    eng = Engine(stars=[dict(s, fixedpars={'Inst_R': v}) for s, v in zip(stars, lsfs)], spec=spec, fitpars_i=fit)
    assert eng.query('lsf') == 1
    assert lib.payne_ctx_set_lsf(eng._ctx, lsfs[0].ctypes.data, len(lsfs[0])) == _UNSUPPORTED
    eng.close()


def test_contexts_without_options_unchanged():
    """NULL opts and opts whose fields are all NULL give exactly what payne_ctx_create_stars gives (joint fit,
    polynomial, fixed values in the layout)."""
    lib = _lib.load()
    spec = _spec('mini')
    net = synth.make_photnet(BANDS, H=16)
    stars = _stars(spec, False)
    for k, st in enumerate(stars):
        st['mag'] = [5.0 + k + 0.1 * i for i in range(len(BANDS))]
    fit = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'log(A)', 'Av', 'pc_0', 'pc_1']
    rb = [True, True, True, True, False]
    box = dict(synth._BOX, pc_0=(0.75, 1.25), pc_1=(-0.1, 0.1))
    th = np.ascontiguousarray(_thetas(fit, box, 300, seed=6))
    star = (np.arange(300) % len(stars)).astype(np.int32)
    outs = []
    for opts in ('none', None, [{}] * len(stars)):
        rc, ctx = _raw_create(spec, net, stars, opts, fit, rb, fixed={'Inst_R': 33000.0})
        assert rc == 0, lib.payne_last_error()
        out = np.empty(300)
        assert lib.payne_lnlike_batch_stars_host(ctx, th.ctypes.data, star.ctypes.data, 300, len(fit),
                                                 out.ctypes.data) == 0
        lib.payne_ctx_destroy(ctx)
        outs.append(out)
    assert np.isfinite(outs[0]).sum() > 100
    assert np.array_equal(outs[0], outs[1], equal_nan=True) and np.array_equal(outs[0], outs[2], equal_nan=True)


# ------------------------------------------------------------------ FitPayneMany

def _run_many(tmp_path, dicts):
    from thepayne_b200.fitting.fitstar import FitPayne
    from thepayne_b200.fitting.multistar import FitPayneMany
    single, calls = [], []
    for k, d in enumerate(dicts):
        d1 = dict(d, output=str(tmp_path / ('one%d.dat' % k)))
        s = FitPayne().run(inputdict=d1, verbose=False)
        calls.append(len(s.batch_sizes))
        single.append(open(d1['output'], 'rb').read())
    many = FitPayneMany()
    dm = [dict(d, output=str(tmp_path / ('many%d.dat' % k))) for k, d in enumerate(dicts)]
    samplers = many.run(inputdicts=dm, verbose=False)
    for k in range(len(dicts)):
        assert open(dm[k]['output'], 'rb').read() == single[k], k
        assert len(samplers[k].batch_sizes) == calls[k]
    assert many.batcher.ncalls == max(calls) == many.likeobj.ncalls
    return many


def _sampler(seed, maxiter):
    return {'samplertype': 'Static', 'samplemethod': 'rwalk', 'npoints': 32, 'walks': 10, 'delta_logz_final': 0.5,
            'flushnum': 10, 'seed': seed, 'maxiter': maxiter}


def test_fitpaynemany_fixed_inst_r_and_band_subsets(tmp_path):
    from conftest import load_case
    cfg, _ = load_case('mini_joint')
    n = len(cfg.obs_wave)
    sels = [slice(0, n), slice(n // 5, n - n // 7), slice(0, n // 2)]
    bands = [list(cfg.obs_phot), ['2MASS_J', 'Bessell_V'], ['Bessell_I', 'Bessell_B', '2MASS_Ks']]
    inst = [32000.0, 28000.0, 36000.0]
    free = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'log(A)', 'Av']
    dicts = []
    for k in range(3):
        pri = {p: {'pv_uniform': list(cfg.box[p])} for p in free}
        pri['Inst_R'] = {'fixed': inst[k]}
        dicts.append({'spec': {'obs_wave': cfg.obs_wave[sels[k]], 'obs_flux': cfg.obs_flux[sels[k]],
                               'obs_eflux': cfg.obs_eflux[sels[k]], 'convertair': False, 'modpoly': False},
                      'phot': {b: cfg.obs_phot[b] for b in bands[k]}, 'photscale': True,
                      'specANNpath': cfg.spec, 'photANNpath': cfg.phot, 'NNtype': 'LinNet',
                      'sampler': _sampler(200 + k, [60, 40, 50][k]), 'priordict': pri})
    many = _run_many(tmp_path, dicts)
    assert many.likeobj.bands == list(cfg.obs_phot)
    assert [many.fits[k].likeobj.fixedpars['Inst_R'] for k in range(3)] == inst


def test_fitpaynemany_lsf_vectors(tmp_path):
    """Three stars with their own LSF vectors (FitPayne with priordict['Inst_R']['fixed'] = lsf runs to the end,
    and FitPayneMany gives each star's file byte for byte)."""
    from conftest import load_case
    cfg, _ = load_case('mini_spec')
    n = len(cfg.obs_wave)
    sels = [slice(0, n), slice(n // 5, n - n // 7), slice(0, n // 2)]
    free = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot']
    dicts = []
    for k in range(3):
        w = cfg.obs_wave[sels[k]]
        pri = {p: {'pv_uniform': list(cfg.box[p])} for p in free}
        pri['Inst_R'] = {'fixed': _lsf(w, k)}
        dicts.append({'spec': {'obs_wave': w, 'obs_flux': cfg.obs_flux[sels[k]], 'obs_eflux': cfg.obs_eflux[sels[k]],
                               'convertair': False, 'modpoly': False},
                      'specANNpath': cfg.spec, 'NNtype': 'LinNet', 'sampler': _sampler(300 + k, [40, 25, 30][k]),
                      'priordict': pri})
    many = _run_many(tmp_path, dicts)
    assert many.likeobj.engine.query('lsf') == 1
