"""The photometry kernel (phot.cuh) against the oracle's sed / genphot, float64 both, at the shapes and values where
it branches.

phot_kernel evaluates kPhotTile = 8 points per CTA against every band, its two hidden layers in 128 H bytes of dynamic
shared memory (plus 64 nb bytes with band lists): above H = 384 that needs the opt-in beyond 48 KB, and H = 1600
without band lists is exactly the 200 KB the context accepts.  It branches on Av (the high-Av extension from Av = 5 on,
predictsed.py:86), on the distance / photscale mode, and with band lists (the SLOTS form) skips a band no point of the
tile has.

CASES is the matrix as plain data; `test_matrix_covers_every_branch` (no GPU) checks what it reaches.  Every case runs
photometry-only (lnl_from_sed_kernel) and, where `spec` is set, with a spectrum too (the tail adds chi2_sed).  Rows:
Av at nextafter(5, -inf), 5 and nextafter(5, +inf), NaN Av, Teff <= 0 and Dist <= 0 (NaN / inf patterns), then random
draws with Av in [0, 6].  Bars: magnitudes within 1e-12 absolute and relative (test_band_subset_vs_oracle), lnL within
1e-10 relative, non-finite values identical.
"""
import numpy as np
import pytest

from oracle import payne_oracle as O
from thepayne_b200 import synth

KTILE = 8
SMEM_LIMIT = 200 * 1024
ALL_BANDS = synth.C1_BANDS + ['Extra_%d' % i for i in range(13)]       # 40; no high-Av table for the extra ones

# H hidden width, nb bands, B points, mode ('scaled': log(A), photscale; 'dist': log(R), Dist), slab (max_batch, or
# None), spec (also through the spectrum path)
CASES = [
    dict(H=1, nb=2, B=9, mode='scaled'),
    dict(H=7, nb=27, B=7, mode='dist'),
    dict(H=31, nb=1, B=4097, mode='scaled'),
    dict(H=32, nb=40, B=8, mode='dist', spec=True),
    dict(H=33, nb=27, B=4097, mode='dist'),
    dict(H=128, nb=2, B=1, mode='scaled', spec=True),
    dict(H=129, nb=40, B=9, mode='scaled'),
    dict(H=384, nb=1, B=4097, mode='dist'),
    dict(H=385, nb=2, B=7, mode='scaled', spec=True),
    dict(H=385, nb=27, B=30, mode='dist', slab=12),
    dict(H=1600, nb=1, B=9, mode='dist'),
    dict(H=1600, nb=2, B=8, mode='scaled', slab=4),
]


def _name(c):
    return 'H%d_nb%d_B%d_%s%s' % (c['H'], c['nb'], c['B'], c['mode'], '_slab%d' % c['slab'] if c.get('slab') else '')


def smem(H, nb, slots):
    return 2 * KTILE * H * 8 + (KTILE * nb * 8 if slots else 0)


def _fit(mode):
    return ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]'] + (['log(A)', 'Av'] if mode == 'scaled' else ['log(R)', 'Dist', 'Av'])


def _rows(fit, B, seed):
    """the edge rows first, then draws in the box with Av in [0, 6]"""
    ix = {p: i for i, p in enumerate(fit)}
    box = dict(synth._BOX, Av=(0.0, 6.0), Teff=(3000.0, 9000.0))
    rng = np.random.default_rng(seed)
    lo, hi = np.array([box[p][0] for p in fit]), np.array([box[p][1] for p in fit])
    th = lo + (hi - lo) * rng.random((max(B, 12), len(fit)))
    edges = [('Av', np.nextafter(5.0, -np.inf)), ('Av', 5.0), ('Av', np.nextafter(5.0, np.inf)), ('Av', np.nan),
             ('Teff', 0.0), ('Teff', -50.0)]
    if 'Dist' in ix:
        edges += [('Dist', 0.0), ('Dist', -3.0)]
    for r, (p, v) in enumerate(edges):
        th[r, ix[p]] = v
    # Av = 5 exactly again at a row of the second tile
    th[9, ix['Av']] = 5.0
    return np.ascontiguousarray(th[:B])


def _net(H, nb, seed=5):
    return synth.make_photnet(ALL_BANDS[:nb], H=H, seed=seed)


def _obs(bands, seed):
    rng = np.random.default_rng(seed)
    return {b: (float(5.0 + rng.random()), float(0.02 + 0.05 * rng.random())) for b in bands}


def oracle(net, bands, fit, th, obs):
    """magnitudes [B, len(bands)] and SED chi2 [B] of genphot (genmod.py:110-187) with the net of ``bands``"""
    idx = [net.bands.index(b) for b in bands]
    sub = synth.PhotNet(list(bands), net.w1[idx], net.b1[idx], net.w2[idx], net.b2[idx], net.w3[idx], net.b3[idx],
                        net.xmin, net.xmax, net.hiav[idx])
    scaled = 'log(A)' in fit
    mags = np.empty((len(th), len(bands)))
    with np.errstate(all='ignore'):
        for i, t in enumerate(th):
            mags[i] = np.atleast_1d(O.genphot(sub, list(t), scaled))
        o = np.array([obs[b][0] for b in bands])
        e = np.array([obs[b][1] for b in bands])
        chi2 = np.zeros(len(th))
        for j in range(len(bands)):                      # likelihood.py:109-112: summed in the star's band order
            chi2 = chi2 + ((mags[:, j] - o[j]) ** 2.0) / (e[j] ** 2.0)
    return mags, chi2


def _same(got, ref, rtol, atol):
    """finite values within the bars, every other value identical (NaN, +-inf)"""
    fin = np.isfinite(ref)
    if not np.array_equal(fin, np.isfinite(got)) or not np.array_equal(got[~fin], ref[~fin], equal_nan=True):
        return False
    return bool(np.all(np.abs(got[fin] - ref[fin]) <= atol + rtol * np.abs(ref[fin])))


def test_matrix_covers_every_branch():
    """CPU: hidden widths across the 48 KB opt-in and at the 200 KB edge, batches off the tile, every band count."""
    hs = {c['H'] for c in CASES}
    print('H:', sorted(hs), ' dynamic shared memory (KB):', sorted({smem(h, 0, False) / 1024 for h in hs}))
    assert {1, 7, 31, 32, 33, 128, 129, 384, 385, 1600} <= hs
    assert smem(384, 0, False) <= 48 * 1024 < smem(385, 0, False)
    assert smem(1600, 0, False) == SMEM_LIMIT and smem(1601, 0, False) > SMEM_LIMIT and smem(1600, 1, True) > SMEM_LIMIT
    assert {c['nb'] for c in CASES} == {1, 2, 27, 40} and {1, 7, 8, 9, 4097} <= {c['B'] for c in CASES}
    assert any(c.get('slab') and c['slab'] % KTILE for c in CASES)
    assert {c['mode'] for c in CASES} == {'scaled', 'dist'} and any(c.get('spec') for c in CASES)
    for mode in ('scaled', 'dist'):
        th = _rows(_fit(mode), 12, 0)
        av = th[:, _fit(mode).index('Av')]
        assert np.nextafter(5.0, -np.inf) in av and 5.0 in av and np.nextafter(5.0, np.inf) in av and np.isnan(av).any()
        assert (th[:, 0] <= 0).any()
    assert (_rows(_fit('dist'), 12, 0)[:, _fit('dist').index('Dist')] <= 0).any()
    # the band-slot test: whole tiles with no point that has a given band
    star = _slot_stars(64)
    assert any(set(star[t:t + KTILE]) == {0} for t in range(0, 64, KTILE))
    assert any(len(set(star[t:t + KTILE])) > 1 for t in range(0, 64, KTILE))


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES, ids=_name)
def test_phot_kernel_against_oracle(case):
    import torch
    from thepayne_b200.engine import Engine
    H, nb, B, mode = case['H'], case['nb'], case['B'], case['mode']
    net = _net(H, nb)
    fit = _fit(mode)
    obs = _obs(net.bands, nb)
    th = _rows(fit, B, H)
    mags_ref, chi2_ref = oracle(net, net.bands, fit, th, obs)
    eng = Engine(phot=net, obs_phot=obs, fitpars_i=fit, runbools=[False, True, False, mode == 'scaled', False])
    if case.get('slab'):
        eng.set('max_batch', case['slab'])
    thd = torch.from_numpy(th).cuda()
    _, mags, lnl_m = eng.model_batch(thd)
    lnl = eng.lnlike_batch(thd)
    lnl_h = eng.lnlike_batch(th)
    mags, lnl_m, lnl = mags.cpu().numpy(), lnl_m.cpu().numpy(), lnl.cpu().numpy()
    dm = np.abs(mags - mags_ref)[np.isfinite(mags_ref)]
    print('%s: max |dmag| %.2e, max |dlnL| %.2e' % (_name(case), np.max(dm, initial=0.0),
                                                   np.max(np.abs(lnl - -0.5 * chi2_ref)[np.isfinite(chi2_ref)], initial=0.0)))
    assert np.isfinite(mags_ref).sum() >= min(B, 4) * nb // 2
    assert _same(mags, mags_ref, 1e-12, 1e-12)
    for l in (lnl, lnl_m, lnl_h):
        assert _same(l, -0.5 * chi2_ref, 1e-10, 1e-9)
    assert eng.query('status') == 0
    eng.close()
    if not case.get('spec'):
        return
    # spectrum + photometry: lnL = -0.5 (chi2_spec + chi2_sed), the spectrum's part from a spectrum-only engine
    cfg = synth.config_mini(O.model_fn, n_obs=300, H=16)
    sfit = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Inst_R']
    rng = np.random.default_rng(4)
    srows = np.column_stack([rng.uniform(-1, 1, B), rng.uniform(0, 5, B), rng.uniform(30000, 37000, B)])
    jth = np.ascontiguousarray(np.column_stack([th[:, :4], srows, th[:, 4:]]))
    kw = dict(spec=cfg.spec, obs_wave=cfg.obs_wave, obs_flux=cfg.obs_flux, obs_eflux=cfg.obs_eflux)
    joint = Engine(phot=net, obs_phot=obs, fitpars_i=sfit + fit[4:], runbools=[True, True, False, mode == 'scaled', False],
                   **kw)
    alone = Engine(fitpars_i=sfit, runbools=[True, False, False, False, False], **kw)
    jt = torch.from_numpy(jth).cuda()
    _, jm, jl = joint.model_batch(jt)
    sl = alone.lnlike_batch(torch.from_numpy(np.ascontiguousarray(jth[:, :7])).cuda()).cpu().numpy()
    jm, jl = jm.cpu().numpy(), jl.cpu().numpy()
    assert _same(jm, mags_ref, 1e-12, 1e-12)
    with np.errstate(invalid='ignore'):
        want = -0.5 * (-2.0 * sl + chi2_ref)
    assert _same(jl, want, 1e-10, 1e-9)
    joint.close()
    alone.close()


def _slot_stars(B):
    """star of every point: tiles 0, 2, 4, ... all star 0 or all star 2, the odd tiles mixed"""
    star = np.empty(B, np.int32)
    for p in range(B):
        t = p // KTILE
        star[p] = (0 if t % 4 == 0 else 2) if t % 2 == 0 else p % 3
    return star


@pytest.mark.gpu
@pytest.mark.parametrize('H,nb', [(33, 27), (385, 40)])
def test_band_slots_against_oracle(H, nb):
    """Band lists on a spectrum + photometry engine: star 0 has the first half of the bands, star 1 the second half in
    reverse order, star 2 none (its own layout without photometry); whole tiles of star 0 or star 2 skip the bands no
    point of theirs has.  lnL = -0.5 (chi2_spec + chi2_sed), chi2_spec from a spectrum-only engine."""
    import torch
    from thepayne_b200.engine import Engine
    net = _net(H, nb)
    cfg = synth.config_mini(O.model_fn, n_obs=300, H=16)
    sfit = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Inst_R']
    fit = sfit + ['log(A)', 'Av']
    half = max(1, nb // 2)
    b0, b1 = net.bands[:half], net.bands[half:][::-1]
    obs = dict(wave=cfg.obs_wave, flux=cfg.obs_flux, eflux=cfg.obs_eflux)
    stars = [dict(obs, phot=_obs(b0, 1), bands=b0, fitpars_i=fit, runbools=[True, True, False, True]),
             dict(obs, phot=_obs(b1, 2), bands=b1, fitpars_i=fit, runbools=[True, True, False, True]),
             dict(obs, phot=None, fitpars_i=sfit, runbools=[True, False, False, False])]
    eng = Engine(spec=cfg.spec, phot=net, stars=stars)
    alone = Engine(spec=cfg.spec, fitpars_i=sfit, runbools=[True, False, False, False, False], obs_wave=cfg.obs_wave,
                   obs_flux=cfg.obs_flux, obs_eflux=cfg.obs_eflux)
    B = 64
    pth = _rows(_fit('scaled'), B, 7)
    rng = np.random.default_rng(4)
    srows = np.column_stack([rng.uniform(-1, 1, B), rng.uniform(0, 5, B), rng.uniform(30000, 37000, B)])
    th = np.ascontiguousarray(np.column_stack([pth[:, :4], srows, pth[:, 4:]]))
    star = _slot_stars(B)
    _, mags, lnl_m = eng.model_batch(torch.from_numpy(th).cuda(), torch.from_numpy(star).cuda())
    mags, lnl_m = mags.cpu().numpy(), lnl_m.cpu().numpy()
    sl = alone.lnlike_batch(torch.from_numpy(np.ascontiguousarray(th[:, :7])).cuda()).cpu().numpy()
    for k, bands in ((0, b0), (1, b1)):
        rows = np.nonzero(star == k)[0]
        mr, cr = oracle(net, bands, _fit('scaled'), pth[rows], stars[k]['phot'])
        assert _same(mags[rows, :len(bands)], mr, 1e-12, 1e-12), k
        assert np.isnan(mags[rows, len(bands):]).all()
        with np.errstate(invalid='ignore'):
            assert _same(lnl_m[rows], -0.5 * (-2.0 * sl[rows] + cr), 1e-10, 1e-9), k
    rows = np.nonzero(star == 2)[0]
    assert np.isnan(mags[rows]).all() and _same(lnl_m[rows], sl[rows], 1e-10, 1e-9)
    assert eng.query('status') == 0
    eng.close()
    alone.close()


@pytest.mark.gpu
def test_shared_memory_limit():
    """H = 1600 without band lists is exactly the 200 KB limit and is accepted; with band lists, or H = 1601, refused."""
    from thepayne_b200 import _lib
    from thepayne_b200.engine import Engine
    fit = _fit('scaled')
    rb = [False, True, False, True, False]
    net = _net(1600, 2)
    Engine(phot=net, obs_phot=_obs(net.bands, 0), fitpars_i=fit, runbools=rb).close()
    with pytest.raises(_lib.PayneError, match='error -4'):
        Engine(phot=net, stars=[{'phot': _obs(net.bands[:1], 0), 'bands': net.bands[:1]}], fitpars_i=fit, runbools=rb)
    net = _net(1601, 1)
    with pytest.raises(_lib.PayneError, match='error -4'):
        Engine(phot=net, obs_phot=_obs(net.bands, 0), fitpars_i=fit, runbools=rb)
