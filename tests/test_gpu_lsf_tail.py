"""The LSF-vector tail (tail_lsf.cuh) against the oracle's smooth_lsf at every transform size it branches on.

An LSF vector (a fixed ``Inst_R`` array, the dispersion in AA at every observed pixel) runs on tail_lsf_kernel whatever
the emulator grid, and the kernel's shape depends on the point (DESIGN §3.5):

  * nx = 2^ceil(log2(2 / x_per_sigma)) samples for the convolution, x_per_sigma the median over the mask of
    gradient(cdf) / (dw / sigma): nx = 1 is NaN (the reference's irfft raises), nx = 2 .. 16 a direct convolution,
    32 .. 2^log2nx_max the runtime-planned FFT, above that NaN and status bit 0 (log2nx_max = min(15, log2 N1));
  * the cumulative sum is a block scan of ceil(nM / 256) elements per thread (nM = masked emulator pixels);
  * the median is an exact radix selection (ties from a constant vector, odd and even nM);
  * the last np.interp clamps at the ends of the transform grid when observed pixels lie outside the emulator's.

GRIDS is the matrix as plain data.  Every grid gets one star per transform size log2nx = 0 .. log2nx_max + 1, its LSF
vector scaled on the host so that the truth row lands at 2 / x_per_sigma = 2^(log2nx - 1/2) (x_per_sigma scales with
the vector), in the middle of its size, away from the power-of-two ties the device's chunked cumsum may round
differently.  The stars cycle through four vector shapes, three observed layouts and three pixel counts.
`test_matrix_covers_every_size` (no GPU) recomputes every row's log2nx and nM with the oracle's formula and asserts the
union reaches every branch.  The GPU test compares flux and lnL of every row with the oracle, and evaluates every star
again as a one-member target (the target form of the kernel), which must be bit-identical.

Rows per star: truth, Vrot = 0, Vrad = 0, Vrad = +-250 km/s, Vrot = 100 km/s (a wide rotation kernel), four random
draws.  Bars as in test_gpu_transform_sizes.py: NaN patterns identical; flux within 1e-5 relative and FLUX_GUARD; lnL
within max(1e-3, 1e-8 |lnL|), or under the float64-emulator rule of `_lnl_ok` far from the truth, where a transform
of few samples adds the coherent rounding of the fp32 convolved spectrum (half an ulp of every model pixel, with the
sign of its residual); status 0, except bit 0 on the rows above log2nx_max.
"""
import math

import numpy as np
import pytest

from oracle import payne_oracle as O
from thepayne_b200 import synth

W0 = 5000.0
R_FWHM = 50000.0
FLUX_GUARD = 5e-7
LABELS = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot']
SHAPES = ['constant', 'ramp', 'step', 'noisy']
LAYOUTS = ['inside', 'full', 'outside']
N_OBS = [8, 300, 2000]

# name: n emulator pixels; grid: 'log' (ann_wavegrid) or 'linear'; npoly: continuum coefficients (0: none)
GRIDS = []
for _L in (10, 12, 13, 14, 15):
    GRIDS += [dict(name='L%d_pow2' % _L, n=1 << _L, grid='log', npoly=3 if _L % 2 else 0),
              dict(name='L%d_pow2h1' % _L, n=(1 << (_L - 1)) + 1, grid='log', npoly=0 if _L % 2 else 3)]
# both sides of the scan's chunk edges (nM = 256, 512) and log2 N1 = 8, 9
for _n in (200, 255, 256, 257, 511, 512, 513):
    GRIDS.append(dict(name='n%d' % _n, n=_n, grid='log', npoly=3 if _n % 2 else 0))
GRIDS += [dict(name='linear3000', n=3000, grid='linear', npoly=3),
          dict(name='linear20000', n=20000, grid='linear', npoly=0)]
BY_NAME = {g['name']: g for g in GRIDS}


def log2_of(n):
    return int(math.ceil(math.log2(n)))


def log2nx_max(g):
    return min(15, log2_of(g['n']))


def _wave(g):
    n = g['n']
    if g['grid'] == 'linear':
        return np.linspace(W0, W0 * 1.06, n)
    rsig = R_FWHM * synth.SIGMA_TO_FWHM_TRAIN
    w, _ = synth.ann_wavegrid(W0, W0 * (1.0 + 1.0 / (3.0 * rsig)) ** (n - 1.0), R_FWHM)
    assert len(w) == n
    return w


def _obs_wave(w, layout, n):
    a, b = w[0], w[-1]
    if layout == 'inside':
        return np.linspace(a + 0.3 * (b - a), a + 0.6 * (b - a), n)
    if layout == 'full':          # a quarter pixel inside the grid's ends
        q = 0.25 * (w[1] - w[0])
        return np.linspace(a + q, b - q, n)
    return np.linspace(a - 0.1 * (b - a), b + 0.1 * (b - a), n)    # beyond the emulator on both sides


def _shape(kind, ow, seed):
    x = (ow - ow[0]) / (ow[-1] - ow[0])
    if kind == 'constant':
        return np.ones(len(ow))
    if kind == 'ramp':
        return 1.0 + 9.0 * x
    if kind == 'step':
        return np.where(x < 0.5, 1.0, 3.0)
    return 1.0 + 0.3 * np.random.default_rng(seed).uniform(-1.0, 1.0, len(ow))


def _nf(w, theta, ow, lsf):
    """(2 / x_per_sigma, nM) of one row: smoothing.py:126-133, 525-565 on the Doppler-shifted grid, as the oracle has
    them."""
    vrad = theta[LABELS.index('Vrad')]
    mw = w * (1.0 + vrad / O.SPEEDOFLIGHT) if vrad != 0.0 else w
    disp = np.interp(mw, ow, lsf)
    m = (mw > ow.min() - 2000.0) & (mw < ow.max() + 2000.0)
    dw = np.gradient(mw[m])
    cdf = np.cumsum(dw / disp[m])
    cdf /= cdf.max()
    return 2.0 / np.nanmedian(np.gradient(cdf) / (dw / disp[m])), int(m.sum())


def lsf_size(w, theta, ow, lsf):
    """(log2nx, nM) of one row."""
    nf, nm = _nf(w, theta, ow, lsf)
    return int(np.ceil(np.log2(nf))), nm


_built = {}


def build(name):
    """(emulator, stars, per-star target log2nx) of a grid: one star per log2nx = 0 .. log2nx_max + 1."""
    if name in _built:
        return _built[name]
    g = BY_NAME[name]
    w = _wave(g)
    spec = synth.make_specnet(4, 16, w, R_FWHM * synth.SIGMA_TO_FWHM_TRAIN, seed=g['n'] % 97)
    fit = LABELS + ['pc_%d' % i for i in range(g['npoly'])]
    truth = np.array([5770.0, 4.44, 0.0, 0.0, 0.5, 3.0] + [1.0, -0.02, 0.02][:g['npoly']])
    net = O.make_net(spec)
    stars, sizes = [], list(range(0, log2nx_max(g) + 2))
    for k, l2 in enumerate(sizes):
        j = k + GRIDS.index(g)                 # the grids start the cycles at different sizes
        ow = _obs_wave(w, LAYOUTS[j % 3], N_OBS[(j // 3) % 3])
        base = _shape(SHAPES[j % 4], ow, seed=k)
        lsf = base * (_nf(w, truth, ow, base)[0] / 2.0 ** (l2 - 0.5))   # 2 / x_per_sigma goes as 1 / scale
        assert lsf_size(w, truth, ow, lsf)[0] == l2, (name, k, l2)
        f = _oracle_flux(net, spec, lsf, ow, truth, g['npoly'])
        f = np.ones(len(ow)) if not np.all(np.isfinite(f)) else f
        e = np.abs(f) / 50.0
        stars.append({'wave': ow, 'flux': f + e * np.random.default_rng(k).standard_normal(len(ow)), 'eflux': e,
                      'fixedpars': {'Inst_R': lsf}, 'fitpars_i': fit, 'layout': LAYOUTS[j % 3],
                      'shape': SHAPES[j % 4]})
    _built[name] = (spec, stars, sizes, fit, truth)
    return _built[name]


def rows(g, fit, truth, seed):
    out = []
    for vrad, vrot in [(None, None), (None, 0.0), (0.0, None), (250.0, None), (-250.0, None), (None, 100.0)]:
        r = truth.copy()
        if vrad is not None:
            r[4] = vrad
        if vrot is not None:
            r[5] = vrot
        out.append(r)
    box = dict(synth._BOX, pc_0=(0.75, 1.25), pc_1=(-0.1, 0.1), pc_2=(-0.1, 0.1))
    rng = np.random.default_rng(seed)
    lo, hi = np.array([box[p][0] for p in fit]), np.array([box[p][1] for p in fit])
    out += list(lo + (hi - lo) * rng.random((4, len(fit))))
    return np.array(out)


def _oracle_flux(net, spec, lsf, ow, th, npoly):
    """model spectrum of one row (genmod.py:58-108 with an LSF vector); NaN where the reference raises (nx = 1)"""
    pars = list(th[:4]) + [th[4], th[5], np.nan, lsf] + list(th[6:6 + npoly])
    try:
        return O.genspec(net, spec, pars, ow, npoly > 0)[1]
    except (ValueError, ZeroDivisionError):        # nx = 1: irfft of no point; nx = 0: dx = 1 / 0
        return np.full(len(ow), np.nan)


def cells():
    """Every (grid, star, log2nx the star was scaled for, log2nx of the row, nM, layout, shape, n_obs, npoly) the
    matrix has."""
    out = []
    for g in GRIDS:
        spec, stars, sizes, fit, truth = build(g['name'])
        for k, st in enumerate(stars):
            for th in rows(g, fit, truth, k):
                l2, nm = lsf_size(spec.wavelength, th, st['wave'], st['fixedpars']['Inst_R'])
                out.append((g['name'], k, sizes[k], l2, nm, st['layout'], st['shape'], len(st['wave']), g['npoly']))
    return out


def test_matrix_covers_every_size():
    """CPU: every row lands on the transform size its star was scaled for, and the union reaches every branch."""
    cs = cells()
    # the truth row of every star lands on the size it was scaled for (Vrad = +-250 km/s moves a small grid by a
    # tenth of its span against the observed pixels, so other rows may land elsewhere)
    for g in GRIDS:
        spec, stars, sizes, fit, truth = build(g['name'])
        for k, st in enumerate(stars):
            assert lsf_size(spec.wavelength, truth, st['wave'], st['fixedpars']['Inst_R'])[0] == sizes[k], (g['name'], k)
    got = {c[3] for c in cs}
    print('log2nx reached:', sorted(got))
    assert set(range(0, 16)) <= got
    for g in GRIDS:
        mx = log2nx_max(g)
        mine = {c[3] for c in cs if c[0] == g['name']}
        assert set(range(0, mx + 2)) <= mine, g['name']
        print('%s: log2 N1 %d, log2nx_max %d, log2nx %d..%d' % (g['name'], log2_of(g['n']), mx, min(mine), max(mine)))
    nms = {c[4] for c in cs}
    print('nM on the scan chunk edges:', sorted(nms & {255, 256, 257, 511, 512, 513}))
    assert {255, 256, 257, 511, 512, 513} <= nms
    assert {log2_of(g['n']) for g in GRIDS} >= {8, 9, 10, 12, 13, 14, 15}
    assert any(g['grid'] == 'linear' for g in GRIDS)
    # every vector shape, observed layout and pixel count at a directly convolved size, an FFT size and the limit
    for pick in (lambda c: 1 <= c[3] <= 4, lambda c: 5 <= c[3] <= log2nx_max(BY_NAME[c[0]])):
        sub = [c for c in cs if pick(c)]
        assert {c[5] for c in sub} == set(LAYOUTS) and {c[6] for c in sub} == set(SHAPES)
        assert {c[7] for c in sub} == set(N_OBS) and {c[8] > 0 for c in sub} == {False, True}
    # odd and even mask widths at the ties of the constant vector
    assert {c[4] % 2 for c in cs if c[6] == 'constant'} == {0, 1}


def _close(a, b):
    fin = np.isfinite(b)
    return np.array_equal(np.isnan(a), ~fin) and np.all(np.abs(a[fin] - b[fin]) <= np.maximum(1e-3, 1e-8 * np.abs(b[fin])))


def _lnl(f, st):
    return -0.5 * np.sum(((f - st['flux']) ** 2.0) / (st['eflux'] ** 2.0))


@pytest.mark.gpu
@pytest.mark.parametrize('name', [g['name'] for g in GRIDS])
def test_lsf_tail_against_oracle(name):
    import torch
    from thepayne_b200.engine import Engine
    g = BY_NAME[name]
    spec, stars, sizes, fit, truth = build(name)
    net, ideal = O.make_net(spec), O.make_net(spec, ideal=True)
    th, sv, ref_f, ref_l, over = [], [], [], [], []
    for k, st in enumerate(stars):
        for r in rows(g, fit, truth, k):
            th.append(r)
            sv.append(k)
            f = _oracle_flux(net, spec, st['fixedpars']['Inst_R'], st['wave'], r, g['npoly'])
            l2 = lsf_size(spec.wavelength, r, st['wave'], st['fixedpars']['Inst_R'])[0]
            if l2 > log2nx_max(g):
                f = np.full(len(f), np.nan)                    # above the largest transform: NaN and status bit 0
            ref_f.append(f)
            over.append(l2 > log2nx_max(g))
            ref_l.append(_lnl(f, st))
    th, sv, ref_l, over = np.array(th), np.array(sv, np.int32), np.array(ref_l), np.array(over)
    eng = Engine(spec=spec, stars=[{k: v for k, v in st.items() if k not in ('layout', 'shape')} for st in stars],
                 targets=[1] * len(stars), runbools=[True, False, g['npoly'] > 0, False, False])
    assert eng.query('lsf') == 1
    dev = torch.device('cuda', eng.device)
    max_rel = max_dl = 0.0
    for part in (~over, over):                             # status is sticky: the rows above the limit go last
        idx = np.nonzero(part)[0]
        thd, sd = torch.from_numpy(np.ascontiguousarray(th[idx])).to(dev), torch.from_numpy(sv[idx]).to(dev)
        flux, _, lnl_m = eng.model_batch(thd, sd, want_mags=False)
        lnl = eng.lnlike_batch(thd, sd)
        ft, _, _, lt = eng.model_batch_targets(thd, sd, want_chi2=False, want_mags=False)
        lt2 = eng.lnlike_batch_targets(thd, sd)
        torch.cuda.synchronize()
        flux, lnl_m, lnl, ft, lt, lt2 = [x.cpu().numpy() for x in (flux, lnl_m, lnl, ft, lt, lt2)]
        # the target form of the kernel: bit-identical to the star form, NaN patterns included
        assert np.array_equal(ft, flux, equal_nan=True) and np.array_equal(lt, lnl_m, equal_nan=True)
        assert np.array_equal(lt2, lnl, equal_nan=True) and np.array_equal(lnl, lnl_m, equal_nan=True)
        for i, p in enumerate(idx):
            st = stars[sv[p]]
            n = len(st['wave'])
            f, rf = flux[i, :n], ref_f[p]
            fin = np.isfinite(rf)
            assert np.array_equal(np.isnan(f), ~fin), (name, sv[p], sizes[sv[p]], th[p])
            rel = np.max(np.abs(f[fin] - rf[fin]) / np.abs(rf[fin]), initial=0.0)
            assert rel < 1e-5 and rel <= FLUX_GUARD, (name, sv[p], sizes[sv[p]], rel)
            max_rel = max(max_rel, rel)
            if np.isfinite(ref_l[p]):
                max_dl = max(max_dl, abs(lnl[i] - ref_l[p]))
            if not _close(lnl[i:i + 1], ref_l[p:p + 1]):
                # far from the truth the fp32 emulator alone moves lnL: judge against a float64 emulator.  The
                # convolved spectrum is held in fp32 (DESIGN §4), and a transform of few samples spreads each one's
                # rounding over many observed pixels, coherently: that floor is half an fp32 ulp of every model pixel
                # with the sign of its residual.
                fe = _oracle_flux(ideal, spec, st['fixedpars']['Inst_R'], st['wave'], th[p], g['npoly'])
                e = _lnl(fe, st)
                floor = 2.0 ** -24 * np.sum(np.abs(fe - st['flux']) * np.abs(fe) / st['eflux'] ** 2)
                assert abs(lnl[i] - e) <= abs(ref_l[p] - e) + floor or abs(lnl[i] - e) <= max(1e-3, 3e-8 * abs(e)), \
                    (name, sv[p], lnl[i], ref_l[p], e, floor)
        assert eng.query('status') == (1 if over[idx].any() else 0), name
    print('%s: max flux rel err %.2e, max |dlnL| %.2e' % (name, max_rel, max_dl))
    eng.close()
