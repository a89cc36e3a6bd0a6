"""Every transform size and stage-2 branch of the fused tail against the oracle.

The tail's code path is chosen by problem shape (DESIGN §3.3, §3.3b):

  * stage 1 (rotation) runs one transform of N1 = 2^ceil(log2 n) samples, n = emulator pixels; the fast tail is compiled
    once per log2 N1 = 10..16, with and without the continuum polynomial (tail_fast_tu.inl);
  * stage 2 (instrument) transforms the mask around the observed window, nM pixels, at N2 = 2^ceil(log2 nM):
    N2 = N1 and N2 = N1/2 use compile-time-planned transforms, anything smaller the runtime-planned FFT of fft.cuh;
  * N1 = 65536 runs on the cluster kernel (default) or the split single-CTA kernel, N1 = 32768 on one CTA (default) or the
    cluster; the general-grid tail (`fast_tail` 0) is the only path for grids that are not log-uniform or have <= 512
    pixels, and the fallback for every log-uniform grid up to N1 = 32768.

CONFIGS below is the matrix as plain data; `test_matrix_covers_every_path` (no GPU) recomputes each row's
(log2 N1, log2 N2) on the host from the oracle's own mask and asserts the union still reaches every branch, so a change of
the synthetic defaults cannot silently empty a path.  The GPU test compares flux and lnL of every row, for every kernel
the shape can run on, with the oracle.

Rows per configuration: truth, Vrot = 0, Vrad = 0, Vrad = +-250 km/s (moves the mask ends, clips it at the grid ends),
Vrot = 100 km/s (its rotation-kernel table range overflows the shared-memory window of the fast kernels), four random
draws; the narrow-mask edge case adds a Vrad sweep that moves nM across 16 / 17.

Where a configuration asks for a narrow mask, its instrumental resolution is scaled up (Inst_R x `inst`, emulator
resolution above that) so that the +-20 sigma pads of mask_wave (smoothing.py:631-647) shrink to a few pixels.

Bars: NaN patterns identical; flux within 1e-5 relative (the parity bar) and within FLUX_GUARD, a regression guard set
from what B200 measures (1.5e-7; measured at most 7.8e-8); lnL within max(1e-3, 1e-8 |lnL|); no status bit.  Far from
the truth (|lnL| ~ 1e5) the fp32 emulator alone moves lnL by a few 1e-8 relative, in the reference as here (DESIGN §6,
test_fuzz_far_points_sit_at_the_float32_noise_floor); a row beyond the bar passes under the rule of that test: at least as
close as the reference to the oracle with a float64 emulator, or within max(1e-3, 3e-8 |lnL|) of it.  A mask narrower
than 17 pixels must give NaN (DESIGN §5: the reference raises there).
"""
import math

import numpy as np
import pytest

from oracle import payne_oracle as O
from thepayne_b200 import synth

W0 = 5000.0
R_FWHM = 50000.0
VROT_WIDE = 100.0
FLUX_GUARD = 1.5e-7

# name: L = log2 N1; n: 'pow2' (n = 2^L), 'pow2h1' (n = 2^(L-1) + 1) or a pixel count; win: 'full' (observed window =
# emulator grid) or the target log2 N2; npoly: continuum polynomial order + 1 (0: none); inst: Inst_R scale
# (narrow masks); sweep: add Vrad sweep rows; grid: 'log' or 'linear' (general tail only)
CONFIGS = []
for _L in range(10, 17):
    CONFIGS += [dict(name='L%d_pow2_full' % _L, L=_L, n='pow2', win='full', npoly=0),
                dict(name='L%d_pow2h1_full' % _L, L=_L, n='pow2h1', win='full', npoly=3),
                dict(name='L%d_pow2_half' % _L, L=_L, n='pow2', win=_L - 1, npoly=2),
                dict(name='L%d_pow2h1_half' % _L, L=_L, n='pow2h1', win=_L - 1, npoly=0)]
# runtime-planned stage 2: every log2 N2 from 5 to 14 at least once, at every L
for _L, _k in [(10, 8), (10, 5), (11, 9), (11, 6), (12, 10), (12, 7), (13, 11), (13, 6), (14, 12), (14, 8),
               (15, 13), (15, 9), (16, 14), (16, 13), (16, 7)]:
    CONFIGS.append(dict(name='L%d_narrow%d' % (_L, _k), L=_L, n='pow2' if _k % 2 else 'pow2h1', win=_k,
                        npoly=2 if _k % 3 else 0, inst=float(max(1, 2 ** (10 - _k)))))
CONFIGS += [
    # nM = 16 / 17: the smallest accepted mask and the first one refused
    dict(name='L10_mask17', L=10, n='pow2', win=('nM', 16.5), npoly=0, inst=16.0, sweep=True),
    # general-tail-only shapes: <= 512 emulator pixels, and a linearly spaced grid
    dict(name='L9_full', L=9, n='pow2h1', win='full', npoly=2),
    dict(name='L9_narrow', L=9, n='pow2', win=6, npoly=0, inst=16.0),
    dict(name='L8_full', L=8, n=200, win='full', npoly=0),
    dict(name='L8_narrow', L=8, n='pow2', win=7, npoly=2, inst=8.0),
    dict(name='L12_linear', L=12, n=3000, win=11, npoly=2, grid='linear'),
    dict(name='L14_linear', L=14, n=9000, win=10, npoly=0, grid='linear', inst=2.0),
]
BY_NAME = {c['name']: c for c in CONFIGS}


def n_pixels(c):
    if c['n'] == 'pow2':
        return 1 << c['L']
    if c['n'] == 'pow2h1':
        return (1 << (c['L'] - 1)) + 1
    return int(c['n'])


def kernels(c):
    """The tail kernels a configuration can run on ('fast' = tail_fast single CTA, 'split' = its 65536-sample variant)."""
    if c.get('grid') == 'linear' or c['L'] <= 9:
        return ['general']
    if c['L'] == 16:
        return ['cluster', 'split']
    return ['fast', 'cluster', 'general'] if c['L'] == 15 else ['fast', 'general']


def _grid(c):
    n = n_pixels(c)
    if c.get('grid') == 'linear':
        return np.linspace(W0, W0 * 1.06, n)
    rsig = R_FWHM * synth.SIGMA_TO_FWHM_TRAIN
    w1 = W0 * (1.0 + 1.0 / (3.0 * rsig)) ** (n - 1.0)      # ann_wavegrid's own recurrence: the grid stops exactly here
    w, _ = synth.ann_wavegrid(W0, w1, R_FWHM)
    assert len(w) == n
    return w


def _window(c, w, instR):
    """Observed pixels: the whole grid, or a window centred in it whose mask at the truth is ~3/4 of 2^win pixels."""
    if c['win'] == 'full':
        # a quarter pixel inside the grid ends: an observed pixel exactly on an end is an fp tie between the reference's
        # exp(log(w)) grid and the log-space position of the CUDA path, not a shape this file is about
        q = 0.25 * (math.log(w[-1]) - math.log(w[0])) / (len(w) - 1)
        return np.linspace(w[0] * math.exp(q), w[-1] * math.exp(-q), min(len(w), 2000))
    nm = c['win'][1] if isinstance(c['win'], tuple) else 0.75 * 2 ** c['win']
    dlnw = (math.log(w[-1]) - math.log(w[0])) / (len(w) - 1)
    mid, h = 0.5 * (math.log(w[0]) + math.log(w[-1])), 0.5 * nm * dlnw
    pad = 20.0 / (O.FWHM_FACTOR_FIT * instR)
    lo, hi = math.exp(mid - h) / (1.0 - pad), math.exp(mid + h) / (1.0 + pad)
    assert lo < hi, c['name']
    return np.linspace(lo, hi, int(min(max(nm, 8), 2000)))


_built = {}


def build(name):
    """SynthConfig of a matrix entry (deterministic, cached)."""
    if name in _built:
        return _built[name]
    c = BY_NAME[name]
    w = _grid(c)
    inst = c.get('inst', 1.0)
    instR = 32000.0 * inst
    cfg = synth.build_config(name, model_fn=O.model_fn, ann_range=(w[0], w[-1]), r_fwhm=R_FWHM,
                             obs_wave=_window(c, w, instR), H=16 if c['L'] >= 14 else 32, npoly=c['npoly'],
                             seed_net=c['L'])
    assert np.array_equal(cfg.spec.wavelength, w) or c.get('grid') == 'linear'
    if c.get('grid') == 'linear' or inst != 1.0:
        if c.get('grid') == 'linear':
            cfg.spec = synth.make_specnet(4, cfg.spec.weights[0].shape[0], w, R_FWHM * synth.SIGMA_TO_FWHM_TRAIN,
                                          seed=c['L'])
        if inst != 1.0:
            ip = cfg.fitpars_i.index('Inst_R')
            cfg.box = dict(cfg.box)
            cfg.box['Inst_R'] = (30000.0 * inst, 37000.0 * inst)
            cfg.theta_true = cfg.theta_true.copy()
            cfg.theta_true[ip] = instR
            # the emulator must resolve finer than the narrowest requested profile (else NaN, smoothing.py:271)
            cfg.spec.resolution = 2.0 * O.FWHM_FACTOR_FIT * 37000.0 * inst
        flux, _ = O.model_fn(cfg, cfg.theta_true[None, :])
        e = np.abs(flux[0]) / 50.0
        cfg.obs_eflux = e
        cfg.obs_flux = flux[0] + e * np.random.default_rng(3).standard_normal(len(e))
    _built[name] = cfg
    return cfg


def rows(cfg, c):
    ix = {p: cfg.fitpars_i.index(p) for p in ('Vrad', 'Vrot')}
    out = []
    for vrad, vrot in [(None, None), (None, 0.0), (0.0, None), (250.0, None), (-250.0, None), (None, VROT_WIDE)]:
        r = cfg.theta_true.copy()
        if vrad is not None:
            r[ix['Vrad']] = vrad
        if vrot is not None:
            r[ix['Vrot']] = vrot
        out.append(r)
    if c['win'] == 'full':
        # the blue end of the grid leaves the mask by exactly one pixel: nM = n - 1 (2^(L-1) on the 2^(L-1) + 1 grids)
        w = cfg.spec.wavelength
        pad = 20.0 / (O.FWHM_FACTOR_FIT * cfg.theta_true[cfg.fitpars_i.index('Inst_R')])
        r = cfg.theta_true.copy()
        r[ix['Vrad']] = O.SPEEDOFLIGHT * (cfg.obs_wave.min() / w[0] * (1.0 - pad) * math.sqrt(w[0] / w[1]) - 1.0)
        out.append(r)
    if c.get('sweep'):
        for v in np.linspace(-1.5, 1.5, 13):
            r = cfg.theta_true.copy()
            r[ix['Vrad']] = v
            out.append(r)
    th = np.concatenate([np.array(out), cfg.draw(4, seed=len(c['name']))])
    return np.ascontiguousarray(th)


def mask_width(cfg, theta):
    """nM of one row: the oracle's mask_wave on the Doppler-shifted grid (predictspec.py:243-263)."""
    p = dict(zip(cfg.fitpars_i, theta))
    w = cfg.spec.wavelength
    if p['Vrad'] != 0.0:
        w = w * (1.0 + p['Vrad'] / O.SPEEDOFLIGHT)
    return int(O._mask(w, O.FWHM_FACTOR_FIT * p['Inst_R'], cfg.obs_wave).sum())


def log2_of(n):
    return int(math.ceil(math.log2(n)))


def stage2_branch(kernel, L, l2):
    """Which stage-2 transform a row with log2 N2 = l2 takes (tail_fast.cuh, tail_cluster.cuh, tail_general.cuh)."""
    if kernel == 'split':
        return {16: 'split', 15: 'ct', 14: 'ct'}.get(l2, 'runtime')
    if kernel == 'cluster':
        return 'cluster' if l2 >= L - 1 else 'runtime'
    LA = max(10, min(L, 15))
    return 'ct' if l2 in (LA, LA - 1) else 'runtime'


def cells():
    """Every (config, kernel, L, nM) the matrix evaluates."""
    out = []
    for c in CONFIGS:
        cfg = build(c['name'])
        L = log2_of(len(cfg.spec.wavelength))
        for th in rows(cfg, c):
            nm = mask_width(cfg, th)
            for k in kernels(c):
                out.append((c['name'], k, L, nm))
    return out


def test_matrix_covers_every_path():
    """CPU: the shapes land on the branches they are meant for."""
    cs = cells()
    seen = {(k, L, log2_of(nm)) for _, k, L, nm in cs if nm >= 17}
    print('(kernel, log2N1, log2N2) cells:', sorted(seen))
    for c in CONFIGS:
        assert log2_of(n_pixels(c)) == c['L'] and len(build(c['name']).spec.wavelength) == n_pixels(c)
    # every fast-tail instantiation, with and without the polynomial, on n = 2^L and n = 2^(L-1) + 1
    for L in range(10, 17):
        at = [c for c in CONFIGS if c['L'] == L and c.get('grid') != 'linear']
        assert {c['npoly'] > 0 for c in at} == {False, True}, L
        assert {n_pixels(c) for c in at} >= {1 << L, (1 << (L - 1)) + 1}, L
    # both compile-time branches and the runtime plan at every L, on every kernel
    for L in range(10, 17):
        for k in (['cluster', 'split'] if L == 16 else ['fast', 'cluster', 'general'] if L == 15 else ['fast', 'general']):
            got = {l2 for kk, LL, l2 in seen if kk == k and LL == L}
            assert {L, L - 1} <= got, (k, L, got)
            assert any(stage2_branch(k, L, l2) == 'runtime' for l2 in got), (k, L, got)
    # the split kernel's stage 2 below N1 (compile-time 32768 / 16384, runtime below)
    assert {l2 for k, L, l2 in seen if k == 'split'} >= {16, 15, 14, 13}
    # every runtime plan size, log2 N2 = 5 .. 14
    rt = {l2 for k, L, l2 in seen if stage2_branch(k, L, l2) == 'runtime'}
    assert rt >= set(range(5, 15)), sorted(rt)
    # mask widths on both sides of a power of two at every L, and the 16 / 17 edge
    nms = {(L, nm) for _, _, L, nm in cs}
    for L in range(10, 17):
        assert (L, 1 << (L - 1)) in nms and (L, (1 << (L - 1)) + 1) in nms, L
        assert (L, 1 << L) in nms, L
    assert {16, 17} <= {nm for _, _, _, nm in cs}
    # general tail alone: <= 512 pixels (log2 N1 8 and 9) and a grid that is not log-uniform
    assert {L for k, L, _ in seen if k == 'general'} >= set(range(8, 16))
    assert any(c.get('grid') == 'linear' for c in CONFIGS)
    # the wide-Vrot row overflows the rotation-table window of the fast kernels (32768 bytes = 2048 intervals)
    for c in CONFIGS:
        if 'general' in kernels(c) and len(kernels(c)) == 1:
            continue
        w = build(c['name']).spec.wavelength
        N1 = 1 << log2_of(len(w))
        dv1 = O.CKMS * (math.log(w[-1]) - math.log(w[0])) / (N1 - 1)
        assert 32.0 * math.pi * VROT_WIDE / dv1 > 2048, c['name']


def _engine(cfg, prec='parity'):
    from thepayne_b200.engine import engine_from_config
    return engine_from_config(cfg, precision=prec)


def _close(a, b):
    fin = np.isfinite(b)
    return np.array_equal(np.isnan(a), ~fin) and np.all(np.abs(a[fin] - b[fin]) <= np.maximum(1e-3, 1e-8 * np.abs(b[fin])))


def _lnl_ok(got, ref, cfg, th, exact):
    """lnL bar, with the float32-emulator floor of far-off rows judged against a float64 emulator (see the docstring)."""
    fin = np.isfinite(ref)
    if not np.array_equal(np.isnan(got), ~fin):
        return False
    far = fin & ~(np.abs(got - ref) <= np.maximum(1e-3, 1e-8 * np.abs(ref)))
    if not far.any():
        return True
    for i in np.nonzero(far)[0]:
        if i not in exact:
            exact[i] = O.OracleLikelihood(cfg, ideal_mlp=True).lnlike_batch(th[i:i + 1])[0]
        e = exact[i]
        if not (abs(got[i] - e) <= abs(ref[i] - e) or abs(got[i] - e) <= max(1e-3, 3e-8 * abs(e))):
            return False
    return True


@pytest.mark.gpu
@pytest.mark.parametrize('name', [c['name'] for c in CONFIGS])
def test_tail_against_oracle(name):
    import torch
    c = BY_NAME[name]
    cfg = build(name)
    th = rows(cfg, c)
    nms = np.array([mask_width(cfg, r) for r in th])
    ok = nms >= 17
    ref_l = np.full(len(th), np.nan)
    ref_f = np.full((len(th), len(cfg.obs_wave)), np.nan)
    ref_l[ok], ref_f[ok], _ = O.OracleLikelihood(cfg).lnlike_batch(th[ok], return_model=True)
    eng = _engine(cfg)
    L = log2_of(len(cfg.spec.wavelength))
    assert eng.query('nfft1') == 1 << L
    assert eng.query('fast_tail') == (1 if 'fast' in kernels(c) or 'cluster' in kernels(c) else 0)
    tht = torch.from_numpy(th).cuda()
    exact = {}
    for k in kernels(c):
        eng.set('fast_tail', 0 if k == 'general' else 1)
        eng.set('tail_cluster', 1 if k == 'cluster' else 0)
        assert eng.query('fast_tail') == (k != 'general') and eng.query('tail_cluster') == (k == 'cluster')
        flux, _, lnl_m = eng.model_batch(tht)
        lnl = eng.lnlike_batch(tht)
        torch.cuda.synchronize()
        f, lm, l = flux.cpu().numpy(), lnl_m.cpu().numpy(), lnl.cpu().numpy()
        assert np.all(np.isnan(f[~ok])) and np.all(np.isnan(l[~ok])), (k, nms)     # nM < 17: NaN (DESIGN §5)
        fin = np.isfinite(ref_f)
        assert np.array_equal(np.isnan(f), ~fin), k
        rel = np.max(np.abs(f[fin] - ref_f[fin]) / np.abs(ref_f[fin]), initial=0.0)
        dl = np.abs(l - ref_l)[np.isfinite(ref_l)]
        print('%s %s: nM %d..%d, max flux rel err %.2e, max |dlnL| %.2e' % (name, k, nms.min(), nms.max(), rel,
                                                                          np.max(dl, initial=0.0)))
        assert rel < 1e-5 and rel <= FLUX_GUARD, (k, rel)
        assert _lnl_ok(lm, ref_l, cfg, th, exact) and _lnl_ok(l, ref_l, cfg, th, exact), (k, lm - ref_l, l - ref_l, ref_l)
        assert eng.query('status') == 0
    eng.close()
