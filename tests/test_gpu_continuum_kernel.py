"""The continuum multiply (continuum.cuh) against a float64 restatement of predictspec.py:208-226.

continuum_kernel takes the continuum net's row, converts it to F_lambda, divides by its nanmedian (an exact radix
selection: odd and even n_c, ties, negative values) and multiplies the emulator's line depth by its np.interp onto the
emulator grid: NaN outside [wc[0], wc[n_c - 1]], the j == n_c - 1 branch on the last continuum wavelength, the
x == x0 branch on an interior one, numpy's slope formula between.

Exact part: both nets have their output-layer weights zeroed, so that their rows are their biases exactly, dyadic
values of few bits (the line-depth forms c - 1 and b - 1 are exact in fp32).  With no Inst_R, Vrot = 0, Vrad = 0 and
the observed pixels on the emulator pixels the model is the multiplied row itself, which must lie within 1 fp32 ulp of
the line depth of the numpy float64 evaluation on the same inputs, NaN patterns identical.  CASES is the matrix as
plain data; `test_matrix_covers_every_branch` (no GPU) recomputes which branch every emulator pixel takes.

End to end: rotation, shift, scalar R and an LSF vector behind the continuum (NaN pixels meet nan_to_num inside the
smoothing stages) against oracle.getspec(cont=...) in parity and simt modes at the 5e-7 bar of test_gpu_f3.py.
"""
import numpy as np
import pytest

from oracle import payne_oracle as O
from thepayne_b200 import synth

LABELS = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]']
PATTERNS = ['equal', 'halves', 'negative', 'mixed', 'outlier']
GEOMETRIES = ['inside', 'last_on_pixel', 'on_pixels', 'wider', 'coarse6', 'fine2']
# (n_c, geometry, pattern)
CASES = [(32, 'inside', 'halves'), (33, 'last_on_pixel', 'equal'), (32, 'on_pixels', 'mixed'), (32, 'wider', 'negative'),
         (255, 'coarse6', 'outlier'), (256, 'fine2', 'halves'), (257, 'on_pixels', 'negative'),
         (256, 'last_on_pixel', 'mixed'), (255, 'inside', 'equal'), (1000, 'coarse6', 'halves'),
         (1000, 'wider', 'outlier'), (4099, 'fine2', 'mixed'), (4099, 'on_pixels', 'equal'), (33, 'fine2', 'outlier'),
         (257, 'wider', 'halves'), (33, 'inside', 'negative')]
_W = {}


def emulator_wave():
    if 'w' not in _W:
        _W['w'] = synth.ann_wavegrid(5140.0, 5230.0, 50000.0)
    return _W['w']


def cont_wave(n_c, geometry):
    w, _ = emulator_wave()
    n = len(w)
    dw = (w[-1] - w[0]) / (n - 1)
    mid = 0.5 * (w[0] + w[-1])
    if geometry == 'inside':
        return np.linspace(w[n // 8] + 0.3 * dw, w[7 * n // 8] - 0.3 * dw, n_c)
    if geometry == 'last_on_pixel':                    # linspace ends exactly on its stop
        return np.linspace(w[n // 8] + 0.3 * dw, w[3 * n // 4], n_c)
    if geometry == 'on_pixels':
        return w[np.round(np.linspace(n // 10, n - 1 - n // 10, n_c)).astype(int)]
    if geometry == 'wider':
        return np.linspace(w[0] - 2.0, w[-1] + 2.0, n_c)
    step = 6.0 * dw if geometry == 'coarse6' else 0.5 * dw
    return mid + step * (np.arange(n_c) - (n_c - 1) / 2.0) + 0.37 * dw


def cont_values(n_c, pattern):
    j = np.arange(n_c)
    if pattern == 'equal':
        v = np.full(n_c, 1.5)
    elif pattern == 'halves':
        v = np.where(j < n_c // 2, 1.25, 1.75)
    elif pattern == 'negative':
        v = -(1.0 + (j % 4) / 4.0)
    elif pattern == 'mixed':
        v = np.where(j % 2 == 0, 1.0 + (j % 8) / 8.0, -(0.5 + (j % 4) / 8.0))
    else:
        v = np.full(n_c, 1.0)
        v[n_c // 3] = 1024.0
    return v.astype(np.float32)


def _zeroed(net, bias):
    """the net with its output layer zeroed: its row is `bias` exactly"""
    net.weights[-1] = np.zeros_like(net.weights[-1])
    net.biases[-1] = np.asarray(bias, dtype=np.float32)
    return net


def emulators(n_c, geometry, pattern):
    w, rsig = emulator_wave()
    row = (1.0 - np.random.default_rng(1).integers(0, 32, len(w)) / 64.0).astype(np.float32)
    spec = _zeroed(synth.make_specnet(4, 16, w, rsig, seed=1), row)
    cont = _zeroed(synth.make_specnet(4, 8, cont_wave(n_c, geometry), rsig, seed=2), cont_values(n_c, pattern))
    return spec, cont


def reference_depth(spec, cont):
    """predictspec.py:208-226 in float64 on the nets' fp32 rows: the multiplied line depth before its fp32 rounding"""
    wc, w = cont.wavelength, spec.wavelength
    modcont = cont.biases[-1].astype(np.float64) * (O.SPEEDOFLIGHT / ((wc * 1E-8) ** 2.0))
    modcont = modcont / np.nanmedian(modcont)
    ci = np.interp(w, wc, modcont, right=np.nan, left=np.nan)
    return (1.0 + (spec.biases[-1].astype(np.float64) - 1.0)) * ci - 1.0


def branches(spec, cont):
    """which branch of continuum_kernel every emulator pixel takes"""
    wc, w = cont.wavelength, spec.wavelength
    j = np.searchsorted(wc, w, side='right') - 1
    out = np.where((w < wc[0]) | (w > wc[-1]), 'nan', 'slope')
    on = (j >= 0) & (j < len(wc)) & (out != 'nan')
    out[on & (j == len(wc) - 1)] = 'last'
    out[on & (j < len(wc) - 1) & (wc[np.clip(j, 0, len(wc) - 1)] == w)] = 'on_x0'
    return set(out)


def test_matrix_covers_every_branch():
    """CPU: odd and even n_c around 256, every pattern and geometry, and every branch of the interpolation."""
    ncs = {c[0] for c in CASES}
    print('n_c:', sorted(ncs))
    assert {32, 33, 255, 256, 257, 1000, 4099} <= ncs
    assert {c[1] for c in CASES} == set(GEOMETRIES) and {c[2] for c in CASES} == set(PATTERNS)
    seen = {}
    for c in CASES:
        spec, cont = emulators(*c)
        b = branches(spec, cont)
        for k in b:
            seen.setdefault(k, []).append(c)
        assert np.all(np.diff(cont.wavelength) > 0), c
        if c[1] in ('inside', 'last_on_pixel', 'on_pixels'):
            assert 'nan' in b, c
        if c[1] == 'last_on_pixel':
            assert 'last' in b, c
        if c[1] == 'on_pixels':
            assert 'on_x0' in b and 'last' in b, c
        if c[1] == 'wider':
            assert b == {'slope'} or b == {'slope', 'on_x0'}, c
        # the line-depth forms are exact in fp32, and every continuum value is its own
        v = cont_values(c[0], c[2]).astype(np.float64)
        assert np.array_equal(np.float32(v - 1.0).astype(np.float64), v - 1.0)
    print('branches:', sorted(seen))
    assert set(seen) == {'nan', 'last', 'on_x0', 'slope'}
    # even counts average the two middle values: they differ on the 'halves' and 'mixed' rows
    for c in CASES:
        if c[0] % 2 == 0 and c[2] in ('halves', 'mixed'):
            spec, cont = emulators(*c)
            m = np.sort(cont.biases[-1].astype(np.float64) * (O.SPEEDOFLIGHT / ((cont.wavelength * 1E-8) ** 2.0)))
            assert m[c[0] // 2 - 1] != m[c[0] // 2], c


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES, ids=['%d_%s_%s' % c for c in CASES])
def test_continuum_multiply_exact(case):
    import torch
    from thepayne_b200.engine import Engine
    spec, cont = emulators(*case)
    w = spec.wavelength
    eng = Engine(spec=spec, obs_wave=w, obs_flux=np.ones(len(w)), obs_eflux=np.ones(len(w)), fitpars_i=LABELS,
                 fixedpars={'Vrad': 0.0, 'Vrot': 0.0})
    eng.attach_continuum(cont)
    th = np.array([[5770.0, 4.44, 0.0, 0.0], [4500.0, 2.0, -1.0, 0.3]])
    flux = eng.model_batch(torch.from_numpy(th).cuda(), want_mags=False)[0].cpu().numpy()
    ref = reference_depth(spec, cont)
    fin = np.isfinite(ref)
    ulp = np.spacing(np.abs(ref[fin]).astype(np.float32)).astype(np.float64)
    for f in flux:
        assert np.array_equal(np.isnan(f), ~fin), case
        err = np.abs((f[fin] - 1.0) - ref[fin])
        print('%s: max error %.2f fp32 ulp of the line depth' % (case, np.max(err / ulp, initial=0.0)))
        assert np.all(err <= ulp), (case, np.max(err / ulp))
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize('prec', ['parity', 'simt'])
@pytest.mark.parametrize('geometry', ['inside', 'on_pixels', 'coarse6'])
def test_continuum_end_to_end(prec, geometry):
    """rotation, shift, scalar R and an LSF vector behind the continuum, against oracle.getspec(cont=...)"""
    import torch
    from thepayne_b200.engine import Engine
    w, rsig = emulator_wave()
    spec = synth.make_specnet(4, 16, w, rsig, seed=3)
    n_c = {'inside': 257, 'on_pixels': 256, 'coarse6': 255}[geometry]
    cont = _zeroed(synth.make_specnet(4, 8, cont_wave(n_c, geometry), rsig, seed=2), cont_values(n_c, 'halves'))
    cont.weights[-1] = np.full_like(cont.weights[-1], 1.0 / 64.0)       # a row that depends on the labels again
    n = len(w)
    ow = np.linspace(w[n // 5], w[4 * n // 5], 900)
    lsf = 0.05 + 0.05 * (ow - ow[0]) / (ow[-1] - ow[0])
    rng = np.random.default_rng(5)
    kw = dict(spec=spec, obs_wave=ow, obs_flux=1.0 + 0.02 * rng.standard_normal(len(ow)), obs_eflux=np.full(len(ow), 0.02),
              precision=prec)
    scalar = Engine(fitpars_i=LABELS + ['Vrad', 'Vrot', 'Inst_R'], **kw)
    vec = Engine(fitpars_i=LABELS + ['Vrad', 'Vrot'], fixedpars={'Inst_R': lsf}, **kw)
    th = np.array([[5770.0, 4.44, 0.0, 0.0, 0.0, 0.0, 32000.0], [5770.0, 4.44, 0.0, 0.0, 0.5, 3.0, 32000.0],
                   [6200.0, 4.0, -0.05, 0.05, -40.0, 25.0, 30000.0], [5100.0, 4.8, 0.05, -0.05, 120.0, 80.0, 36000.0]])
    net, cnet = O.make_net(spec), O.make_net(cont)
    worst = 0.0
    for eng, lsf_or_none in ((scalar, None), (vec, lsf)):
        eng.attach_continuum(cont)
        t = th if lsf_or_none is None else np.ascontiguousarray(th[:, :6])
        flux = eng.model_batch(torch.from_numpy(t).cuda(), want_mags=False)[0].cpu().numpy()
        for i, r in enumerate(th):
            inst = 2.355 * r[6] if lsf_or_none is None else lsf
            _, fr = O.getspec(net, spec, *r[:4], np.nan, r[5], r[4], inst, ow, cont=(cnet, cont))
            assert np.array_equal(np.isnan(flux[i]), np.isnan(fr)), (i, lsf_or_none is None)
            ok = np.isfinite(fr)
            assert ok.sum() > len(ow) // 2
            err = np.max(np.abs(flux[i][ok] - fr[ok]) / np.abs(fr[ok]))
            worst = max(worst, err)
            assert err <= 5e-7, (i, lsf_or_none is None, err)
        assert eng.query('status') == 0
        eng.close()
    print('%s %s: max flux rel err %.2e' % (geometry, prec, worst))
