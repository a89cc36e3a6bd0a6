"""Double-lined binaries (payne_ctx_set_binary, Engine(binary=True)): one spectrum as the flux-weighted sum of two stars.

The anchor is bit-identity (np.array_equal, NaN patterns included): at Rratio = 0 the binary lnL and model equal the
primary's through payne_model_batch_stars (the polynomial / model-output final pass), and each component's spectrum
equals a single-star model of that component's parameters.  Then the reference evaluation (getspec twice), swap symmetry,
observation sets, the refusals, the old entries, and a small FitPayne fit of a synthetic binary.
"""
import types

import numpy as np
import pytest
import torch

from thepayne_b200 import _lib, synth
from thepayne_b200.engine import Engine

pytestmark = pytest.mark.gpu
_INVALID, _UNSUPPORTED = -1, -4
LABELS = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]']
PRIM = LABELS + ['Vrad', 'Vrot', 'Inst_R']
SEC = ['Teff_sec', 'log(g)_sec', 'Vrad_sec', 'Vrot_sec', 'Rratio']
# secondary column -> the primary column it replaces
SWAP = {'Teff_sec': 'Teff', 'log(g)_sec': 'log(g)', 'Vrad_sec': 'Vrad', 'Vrot_sec': 'Vrot'}

# emulator grids whose transforms are 2^10 .. 2^16 samples (68 pixels per AA at R = 50000)
RANGES = {10: (5140.0, 5152.0), 11: (5140.0, 5165.0), 12: (5140.0, 5190.0), 13: (5140.0, 5240.0),
          14: (5130.0, 5340.0), 15: (5000.0, 5280.0), 16: (4800.0, 5300.0)}
_SPECS = {}


def _emulator(l2, kind='LinNet'):
    key = (l2, kind)
    if key not in _SPECS:
        wave, rsig = synth.ann_wavegrid(*RANGES[l2], 50000.0)
        if kind == 'LinNet':
            _SPECS[key] = synth.make_specnet(4, 64, wave, rsig, seed=0)
        elif kind == 'SMLP':
            _SPECS[key] = synth.make_specnet(4, 32, wave, rsig, seed=1, nntype='SMLP')
        else:
            chunk = ((len(wave) + 2) // 3 + 3) // 4 * 4
            _SPECS[key] = synth.make_multinet(4, 32, wave, rsig, chunk, seed=2)
    return _SPECS[key]


def _obs(spec, n=1500, seed=0, frac=(0.05, 0.95)):
    w = spec.wavelength
    a, b = w[0], w[-1]
    g = np.linspace(a + frac[0] * (b - a), a + frac[1] * (b - a), n)
    rng = np.random.default_rng(seed)
    return g, 1.0 + 0.04 * rng.standard_normal(n), 0.02 + 0.01 * rng.random(n)


def _fit(npoly):
    return PRIM + SEC + ['pc_%d' % k for k in range(npoly)]


def _engine(spec, npoly=0, obs=None, prec='parity', fixedpars=None, fit=None):
    w, f, e = _obs(spec) if obs is None else obs
    return Engine(spec=spec, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=_fit(npoly) if fit is None else fit,
                  fixedpars=fixedpars, runbools=[True, False, npoly > 0, False, False], precision=prec, binary=True)


def _theta(B, seed, npoly=0, rratio=(0.3, 0.9), fit=None, vrad_sec=(-60.0, 60.0)):
    fit = _fit(npoly) if fit is None else fit
    rng = np.random.default_rng(seed)
    box = dict(synth._BOX, Teff=(4800.0, 6500.0), Vrad=(-30.0, 30.0), Vrot=(0.5, 12.0), Inst_R=(25000.0, 40000.0),
               Teff_sec=(3800.0, 5500.0), **{'log(g)_sec': (4.3, 5.0)}, Vrad_sec=vrad_sec,
               Vrot_sec=(0.5, 10.0), Rratio=rratio)
    th = np.zeros((B, len(fit)))
    for i, p in enumerate(fit):
        lo, hi = (0.9, 1.1) if p == 'pc_0' else (-0.05, 0.05) if p.startswith('pc_') else box[p]
        th[:, i] = lo + (hi - lo) * rng.random(B)
    for p in ('Vrot', 'Vrot_sec'):
        if p in fit:
            th[rng.random(B) < 0.25, fit.index(p)] = 0.0
    return th


def _swapped(th, fit, primary_only=False):
    """the secondary's values in the primary's columns (and, unless primary_only, the primary's in the secondary's)"""
    out = th.copy()
    for s, p in SWAP.items():
        i, j = fit.index(p), fit.index(s)
        out[:, i] = th[:, j]
        if not primary_only:
            out[:, j] = th[:, i]
    return out


def _np(*ts):
    return [t.cpu().numpy() if t is not None else None for t in ts]


# ------------------------------------------------------------------ bit-identity
@pytest.mark.parametrize('npoly', [0, 3])
@pytest.mark.parametrize('l2', [10, 11, 12, 13, 14, 15, 16])
def test_rratio_zero_is_the_primary_alone(l2, npoly):
    spec = _emulator(l2)
    eng = _engine(spec, npoly)
    # 65536-sample transforms: binaries take the single-CTA split kernel, so the primary's reference does too;
    # small grids: several slabs per call
    if l2 == 16:
        eng.set('tail_cluster', 0)
    if l2 <= 12:
        eng.set('max_batch', 150)
    B = 300 if l2 <= 14 else 96
    # (a secondary shifted beyond the pixels' coverage has NaN pixels, and 0 * NaN is NaN: keep a_2 finite)
    th = _theta(B, l2, npoly, rratio=(0.0, 0.0), vrad_sec=(-5.0, 5.0))
    f0, _, l0 = _np(*eng.model_batch(th, want_mags=False))
    f, comp, lnl = _np(*eng.model_batch_binary(th))
    assert np.array_equal(lnl, l0, equal_nan=True)
    assert np.array_equal(f, f0, equal_nan=True)
    assert np.array_equal(eng.lnlike_batch_binary(th), l0, equal_nan=True)          # the host entry
    dev = torch.device('cuda', eng.device)
    assert np.array_equal(eng.lnlike_batch_binary(torch.from_numpy(th).to(dev)).cpu().numpy(), l0, equal_nan=True)
    if npoly == 0:
        assert np.array_equal(comp[:, 0], f0, equal_nan=True)
    assert np.isfinite(l0).mean() > 0.9 and eng.query('status') == 0
    eng.close()


def test_rratio_zero_simt():
    spec = _emulator(12)
    eng = _engine(spec, 2, prec='simt')
    th = _theta(200, 5, 2, rratio=(0.0, 0.0))
    f0, _, l0 = _np(*eng.model_batch(th, want_mags=False))
    f, _, lnl = _np(*eng.model_batch_binary(th))
    assert np.array_equal(lnl, l0, equal_nan=True) and np.array_equal(f, f0, equal_nan=True)
    eng.close()


@pytest.mark.parametrize('l2', [12, 16])
def test_each_component_alone(l2):
    """comp[:, c] has the bits of a single-star model of component c; rows with Vrot_sec = 0, Vrad_sec = 0, Inst_R = 0
    (plain interpolation, NaN outside the coverage) and an Inst_R above the emulator's resolution"""
    spec = _emulator(l2)
    w = spec.wavelength
    obs = _obs(spec, n=1200, seed=3, frac=(-0.05, 1.05))     # pixels outside the emulator's coverage
    eng = _engine(spec, 0, obs=obs)
    if l2 == 16:
        eng.set('tail_cluster', 0)
    fit = _fit(0)
    th = _theta(160, 11)
    th[0:20, fit.index('Vrot_sec')] = 0.0
    th[20:40, fit.index('Vrad_sec')] = 0.0
    th[40:60, fit.index('Inst_R')] = 0.0
    th[60:70, fit.index('Inst_R')] = 1.0e6
    f, comp, lnl = _np(*eng.model_batch_binary(th))
    a1 = _np(eng.model_batch(th, want_mags=False)[0])[0]
    a2 = _np(eng.model_batch(_swapped(th, fit, primary_only=True), want_mags=False)[0])[0]
    assert np.array_equal(comp[:, 0], a1, equal_nan=True)
    assert np.array_equal(comp[:, 1], a2, equal_nan=True)
    # Inst_R = 0: NaN outside the coverage (more than 1.5 AA beyond it, the largest Doppler shift here);
    # over-resolved: the whole point is NaN
    out = (obs[0] < w[0] - 1.5) | (obs[0] > w[-1] + 1.5)
    assert out.any() and np.all(np.isnan(comp[40:60][:, :, out]))
    assert np.all(np.isnan(f[60:70])) and np.all(np.isnan(lnl[60:70]))
    eng.close()


# ------------------------------------------------------------------ against the reference
@pytest.mark.parametrize('kind', ['LinNet', 'SMLP', 'MultiNet'])
def test_against_reference(kind):
    from binary_oracle import binary_lnlike_batch
    spec = _emulator(11, kind)
    npoly = 2 if kind == 'LinNet' else 0
    obs = _obs(spec, n=900, seed=4)
    eng = _engine(spec, npoly, obs=obs)
    fit = _fit(npoly)
    th = _theta(5, 21, npoly)
    th[1, fit.index('Vrot_sec')] = 0.0
    th[2, fit.index('Vrad_sec')] = 0.0
    f, comp, lnl = _np(*eng.model_batch_binary(th))
    cfg = types.SimpleNamespace(spec=spec, phot=None, runbools=[True, False, npoly > 0, False, False], fitpars_i=fit,
                                fixedpars={}, obs_wave=obs[0], obs_flux=obs[1], obs_eflux=obs[2])
    lo, fo, co = binary_lnlike_batch(cfg, th, return_model=True)
    for mine, ref in ((f, fo), (comp, co)):
        assert np.array_equal(np.isnan(mine), np.isnan(ref))
        assert np.nanmax(np.abs(mine - ref) / np.abs(ref)) <= 1e-5
    assert np.all(np.abs(lnl - lo) <= np.maximum(1e-3, 1e-5 * np.abs(lo))), (lnl, lo)
    eng.close()


def test_swap_symmetry():
    spec = _emulator(12)
    eng = _engine(spec, 2)
    fit = _fit(2)
    th = _theta(64, 8, 2)
    sw = _swapped(th, fit)
    sw[:, fit.index('Rratio')] = 1.0 / th[:, fit.index('Rratio')]
    f, comp, _ = _np(*eng.model_batch_binary(th))
    g, comp2, _ = _np(*eng.model_batch_binary(sw))
    assert np.array_equal(comp[:, 0], comp2[:, 1], equal_nan=True)
    assert np.array_equal(np.isnan(f), np.isnan(g))
    assert np.nanmax(np.abs(f - g) / np.abs(f)) <= 1e-12
    eng.close()


# ------------------------------------------------------------------ observation sets
def test_observation_sets_match_one_star_engines():
    spec = _emulator(12)
    fit = [p for p in _fit(2) if p != 'Inst_R']
    stars = []
    for k, (fr, instr) in enumerate((((0.05, 0.5), 30000.0), ((0.3, 0.95), 36000.0), ((0.1, 0.9), 0.0))):
        w, fl, e = _obs(spec, n=700 + 200 * k, seed=10 + k, frac=fr)
        stars.append({'wave': w, 'flux': fl, 'eflux': e, 'fixedpars': {'Inst_R': instr}})
    eng = Engine(spec=spec, stars=stars, fitpars_i=fit, runbools=[True, False, True, False, False], binary=True)
    th = _theta(240, 13, 2, fit=fit)
    star = np.random.default_rng(1).integers(0, 3, 240).astype(np.int32)
    f, comp, lnl = _np(*eng.model_batch_binary(th, star))
    for k, st in enumerate(stars):
        one = _engine(spec, 2, obs=(st['wave'], st['flux'], st['eflux']), fixedpars=st['fixedpars'], fit=fit)
        rows = np.nonzero(star == k)[0]
        n = len(st['wave'])
        f1, c1, l1 = _np(*one.model_batch_binary(th[rows]))
        assert np.array_equal(lnl[rows], l1, equal_nan=True)
        assert np.array_equal(f[rows][:, :n], f1, equal_nan=True) and np.all(np.isnan(f[rows][:, n:]))
        assert np.array_equal(comp[rows][:, :, :n], c1, equal_nan=True)
        one.close()
    assert np.array_equal(eng.lnlike_batch_binary(th, star), lnl, equal_nan=True)
    # star indices out of range: the host entry refuses, the device entry gives NaN and status bit 2
    bad = star.copy()
    bad[[5, 17]] = [3, -1]
    with pytest.raises(_lib.PayneError, match='outside'):
        eng.lnlike_batch_binary(th, bad)
    assert eng.query('status') & 4 == 0
    dev = torch.device('cuda', eng.device)
    got = eng.lnlike_batch_binary(torch.from_numpy(th).to(dev), torch.from_numpy(bad).to(dev)).cpu().numpy()
    good = np.ones(240, bool)
    good[[5, 17]] = False
    assert np.all(np.isnan(got[~good])) and eng.query('status') & 4
    assert np.array_equal(got[good], lnl[good], equal_nan=True)
    # star NULL means star 0
    assert np.array_equal(eng.lnlike_batch_binary(th[:8]), eng.lnlike_batch_binary(th[:8], np.zeros(8, np.int32)))
    eng.close()


# ------------------------------------------------------------------ refusals and the old entries
def _bin_struct(fit, **kw):
    from thepayne_b200.engine import _binary
    b = _binary(fit, {})
    for k, v in kw.items():
        setattr(b, k, v)
    return b


def test_refusals():
    import ctypes as C
    spec = _emulator(12)
    fit = _fit(0)
    w, f, e = _obs(spec)
    plain = Engine(spec=spec, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=fit)
    th = _theta(8, 1)
    out = np.empty(8)
    # no binary set
    assert plain.lib.payne_lnlike_batch_binary_host(plain._ctx, th.ctypes.data, None, 8, th.shape[1],
                                                    out.ctypes.data) == _INVALID
    assert b'no binary' in plain.lib.payne_last_error() and plain.query('binary') == 0
    # invalid descriptions
    cases = []
    b = _bin_struct(fit)
    b.col[_lib.PAR_INDEX['Inst_R']] = 0
    cases.append((b, b'Inst_R is shared'))
    b = _bin_struct(fit)
    b.fixed[_lib.PAR_INDEX['Av']] = 0.1
    cases.append((b, b'Av is shared'))
    b = _bin_struct(fit)
    b.col[_lib.PAR_INDEX['Vrad']] = len(fit)
    cases.append((b, b'outside'))
    cases.append((_bin_struct(fit, rratio_col=len(fit)), b'outside'))
    cases.append((_bin_struct(fit, rratio_col=-1, rratio_fixed=float('nan')), b'Rratio'))
    for b, msg in cases:
        assert plain.lib.payne_ctx_set_binary(plain._ctx, C.byref(b)) == _INVALID
        assert msg in plain.lib.payne_last_error(), plain.lib.payne_last_error()
    assert plain.query('binary') == 0
    plain.set_binary(fixedpars={'Rratio': 0.5}, fitpars_i=PRIM)       # a fixed Rratio, the secondary all primary
    assert plain.query('binary') == 1
    plain.set_binary(False)
    assert plain.query('binary') == 0
    plain.close()
    # unsupported contexts, at set time
    from test_gpu_star_opts import BANDS
    net = synth.make_photnet(BANDS, H=16)
    with pytest.raises(_lib.PayneError, match='photometry'):
        Engine(spec=spec, phot=net, obs_wave=w, obs_flux=f, obs_eflux=e, obs_phot={b: (6.0, 0.05) for b in BANDS},
               fitpars_i=fit + ['log(R)', 'Dist', 'Av'], runbools=[True, True, False, False, False], binary=True)
    with pytest.raises(_lib.PayneError, match='LSF'):
        Engine(spec=spec, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=[p for p in fit if p != 'Inst_R'],
               fixedpars={'Inst_R': np.full(len(w), 0.04), 'Rratio': 0.5}, binary=True)
    stars = [{'wave': w, 'flux': f, 'eflux': e}, {'wave': w[:500], 'flux': f[:500], 'eflux': e[:500]}]
    with pytest.raises(_lib.PayneError, match='targets'):
        Engine(spec=spec, stars=stars, fitpars_i=fit, targets=[2], binary=True)
    with pytest.raises(_lib.PayneError, match='per-star layouts'):
        Engine(spec=spec, stars=[dict(stars[0]), dict(stars[1], fitpars_i=fit[::-1])], fitpars_i=fit, binary=True)
    lin = synth.make_specnet(4, 64, np.linspace(5140.0, 5190.0, 3000), spec.resolution, seed=0)
    with pytest.raises(_lib.PayneError, match='fast tail'):
        _engine(lin)
    eng = Engine(spec=spec, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=fit)
    eng.attach_continuum(_emulator(12))
    with pytest.raises(_lib.PayneError, match='continuum'):
        eng.set_binary()
    eng.close()
    handles = np.zeros(_lib.GATHER_HANDLE_BYTES, np.uint8)
    eng = Engine(spec=spec, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=fit)
    assert eng.lib.payne_gather_create(eng._ctx, 1, 0, 16, handles.ctypes.data) == 0
    with pytest.raises(_lib.PayneError, match='gather'):
        eng.set_binary()
    eng.close()
    # ... and again when an entry is called after the context changed
    for change, msg in ((lambda x: x.set_lsf(np.full(len(w), 0.04)), 'LSF'),
                        (lambda x: x.attach_continuum(_emulator(12)), 'continuum'),
                        (lambda x: x.set('fast_tail', 0), 'fast tail'),
                        (lambda x: x.lib.payne_gather_create(x._ctx, 1, 0, 16, handles.ctypes.data), 'gather')):
        eng = _engine(spec)
        change(eng)
        with pytest.raises(_lib.PayneError, match=msg):
            eng.lnlike_batch_binary(th)
        with pytest.raises(_lib.PayneError, match=msg):
            eng.model_batch_binary(th)
        eng.close()


def test_old_entries_unchanged_by_a_binary():
    spec = _emulator(13)
    fit = _fit(2)
    obs = _obs(spec, seed=6)
    w, f, e = obs
    plain = Engine(spec=spec, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=fit, runbools=[True, False, True, False])
    binr = _engine(spec, 2, obs=obs)
    th = _theta(300, 2, 2)
    binr.lnlike_batch_binary(th)                                 # the binary workspace exists
    assert np.array_equal(binr.lnlike_batch(th), plain.lnlike_batch(th), equal_nan=True)
    a, _, la = _np(*binr.model_batch(th, want_mags=False))
    b, _, lb = _np(*plain.model_batch(th, want_mags=False))
    assert np.array_equal(a, b, equal_nan=True) and np.array_equal(la, lb, equal_nan=True)
    plain.close()
    binr.close()


def test_removing_marginalisation_keeps_the_binary():
    """binaries and continuum marginalisation share the per-CTA a_j scratch: clearing the one that is off keeps it"""
    spec = _emulator(13)
    eng = _engine(spec, 2)
    th = _theta(300, 4, 2)
    lnl = eng.lnlike_batch_binary(th)
    flux, comp, lm = _np(*eng.model_batch_binary(th))
    eng.set_cont_marg(None)
    assert np.array_equal(eng.lnlike_batch_binary(th), lnl, equal_nan=True)
    f2, c2, l2 = _np(*eng.model_batch_binary(th))
    assert np.array_equal(f2, flux, equal_nan=True) and np.array_equal(c2, comp, equal_nan=True)
    assert np.array_equal(l2, lm, equal_nan=True) and np.isfinite(lnl).any()
    eng.close()


# ------------------------------------------------------------------ the likelihood and a fit
TRUTH = {'Teff': 5900.0, 'log(g)': 4.3, '[Fe/H]': 0.0, '[a/Fe]': 0.0, 'Vrad': -15.0, 'Vrot': 4.0, 'Inst_R': 32000.0,
         'Teff_sec': 4700.0, 'log(g)_sec': 4.6, 'Vrad_sec': 35.0, 'Vrot_sec': 2.0, 'Rratio': 0.8, 'pc_0': 1.0}


def _sb2(spec, snr=80.0):
    """a synthetic SB2 of the truth at S/N ~ snr"""
    rng = np.random.default_rng(12)
    w = np.linspace(5150.0, 5180.0, 1500)
    fit = PRIM + SEC
    one = Engine(spec=spec, obs_wave=w, obs_flux=np.ones(len(w)), obs_eflux=np.ones(len(w)), fitpars_i=fit,
                 binary=True)
    m = _np(one.model_batch_binary(np.array([[TRUTH[p] for p in fit]]))[0])[0][0]
    one.close()
    e = np.abs(m) / snr
    return {'obs_wave': w, 'obs_flux': m + e * rng.standard_normal(len(w)), 'obs_eflux': e, 'convertair': False,
            'modpoly': True, 'polyorder': 0}


def test_binary_likelihood_interface():
    from thepayne_b200.fitting.binary import BinaryLikelihood
    from thepayne_b200.fitting.fitstar import FitPayne
    spec = _emulator(12)
    sp = _sb2(spec)
    f = FitPayne()
    ind = f._setup(inputdict={'spec': sp, 'specANNpath': spec, 'binary': True,
                              'priordict': {'Vrot': {'fixed': 4.0}, 'Vrot_sec': {'fixed': 2.0}}}, verbose=False)
    L = BinaryLikelihood(ind['fitargs'], ind['fitpars'], ind['runbools'], verbose=False)
    assert L.fitpars_i == LABELS + ['Vrad', 'Inst_R', 'Teff_sec', 'log(g)_sec', 'Vrad_sec', 'Rratio', 'pc_0']
    assert L.fixedpars == {'Vrot': 4.0, 'Vrot_sec': 2.0}
    th = np.array([[TRUTH[p] for p in L.fitpars_i]] * 5)
    th[:, 0] += np.linspace(-200.0, 200.0, 5)
    got = L.lnlike_batch(th)
    assert L.parsdict['Vrot_sec'] == 2.0 and L.parsdict['Teff'] == th[-1, 0]
    assert L.lnlikefn(list(th[1])) == got[1]
    assert np.all(np.isfinite(got)) and len(set(got)) == 5
    eng = Engine(spec=spec, obs_wave=sp['obs_wave'], obs_flux=sp['obs_flux'], obs_eflux=sp['obs_eflux'],
                 fitpars_i=L.fitpars_i, fixedpars=L.fixedpars, runbools=[True, False, True, False, False], binary=True)
    assert np.array_equal(eng.lnlike_batch_binary(th), got)
    eng.close()


def test_fitpayne_binary(tmp_path):
    from thepayne_b200.fitting.fitstar import FitPayne
    spec = _emulator(12)
    pri = {'Teff': {'pv_uniform': [5500.0, 6300.0]}, 'log(g)': {'pv_uniform': [4.0, 4.6]},
           '[Fe/H]': {'fixed': 0.0}, '[a/Fe]': {'fixed': 0.0}, 'Vrad': {'pv_uniform': [-25.0, -5.0]},
           'Vrot': {'fixed': 4.0}, 'Inst_R': {'fixed': 32000.0}, 'Teff_sec': {'pv_uniform': [4200.0, 5200.0]},
           'log(g)_sec': {'fixed': 4.6}, 'Vrad_sec': {'pv_uniform': [20.0, 50.0]}, 'Vrot_sec': {'fixed': 2.0},
           'Rratio': {'pv_uniform': [0.5, 1.0]}}
    out = str(tmp_path / 'sb2.dat')
    FitPayne().run(inputdict={'spec': _sb2(spec), 'specANNpath': spec, 'NNtype': 'LinNet', 'priordict': pri,
                              'binary': True, 'output': out,
                              'sampler': {'samplertype': 'Static', 'samplemethod': 'rwalk', 'npoints': 40, 'walks': 10,
                                          'delta_logz_final': 0.5, 'seed': 5, 'maxiter': 6000}}, verbose=False)
    head = open(out).readline().split()
    assert head[1:8] == ['Teff', 'log(g)', 'Vrad', 'Teff_sec', 'Vrad_sec', 'Rratio', 'pc_0']
    for p in ('log(g)_sec', 'Vrot_sec', 'Inst_R'):
        assert p in head
    d = np.loadtxt(out, skiprows=1)
    lw = d[:, head.index('log(wt)')] - d[:, head.index('log(z)')][-1]
    wt = np.exp(lw - lw.max())
    wt /= wt.sum()
    for p in ('Vrad_sec', 'Teff_sec', 'Vrad', 'Teff'):
        x = d[:, head.index(p)]
        mean = np.sum(wt * x)
        sd = np.sqrt(np.sum(wt * (x - mean) ** 2))
        assert abs(mean - TRUTH[p]) <= 4.0 * sd + 1e-9 * abs(TRUTH[p]), (p, mean, sd, TRUTH[p])
