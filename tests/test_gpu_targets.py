"""Targets: stars observed in several spectra (payne_ctx_set_targets, Engine(stars=[...], targets=[...])).

A target is a run of consecutive stars of an observation set, its members, that share the labels and Vrot.  The core
check is bit-identity (np.array_equal, NaN patterns included): every member's chi2 and model pixels equal what a
single-star engine of that member gives (chi2 = -2 lnL without photometry), and lnL is rebuilt on the host as
-0.5 * ((((chi2_0 + chi2_1) + ...) + chi2_{K-1}) + chi2_sed).  Then the oracle, the refusals, and the star entries of a
context with targets.
"""
import types

import numpy as np
import pytest
import torch

from thepayne_b200 import _lib, synth
from thepayne_b200.engine import Engine
from test_gpu_star_opts import BANDS

pytestmark = pytest.mark.gpu
_INVALID, _UNSUPPORTED = -1, -4
LABELS = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]']

# emulator grids whose transforms are 2^10 .. 2^16 samples (68 pixels per AA at R = 50000)
RANGES = {10: (5140.0, 5152.0), 11: (5140.0, 5165.0), 12: (5140.0, 5190.0), 13: (5140.0, 5240.0),
          14: (5130.0, 5340.0), 15: (5000.0, 5280.0), 16: (4800.0, 5300.0)}
_SPECS = {}


def _emulator(l2):
    if l2 not in _SPECS:
        wave, rsig = synth.ann_wavegrid(*RANGES[l2], 50000.0)
        _SPECS[l2] = synth.make_specnet(4, 64, wave, rsig, seed=0)
    return _SPECS[l2]


# member: (pixel range as fractions of the emulator's coverage, n pixels, Vrad / Inst_R: 'free' or a fixed value)
# target 0: two members with disjoint masks and their own Vrad / Inst_R columns; target 1: one member; target 2: a
# member whose mask covers the other two, one narrow member, one member without instrumental stage (Inst_R = 0);
# target 3: a member whose Inst_R is above the emulator's resolution (NaN) beside a good one.
MEMBERS = [
    [((0.08, 0.45), 900, 'free', 'free'), ((0.55, 0.92), 1100, 'free', 'free')],
    [((0.10, 0.90), 1500, 'free', 'free')],
    [((0.05, 0.95), 1700, 3.0, 'free'), ((0.40, 0.43), 200, 'free', 33000.0), ((0.20, 0.70), 800, -7.0, 0.0)],
    [((0.15, 0.60), 700, 'free', 'free'), ((0.30, 0.80), 600, 'free', 1.0e6)],
]


def _targets(spec, members=MEMBERS, npoly=0, seed=3):
    """stars with their own layouts (the shared labels and Vrot in columns 0-4, the continuum coefficients next,
    then each member's own Vrad / Inst_R columns) and the member counts"""
    w = spec.wavelength
    a, b = w[0], w[-1]
    rng = np.random.default_rng(seed)
    stars, counts, col = [], [], 5 + (npoly + 1 if npoly else 0)
    for tm in members:
        counts.append(len(tm))
        for m, ((f0, f1), n, vrad, instr) in enumerate(tm):
            g = np.linspace(a + f0 * (b - a), a + f1 * (b - a), n)
            npm = npoly + (m % 2) if npoly else 0            # members differ in continuum order
            fit = LABELS + ['Vrot'] + ['pc_%d' % i for i in range(npm)]
            fit += ['pad'] * (col - len(fit))
            fx = {}
            for name, v in (('Vrad', vrad), ('Inst_R', instr)):
                if v == 'free':
                    fit.append(name)
                else:
                    fx[name] = v
            col = len(fit)
            stars.append({'wave': g, 'flux': 1.0 + 0.04 * rng.standard_normal(n), 'eflux': 0.02 + 0.01 * rng.random(n),
                          'fitpars_i': fit, 'fixedpars': fx, 'runbools': [True, False, npm > 0, False]})
    return stars, counts


def _theta(stars, counts, B, seed, vrot_zero=0.3):
    """rows of random targets; every column gets a value that fits the parameter of every star that reads it"""
    rng = np.random.default_rng(seed)
    ndim = max(len(s['fitpars_i']) for s in stars)
    kind = ['pad'] * ndim
    for s in stars:
        for i, p in enumerate(s['fitpars_i']):
            if p != 'pad':
                kind[i] = p
    box = dict(synth._BOX, Vrad=(-30.0, 30.0), Vrot=(0.5, 12.0), Inst_R=(25000.0, 40000.0))
    th = np.zeros((B, ndim))
    for i, p in enumerate(kind):
        if p == 'pad':
            continue
        lo, hi = (0.9, 1.1) if p == 'pc_0' else (-0.05, 0.05) if p.startswith('pc_') else box[p]
        th[:, i] = lo + (hi - lo) * rng.random(B)
    th[rng.random(B) < vrot_zero, 4] = 0.0
    return th, rng.integers(0, len(counts), B).astype(np.int32)


def _single(spec, st, phot=None, obs_phot=None):
    return Engine(spec=spec, obs_wave=st['wave'], obs_flux=st['flux'], obs_eflux=st['eflux'], fitpars_i=st['fitpars_i'],
                  fixedpars=st['fixedpars'], runbools=st['runbools'] + [False], precision=_single.prec)


_single.prec = 'parity'


def _reference(spec, stars, counts, th, tgt, settings, flux_too):
    """per-row member chi2 (-2 lnL of the members' single-star engines), members' model rows, host-rebuilt lnL"""
    first = np.concatenate([[0], np.cumsum(counts)])
    B, K = len(th), max(counts)
    chi2 = np.full((B, K), np.nan)
    nf = max(sum(len(stars[k]['wave']) for k in range(first[t], first[t + 1])) for t in range(len(counts)))
    flux = np.full((B, nf), np.nan)
    for k, st in enumerate(stars):
        one = _single(spec, st)
        for key, v in settings.items():
            if key == 'continuum':
                one.attach_continuum(_emulator(12))
            else:
                one.set(key, v)
        t = np.searchsorted(first, k, side='right') - 1
        m = k - first[t]
        rows = np.nonzero(tgt == t)[0]
        if not len(rows):
            continue
        sub = np.ascontiguousarray(th[rows][:, :len(st['fitpars_i'])])
        if flux_too:
            f, _, l = one.model_batch(sub, want_mags=False)
            off = sum(len(stars[j]['wave']) for j in range(first[t], k))
            flux[rows, off:off + len(st['wave'])] = f.cpu().numpy()
            l = l.cpu().numpy()
        else:
            l = one.lnlike_batch(sub)
        chi2[rows, m] = -2.0 * l
        one.close()
    lnl = np.empty(B)
    for p in range(B):
        t = tgt[p]
        tot = chi2[p, 0]
        for m in range(1, counts[t]):
            tot = tot + chi2[p, m]
        lnl[p] = -0.5 * tot
    return chi2, flux, lnl


def _check(spec, stars, counts, B, settings, seed=1):
    eng = Engine(spec=spec, stars=stars, targets=counts, precision=_single.prec,
                 runbools=[True, False, stars[0]['runbools'][2], False, False])
    for key, v in settings.items():
        if key == 'continuum':
            eng.attach_continuum(_emulator(12))
        else:
            eng.set(key, v)
    th, tgt = _theta(stars, counts, B, seed)
    dev = torch.device('cuda', eng.device)
    thd, tgd = torch.from_numpy(th).to(dev), torch.from_numpy(tgt).to(dev)
    # lnL only (the plain final pass when there is no continuum polynomial)
    chi2, _, lnl = _reference(spec, stars, counts, th, tgt, settings, flux_too=False)
    got = eng.lnlike_batch_targets(thd, tgd).cpu().numpy()
    assert np.array_equal(got, lnl, equal_nan=True), np.nonzero(~((got == lnl) | (np.isnan(got) & np.isnan(lnl))))
    assert np.array_equal(eng.lnlike_batch_targets(th, tgt), lnl, equal_nan=True)      # the host entry
    _, c2, _, l2 = eng.model_batch_targets(thd, tgd, want_flux=False, want_mags=False)
    assert np.array_equal(c2.cpu().numpy(), chi2, equal_nan=True)
    assert np.array_equal(l2.cpu().numpy(), lnl, equal_nan=True)
    # with model rows (the model-output final pass)
    chi2, flux, lnl = _reference(spec, stars, counts, th, tgt, settings, flux_too=True)
    f, c2, _, l2 = eng.model_batch_targets(thd, tgd)
    assert np.array_equal(f.cpu().numpy(), flux, equal_nan=True)
    assert np.array_equal(c2.cpu().numpy(), chi2, equal_nan=True)
    assert np.array_equal(l2.cpu().numpy(), lnl, equal_nan=True)
    assert eng.query('status') & 4 == 0
    # a member above the emulator's resolution: lnL NaN, the other member keeps its chi2
    bad = tgt == 3
    if bad.any():
        assert np.all(np.isnan(lnl[bad])) and np.all(np.isfinite(chi2[bad, 0]))
    eng.close()


@pytest.mark.parametrize('l2', [10, 11, 12, 13, 14, 15, 16])
def test_targets_bit_identical_to_single_star_engines(l2):
    spec = _emulator(l2)
    stars, counts = _targets(spec)
    # 65536-sample transforms: targets take the single-CTA split kernel, so the single-star engines do too
    settings = {'max_batch': 150} if l2 <= 12 else {'tail_cluster': 0} if l2 == 16 else {}
    _check(spec, stars, counts, 400 if l2 <= 14 else 160, settings)


@pytest.mark.parametrize('name', ['poly', 'continuum', 'simt', 'grid_cap1', 'grid_cap2', 'grid_cap3'])
def test_targets_variants(name):
    spec = _emulator(12)
    stars, counts = _targets(spec, npoly=2 if name == 'poly' else 0)
    settings = {'max_batch': 128}
    if name == 'continuum':
        settings['continuum'] = 1
    if name.startswith('grid_cap'):
        settings['tail_grid_cap'] = int(name[-1])
    _single.prec = 'simt' if name == 'simt' else 'parity'
    try:
        _check(spec, stars, counts, 300, settings, seed=7)
    finally:
        _single.prec = 'parity'


def test_one_member_targets_equal_the_star_entry():
    spec = _emulator(12)
    stars, _ = _targets(spec)
    counts = [1] * len(stars)
    eng = Engine(spec=spec, stars=stars, targets=counts)
    th, tgt = _theta(stars, counts, 500, 11)
    dev = torch.device('cuda', eng.device)
    thd, tgd = torch.from_numpy(th).to(dev), torch.from_numpy(tgt).to(dev)
    assert np.array_equal(eng.lnlike_batch_targets(thd, tgd).cpu().numpy(), eng.lnlike_batch(thd, tgd).cpu().numpy(),
                          equal_nan=True)
    f1, _, _, l1 = eng.model_batch_targets(thd, tgd)
    f2, _, l2 = eng.model_batch(thd, tgd)
    assert np.array_equal(l1.cpu().numpy(), l2.cpu().numpy(), equal_nan=True)
    assert np.array_equal(f1.cpu().numpy(), f2.cpu().numpy(), equal_nan=True)


def test_star_entries_unchanged_by_targets():
    spec = _emulator(12)
    stars, counts = _targets(spec)
    plain = Engine(spec=spec, stars=stars)
    grouped = Engine(spec=spec, stars=stars, targets=counts)
    th, _ = _theta(stars, counts, 300, 5)
    star = np.random.default_rng(2).integers(0, len(stars), 300).astype(np.int32)
    dev = torch.device('cuda', plain.device)
    thd, sd = torch.from_numpy(th).to(dev), torch.from_numpy(star).to(dev)
    for a, b in zip(plain.model_batch(thd, sd, want_mags=False), grouped.model_batch(thd, sd, want_mags=False)):
        if a is None:
            continue
        assert np.array_equal(a.cpu().numpy(), b.cpu().numpy(), equal_nan=True)
    assert np.array_equal(plain.lnlike_batch(th, star), grouped.lnlike_batch(th, star), equal_nan=True)


def test_photometry_of_the_first_member():
    """chi2_sed from the first member's magnitudes: lnL = -0.5 (sum of the members' chi2 + chi2_sed), chi2_sed being
    -2 lnL of a photometry-only engine"""
    spec = _emulator(12)
    net = synth.make_photnet(BANDS, H=16)
    stars, counts = _targets(spec)
    phot = {bd: (6.0 + 0.1 * i, 0.05) for i, bd in enumerate(BANDS)}
    first = np.concatenate([[0], np.cumsum(counts)])
    ndim = max(len(s['fitpars_i']) for s in stars)
    for t in range(len(counts)):                         # the first members' photometry columns after everything else
        st = stars[first[t]]
        st['phot'] = phot
        st['fitpars_i'] = st['fitpars_i'] + ['pad'] * (ndim - len(st['fitpars_i'])) + ['log(A)', 'Av']
        st['runbools'] = [True, True, False, True]
    eng = Engine(spec=spec, phot=net, stars=stars, targets=counts)
    th, tgt = _theta(stars, counts, 300, 9)
    specstars = [dict(s, fitpars_i=[p for p in s['fitpars_i'] if p not in ('log(A)', 'Av')],
                      runbools=[True, False, False, False]) for s in stars]
    chi2, _, _ = _reference(spec, specstars, counts, th, tgt, {}, flux_too=False)
    sed = np.empty(len(th))
    for t in range(len(counts)):
        fit = stars[first[t]]['fitpars_i']
        rows = np.nonzero(tgt == t)[0]
        po = Engine(phot=net, obs_phot=phot, fitpars_i=fit, runbools=[False, True, False, True, False])
        sed[rows] = -2.0 * po.lnlike_batch(np.ascontiguousarray(th[rows][:, :len(fit)]))
    want = np.empty(len(th))
    for p in range(len(th)):
        tot = chi2[p, 0]
        for m in range(1, counts[tgt[p]]):
            tot = tot + chi2[p, m]
        want[p] = -0.5 * (tot + sed[p])
    assert np.array_equal(eng.lnlike_batch_targets(th, tgt), want, equal_nan=True)


def test_member_flux_vs_oracle():
    """each member's model spectrum against the oracle's single-spectrum evaluation (1e-5 relative)"""
    from oracle import payne_oracle as O
    spec = _emulator(12)
    w = spec.wavelength
    a, b = w[0], w[-1]
    fit = LABELS + ['Vrot']
    rng = np.random.default_rng(8)
    stars = []
    for (f0, f1), vrad, instr in (((0.1, 0.5), 5.0, 32000.0), ((0.45, 0.9), -12.0, 36000.0)):
        g = np.linspace(a + f0 * (b - a), a + f1 * (b - a), 800)
        stars.append({'wave': g, 'flux': 1.0 + 0.03 * rng.standard_normal(len(g)), 'eflux': np.full(len(g), 0.02),
                      'fixedpars': {'Vrad': vrad, 'Inst_R': instr}})
    eng = Engine(spec=spec, stars=stars, fitpars_i=fit, targets=[2])
    th = np.array([[5770.0, 4.44, 0.0, 0.0, 3.0], [4600.0, 4.7, -0.08, 0.05, 0.0], [6300.0, 4.1, 0.05, -0.02, 9.0]])
    f, c2, _, lnl = eng.model_batch_targets(th, np.zeros(3, np.int32))
    f, c2 = f.cpu().numpy(), c2.cpu().numpy()
    off = 0
    for m, st in enumerate(stars):
        cfg = types.SimpleNamespace(spec=spec, phot=None, runbools=[True, False, False, False, False], fitpars_i=fit,
                                    fixedpars=st['fixedpars'], obs_wave=st['wave'], obs_flux=st['flux'],
                                    obs_eflux=st['eflux'])
        lo, fo, _ = O.OracleLikelihood(cfg).lnlike_batch(th, return_model=True)
        mine = f[:, off:off + len(st['wave'])]
        assert np.array_equal(np.isnan(mine), np.isnan(fo))
        assert np.nanmax(np.abs(mine - fo) / np.abs(fo)) <= 1e-5
        assert np.all(np.abs(-0.5 * c2[:, m] - lo) <= np.maximum(1e-3, 1e-5 * np.abs(lo)))
        off += len(st['wave'])


def test_refusals():
    spec = _emulator(12)
    stars, counts = _targets(spec)
    eng = Engine(spec=spec, stars=stars)
    th, tgt = _theta(stars, counts, 64, 4)
    dev = torch.device('cuda', eng.device)
    # no targets yet
    with pytest.raises(ValueError):
        eng.lnlike_batch_targets(th, tgt)
    r = eng.lib.payne_lnlike_batch_targets_host(eng._ctx, th.ctypes.data, tgt.ctypes.data, 64, th.shape[1],
                                                np.empty(64).ctypes.data)
    assert r == _INVALID
    # first[] rules
    for first in ([1, 2, 3, 6, 8], [0, 2, 2, 6, 8], [0, 2, 3, 6, 7]):
        f = np.array(first, np.int32)
        assert eng.lib.payne_ctx_set_targets(eng._ctx, f.ctypes.data, 4) == _INVALID
    # labels / Vrot must resolve alike
    for name, val in (('Teff', 5000.0), ('Vrot', 2.0), ('Vmic', 1.5)):
        st2 = [dict(s) for s in stars]
        st2[1] = dict(st2[1], fitpars_i=[p if p != name else 'pad' for p in st2[1]['fitpars_i']],
                      fixedpars=dict(st2[1]['fixedpars'], **{name: val}))
        if name == 'Vmic':                               # fixed in both, to different values
            st2[0] = dict(st2[0], fixedpars=dict(st2[0]['fixedpars'], Vmic=1.0))
        with pytest.raises(_lib.PayneError, match='differs from the first member'):
            Engine(spec=spec, stars=st2, targets=counts)
    # photometry on a member other than the first
    net = synth.make_photnet(BANDS, H=16)
    st2 = [dict(s) for s in stars]
    st2[1] = dict(st2[1], phot={BANDS[0]: (6.0, 0.05)}, runbools=[True, True, False, False])
    with pytest.raises(_lib.PayneError, match='photometry on a member'):
        Engine(spec=spec, phot=net, stars=st2, targets=counts)
    # LSF vectors, a grid that is not log-uniform
    lsf = [dict(s, fixedpars=dict(s['fixedpars'], Inst_R=np.full(len(s['wave']), 0.04))) for s in stars]
    with pytest.raises(_lib.PayneError, match='LSF'):
        Engine(spec=spec, stars=lsf, targets=counts)
    lin = synth.make_specnet(4, 64, np.linspace(5140.0, 5190.0, 3000), spec.resolution, seed=0)
    with pytest.raises(_lib.PayneError, match='fast tail'):
        Engine(spec=lin, stars=_targets(lin)[0], targets=counts)
    # out-of-range targets: the host entry refuses, the device entry gives NaN and status bit 2
    eng.set_targets(counts)
    bad = tgt.copy()
    bad[[3, 10]] = [len(counts), -1]
    with pytest.raises(_lib.PayneError, match='outside'):
        eng.lnlike_batch_targets(th, bad)
    assert eng.query('status') & 4 == 0
    got = eng.lnlike_batch_targets(torch.from_numpy(th).to(dev), torch.from_numpy(bad).to(dev)).cpu().numpy()
    assert np.isnan(got[3]) and np.isnan(got[10]) and eng.query('status') & 4
    good = np.ones(64, bool)
    good[[3, 10]] = False
    assert np.array_equal(got[good], eng.lnlike_batch_targets(th[good], tgt[good]), equal_nan=True)
    # removing the targets
    eng.set_targets(None)
    assert eng.query('n_targets') == 0
    assert eng.lib.payne_lnlike_batch_targets_host(eng._ctx, th.ctypes.data, tgt.ctypes.data, 64, th.shape[1],
                                                   np.empty(64).ctypes.data) == _INVALID


def test_fused_gather_refusal():
    """targets and the fused all-gather exclude each other, in either order (a gather context holds one star)"""
    spec = _emulator(12)
    st = _targets(spec, members=[[((0.1, 0.9), 800, 'free', 'free')]])[0][0]
    handles = np.zeros(_lib.GATHER_HANDLE_BYTES, np.uint8)
    eng = _single(spec, st)
    assert eng.lib.payne_gather_create(eng._ctx, 1, 0, 16, handles.ctypes.data) == 0
    first = np.array([0, 1], np.int32)
    assert eng.lib.payne_ctx_set_targets(eng._ctx, first.ctypes.data, 1) == _UNSUPPORTED
    eng.close()
    eng = _single(spec, st)
    eng.set_targets([1])
    assert eng.lib.payne_gather_create(eng._ctx, 1, 0, 16, handles.ctypes.data) == 0
    th, tgt = _theta([st], [1], 8, 2)
    with pytest.raises(_lib.PayneError, match='gather'):
        eng.lnlike_batch_targets(th, tgt)
    eng.close()


# ------------------------------------------------------------------ FitPayne with several spectra

TRUTH = {'Teff': 5770.0, 'log(g)': 4.44, '[Fe/H]': 0.0, '[a/Fe]': 0.0, 'Vrad': 0.5, 'Vrot': 3.0,
         'Inst_R_0': 32000.0, 'Inst_R_1': 28000.0, 'pc_0_0': 1.0, 'pc_1_0': 1.0}
ORDERS = [(5150.0, 5163.0), (5167.0, 5180.0)]


def _two_orders(spec, snr=40.0):
    """two echelle orders of the truth with their own resolving power, noise at S/N ~ snr"""
    rng = np.random.default_rng(12)
    fit = LABELS + ['Vrad', 'Vrot', 'Inst_R']
    specs = []
    for s, (lo, hi) in enumerate(ORDERS):
        w = np.linspace(lo, hi, 700)
        one = Engine(spec=spec, obs_wave=w, obs_flux=np.ones(len(w)), obs_eflux=np.ones(len(w)), fitpars_i=fit)
        th = np.array([[TRUTH[p] for p in LABELS + ['Vrad', 'Vrot']] + [TRUTH['Inst_R_%d' % s]]])
        f = one.model_batch(th, want_mags=False)[0].cpu().numpy()[0]
        one.close()
        e = np.abs(f) / snr
        specs.append({'obs_wave': w, 'obs_flux': f + e * rng.standard_normal(len(w)), 'obs_eflux': e,
                      'convertair': False, 'modpoly': True, 'polyorder': 0})
    return specs


def test_multispec_likelihood_is_the_sum_of_single_spectrum_likelihoods():
    from thepayne_b200.fitting.fitstar import FitPayne
    from thepayne_b200.fitting.likelihood import likelihood
    from thepayne_b200.fitting.multispec import MultiSpecLikelihood
    spec = _emulator(12)
    specs = _two_orders(spec)
    pri = {'Vrot': {'fixed': 3.0}}
    f = FitPayne()
    ind = f._setup(inputdict={'spec': specs, 'specANNpath': spec, 'priordict': pri}, verbose=False)
    L = MultiSpecLikelihood(ind['fitargs'], ind['fitpars'], ind['runbools'])
    assert L.fitpars_i == LABELS + ['Vrad', 'Inst_R_0', 'Inst_R_1', 'pc_0_0', 'pc_1_0']
    assert L.ndim == 9 and L.fixedpars == {'Vrot': 3.0}
    rng = np.random.default_rng(3)
    th = np.array([[TRUTH[p] for p in L.fitpars_i]] * 6)
    th[:, 0] += rng.uniform(-200, 200, 6)
    th[:, 4] += rng.uniform(-3, 3, 6)
    th[:, 5:7] += rng.uniform(-3000, 3000, (6, 2))
    th[:, 7:] += rng.uniform(-0.05, 0.05, (6, 2))
    got = L.lnlike_batch(th)
    assert L.parsdict['Inst_R_1'] == th[-1, 6] and L.parsdict['Vrot'] == 3.0
    assert L.lnlikefn(list(th[2])) == got[2]
    c2 = []
    for s, sp in enumerate(specs):
        fa = {'obs_wave_fit': sp['obs_wave'], 'obs_flux_fit': sp['obs_flux'], 'obs_eflux_fit': sp['obs_eflux'],
              'specANNpath': spec, 'NNtype': 'LinNet', 'fixedpars': {'Vrot': 3.0}}
        names = LABELS + ['Vrad', 'Vrot', 'Inst_R', 'pc_0']
        one = likelihood(fa, [names, {n: n != 'Vrot' for n in names}], [True, False, True, False, False], verbose=False)
        cols = [L.fitpars_i.index(p) for p in LABELS + ['Vrad', 'Inst_R_%d' % s, 'pc_%d_0' % s]]
        c2.append(-2.0 * one.lnlike_batch(np.ascontiguousarray(th[:, cols])))
    assert np.array_equal(got, -0.5 * (c2[0] + c2[1]))


def test_fitpayne_two_orders(tmp_path):
    from thepayne_b200.fitting.fitstar import FitPayne
    spec = _emulator(12)
    pri = {'Teff': {'pv_uniform': [5400.0, 6100.0]}, 'log(g)': {'pv_uniform': [4.0, 4.8]},
           '[Fe/H]': {'pv_uniform': [-0.1, 0.1]}, '[a/Fe]': {'pv_uniform': [-0.1, 0.1]},
           'Vrad': {'pv_uniform': [-3.0, 3.0]}, 'Vrot': {'fixed': 3.0},
           'Inst_R_0': {'pv_uniform': [24000.0, 40000.0]}, 'Inst_R_1': {'pv_uniform': [24000.0, 40000.0]}}
    out = str(tmp_path / 'two_orders.dat')
    FitPayne().run(inputdict={'spec': _two_orders(spec), 'specANNpath': spec, 'NNtype': 'LinNet', 'priordict': pri,
                              'output': out, 'sampler': {'samplertype': 'Static', 'samplemethod': 'rwalk',
                                                         'npoints': 40, 'walks': 10, 'delta_logz_final': 0.5,
                                                         'seed': 5, 'maxiter': 6000}}, verbose=False)
    head = open(out).readline().split()
    assert head[1:11] == LABELS + ['Vrad', 'Inst_R_0', 'Inst_R_1', 'pc_0_0', 'pc_1_0', 'Vrot']
    assert 'Inst_R' not in head
    d = np.loadtxt(out, skiprows=1)
    lw = d[:, head.index('log(wt)')] - d[:, head.index('log(z)')][-1]
    w = np.exp(lw - lw.max())
    w /= w.sum()
    for p in LABELS[:3] + ['Vrad', 'Inst_R_0', 'Inst_R_1', 'pc_0_0', 'pc_1_0']:
        x = d[:, head.index(p)]
        mean = np.sum(w * x)
        sd = np.sqrt(np.sum(w * (x - mean) ** 2))
        assert abs(mean - TRUTH[p]) <= 4.0 * sd + 1e-9 * abs(TRUTH[p]), (p, mean, sd, TRUTH[p])
