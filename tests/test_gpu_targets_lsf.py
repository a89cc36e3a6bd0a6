"""Targets with LSF vectors: every member of a target broadened by its own LSF vector (PayneStarOpts.lsf) behind one
emulator row and one rotation stage per point.

The core check is the one of test_gpu_targets.py: every member's chi2 and model pixels equal, bit for bit, those of a
single-star LSF engine of that member, and lnL is rebuilt on the host in member order.  Then bad members, the
photometry / continuum / simt variants, one-member targets, the oracle, the refusals and the multi-spectrum fit.
The tests without the gpu mark check the fit setup only.
"""
import types

import numpy as np
import pytest
import torch

from thepayne_b200 import _lib, synth
from thepayne_b200.engine import Engine
from test_gpu_star_opts import BANDS, _lsf
from test_gpu_targets import LABELS, _check, _emulator, _reference, _single, _targets, _theta

_INVALID, _UNSUPPORTED = -1, -4
gpu = pytest.mark.gpu

# member: (pixel range as fractions of the emulator's coverage, n pixels, Vrad: 'free' or a fixed value); every member
# gets its own LSF vector.  Target 0 has four members, target 2 a member with a large |Vrad|.  (_check expects every
# member of these three targets to be good, and target 3, where there is one, to have a bad member.)
MEMBERS = [
    [((0.15, 0.60), 700, 'free'), ((0.30, 0.80), 600, 40.0), ((0.50, 0.70), 300, 'free'), ((0.60, 0.95), 500, 'free')],
    [((0.10, 0.90), 1500, 'free')],
    [((0.05, 0.95), 1700, 3.0), ((0.40, 0.43), 200, 'free'), ((0.20, 0.70), 800, -250.0)],
]
# target 3 of the bad-member set: a member pushed off the emulator grid (mask of no pixel) and one whose LSF needs a
# transform above 32768 samples, between two good ones
BAD = MEMBERS + [[((0.15, 0.60), 700, 'free'), ((0.30, 0.80), 600, 2.0e5), ((0.50, 0.70), 300, 'tiny'),
                  ((0.60, 0.95), 500, 'free')]]


def _lsf_targets(spec, members=MEMBERS, npoly=0, seed=3):
    """the stars of _targets with an LSF vector each in place of Inst_R ('tiny': a vector of 0.001 AA)"""
    plain = [[(r, n, 0.0 if v == 'tiny' else v, 0.0) for r, n, v in tm] for tm in members]
    stars, counts = _targets(spec, plain, npoly=npoly, seed=seed)
    kinds = [v for tm in members for _, _, v in tm]
    for k, (st, v) in enumerate(zip(stars, kinds)):
        st['fixedpars']['Inst_R'] = np.full(len(st['wave']), 0.001) if v == 'tiny' else _lsf(st['wave'], k)
    return stars, counts


def _linear_emulator():
    return synth.make_specnet(4, 64, np.linspace(5140.0, 5190.0, 3000), _emulator(12).resolution, seed=0)


@gpu
@pytest.mark.parametrize('grid,npoly', [(10, 0), (12, 0), (12, 2), (14, 0), (15, 0), ('linear', 2)])
def test_lsf_targets_bit_identical_to_single_star_engines(grid, npoly):
    spec = _linear_emulator() if grid == 'linear' else _emulator(grid)
    stars, counts = _lsf_targets(spec, npoly=npoly)
    _check(spec, stars, counts, 300 if grid in (10, 12, 'linear') else 120, {'max_batch': 128})


@gpu
def test_bad_members():
    """a member off the grid and a member above the largest transform: chi2 and pixels NaN, lnL NaN, the other
    members as in their single-star engines"""
    spec = _emulator(12)
    stars, counts = _lsf_targets(spec, BAD)
    _check(spec, stars, counts, 300, {'max_batch': 128})
    eng = Engine(spec=spec, stars=stars, targets=counts)
    th, _ = _theta(stars, counts, 16, 4)
    tgt = np.full(16, 3, np.int32)
    f, c2, _, _ = eng.model_batch_targets(th, tgt, want_mags=False)
    f, c2 = f.cpu().numpy(), c2.cpu().numpy()
    lnl = eng.lnlike_batch_targets(th, tgt)
    assert np.all(np.isnan(lnl)) and np.all(np.isnan(c2[:, 1:3])) and np.all(np.isfinite(c2[:, [0, 3]]))
    assert np.all(np.isnan(f[:, 700:1600])) and np.all(np.isfinite(f[:, :700])) and np.all(np.isfinite(f[:, 1600:2100]))
    assert eng.query('status') & 1 and not eng.query('status') & 4


@gpu
@pytest.mark.parametrize('name', ['continuum', 'simt'])
def test_lsf_targets_variants(name):
    spec = _emulator(12)
    stars, counts = _lsf_targets(spec)
    settings = {'max_batch': 128}
    if name == 'continuum':
        settings['continuum'] = 1
    _single.prec = 'simt' if name == 'simt' else 'parity'
    try:
        _check(spec, stars, counts, 300, settings, seed=7)
    finally:
        _single.prec = 'parity'


@gpu
def test_photometry_of_the_first_member():
    """lnL = -0.5 (members' chi2 in order + chi2_sed), chi2_sed and the magnitudes those of a photometry-only engine"""
    spec = _emulator(12)
    net = synth.make_photnet(BANDS, H=16)
    stars, counts = _lsf_targets(spec)
    phot = {bd: (6.0 + 0.1 * i, 0.05) for i, bd in enumerate(BANDS)}
    first = np.concatenate([[0], np.cumsum(counts)])
    ndim = max(len(s['fitpars_i']) for s in stars)
    for t in range(len(counts)):
        st = stars[first[t]]
        st['phot'] = phot
        st['fitpars_i'] = st['fitpars_i'] + ['pad'] * (ndim - len(st['fitpars_i'])) + ['log(A)', 'Av']
        st['runbools'] = [True, True, False, True]
    eng = Engine(spec=spec, phot=net, stars=stars, targets=counts)
    th, tgt = _theta(stars, counts, 300, 9)
    specstars = [dict(s, fitpars_i=[p for p in s['fitpars_i'] if p not in ('log(A)', 'Av')],
                      runbools=[True, False, False, False]) for s in stars]
    chi2, _, _ = _reference(spec, specstars, counts, th, tgt, {}, flux_too=False)
    sed, mags = np.empty(len(th)), np.empty((len(th), len(BANDS)))
    for t in range(len(counts)):
        fit = stars[first[t]]['fitpars_i']
        rows = np.nonzero(tgt == t)[0]
        po = Engine(phot=net, obs_phot=phot, fitpars_i=fit, runbools=[False, True, False, True, False])
        sub = np.ascontiguousarray(th[rows][:, :len(fit)])
        sed[rows] = -2.0 * po.lnlike_batch(sub)
        mags[rows] = po.model_batch(sub)[1].cpu().numpy()
    want = np.empty(len(th))
    for p in range(len(th)):
        tot = chi2[p, 0]
        for m in range(1, counts[tgt[p]]):
            tot = tot + chi2[p, m]
        want[p] = -0.5 * (tot + sed[p])
    assert np.array_equal(eng.lnlike_batch_targets(th, tgt), want, equal_nan=True)
    _, c2, m, lnl = eng.model_batch_targets(th, tgt, want_flux=False)
    assert np.array_equal(m.cpu().numpy(), mags)
    assert np.array_equal(c2.cpu().numpy(), chi2, equal_nan=True)
    assert np.array_equal(lnl.cpu().numpy(), want, equal_nan=True)


@gpu
def test_one_member_targets_and_star_entries():
    """one-member targets equal the star entry; setting targets leaves the star entries of an LSF context alone"""
    spec = _emulator(12)
    stars, counts = _lsf_targets(spec)
    th, _ = _theta(stars, counts, 400, 11)
    star = np.random.default_rng(2).integers(0, len(stars), 400).astype(np.int32)
    plain = Engine(spec=spec, stars=stars)
    ones = Engine(spec=spec, stars=stars, targets=[1] * len(stars))
    grouped = Engine(spec=spec, stars=stars, targets=counts)
    dev = torch.device('cuda', ones.device)
    thd, sd = torch.from_numpy(th).to(dev), torch.from_numpy(star).to(dev)
    assert np.array_equal(ones.lnlike_batch_targets(thd, sd).cpu().numpy(), ones.lnlike_batch(thd, sd).cpu().numpy(),
                          equal_nan=True)
    f1, _, _, l1 = ones.model_batch_targets(thd, sd)
    f2, _, l2 = ones.model_batch(thd, sd)
    assert np.array_equal(l1.cpu().numpy(), l2.cpu().numpy(), equal_nan=True)
    assert np.array_equal(f1.cpu().numpy(), f2.cpu().numpy(), equal_nan=True)
    for a, b in zip(plain.model_batch(thd, sd, want_mags=False), grouped.model_batch(thd, sd, want_mags=False)):
        if a is not None:
            assert np.array_equal(a.cpu().numpy(), b.cpu().numpy(), equal_nan=True)
    assert np.array_equal(plain.lnlike_batch(th, star), grouped.lnlike_batch(th, star), equal_nan=True)


@gpu
def test_member_flux_vs_oracle():
    """each member's model spectrum against the oracle's single-spectrum LSF evaluation (1e-5 relative)"""
    from oracle import payne_oracle as O
    spec = _emulator(12)
    w = spec.wavelength
    a, b = w[0], w[-1]
    fit = LABELS + ['Vrot']
    rng = np.random.default_rng(8)
    stars = []
    for k, ((f0, f1), vrad) in enumerate((((0.1, 0.5), 5.0), ((0.45, 0.9), -12.0))):
        g = np.linspace(a + f0 * (b - a), a + f1 * (b - a), 800)
        stars.append({'wave': g, 'flux': 1.0 + 0.03 * rng.standard_normal(len(g)), 'eflux': np.full(len(g), 0.02),
                      'fixedpars': {'Vrad': vrad, 'Inst_R': _lsf(g, k)}})
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
        assert np.all(np.isfinite(mine)) and np.all(np.isfinite(fo))
        assert np.max(np.abs(mine - fo) / np.abs(fo)) <= 1e-5
        assert np.all(np.abs(-0.5 * c2[:, m] - lo) <= np.maximum(1e-3, 1e-5 * np.abs(lo)))
        off += len(st['wave'])


@gpu
def test_refusals():
    spec = _emulator(12)
    stars, counts = _lsf_targets(spec)
    # an Inst_R column beside an LSF vector
    col = [dict(s, fitpars_i=s['fitpars_i'] + ['Inst_R']) for s in stars]
    with pytest.raises(_lib.PayneError, match=r'target 0, member 0: Inst_R in theta column \d+ beside its LSF vector'):
        Engine(spec=spec, stars=col, targets=counts)
    eng = Engine(spec=spec, stars=col)
    first = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    assert eng.lib.payne_ctx_set_targets(eng._ctx, first.ctypes.data, len(counts)) == _INVALID
    eng.close()
    # labels / Vrot must resolve alike
    for name, val in (('Teff', 5000.0), ('Vrot', 2.0)):
        st2 = [dict(s) for s in stars]
        st2[1] = dict(st2[1], fitpars_i=[p if p != name else 'pad' for p in st2[1]['fitpars_i']],
                      fixedpars=dict(st2[1]['fixedpars'], **{name: val}))
        with pytest.raises(_lib.PayneError, match='differs from the first member'):
            Engine(spec=spec, stars=st2, targets=counts)
    # photometry on a member other than the first
    net = synth.make_photnet(BANDS, H=16)
    st2 = [dict(s) for s in stars]
    st2[1] = dict(st2[1], phot={BANDS[0]: (6.0, 0.05)}, runbools=[True, True, False, False])
    with pytest.raises(_lib.PayneError, match='photometry on a member'):
        Engine(spec=spec, phot=net, stars=st2, targets=counts)
    # out-of-range targets: the host entry refuses, the device entry gives NaN and status bit 2
    eng = Engine(spec=spec, stars=stars, targets=counts)
    th, tgt = _theta(stars, counts, 64, 4)
    bad = tgt.copy()
    bad[[3, 10]] = [len(counts), -1]
    with pytest.raises(_lib.PayneError, match='outside'):
        eng.lnlike_batch_targets(th, bad)
    assert eng.query('status') & 4 == 0
    dev = torch.device('cuda', eng.device)
    got = eng.lnlike_batch_targets(torch.from_numpy(th).to(dev), torch.from_numpy(bad).to(dev)).cpu().numpy()
    assert np.isnan(got[3]) and np.isnan(got[10]) and eng.query('status') & 4
    good = np.ones(64, bool)
    good[[3, 10]] = False
    assert np.array_equal(got[good], eng.lnlike_batch_targets(th[good], tgt[good]), equal_nan=True)


@gpu
def test_fused_gather_refusal():
    """LSF targets and the fused all-gather exclude each other, in either order"""
    spec = _emulator(12)
    st = _lsf_targets(spec, members=[[((0.1, 0.9), 800, 'free')]])[0][0]
    handles = np.zeros(_lib.GATHER_HANDLE_BYTES, np.uint8)
    eng = _single(spec, st)
    assert eng.query('lsf') == 1
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


@gpu
def test_lsf_switched_off_needs_the_fast_tail():
    """a one-star context whose LSF vector is switched off after set_targets runs the fast target tail, and on a grid
    without it is refused at call time"""
    spec = _emulator(12)
    st = _lsf_targets(spec, members=[[((0.1, 0.9), 800, 'free')]])[0][0]
    th, tgt = _theta([st], [1], 64, 2)
    eng = _single(spec, st)
    eng.set_targets([1])
    assert np.array_equal(eng.lnlike_batch_targets(th, tgt), eng.lnlike_batch(th), equal_nan=True)
    eng.set_lsf(None)
    assert np.array_equal(eng.lnlike_batch_targets(th, tgt), eng.lnlike_batch(th), equal_nan=True)
    lin = _linear_emulator()
    st = _lsf_targets(lin, members=[[((0.1, 0.9), 800, 'free')]])[0][0]
    eng = _single(lin, st)
    eng.set_targets([1])
    assert np.isfinite(eng.lnlike_batch_targets(th, tgt)).any()
    eng.set_lsf(None)
    with pytest.raises(_lib.PayneError, match='fast tail'):
        eng.lnlike_batch_targets(th, tgt)


# ------------------------------------------------------------------ FitPayne with several spectra and LSF vectors

TRUTH = {'Teff': 5770.0, 'log(g)': 4.44, '[Fe/H]': 0.0, '[a/Fe]': 0.0, 'Vrad': 0.5, 'Vrot': 3.0, 'pc_0_0': 1.0,
         'pc_1_0': 1.0}
ORDERS = [(5150.0, 5163.0), (5167.0, 5180.0)]


def _order_lsf(s):
    w = np.linspace(*ORDERS[s], 700)
    return w, _lsf(w, 3 * s)


def _two_orders(spec, snr=40.0):
    """two echelle orders of the truth, each broadened by its own LSF vector, noise at S/N ~ snr"""
    rng = np.random.default_rng(12)
    fit = LABELS + ['Vrad', 'Vrot']
    specs = []
    for s in range(len(ORDERS)):
        w, lsf = _order_lsf(s)
        one = Engine(spec=spec, obs_wave=w, obs_flux=np.ones(len(w)), obs_eflux=np.ones(len(w)), fitpars_i=fit,
                     fixedpars={'Inst_R': lsf})
        f = one.model_batch(np.array([[TRUTH[p] for p in fit]]), want_mags=False)[0].cpu().numpy()[0]
        one.close()
        e = np.abs(f) / snr
        specs.append({'obs_wave': w, 'obs_flux': f + e * rng.standard_normal(len(w)), 'obs_eflux': e,
                      'convertair': False, 'modpoly': True, 'polyorder': 0})
    return specs


def _setup_specs():
    """two orders without the GPU (flux of ones), for the fit setup"""
    return [{'obs_wave': _order_lsf(s)[0], 'obs_flux': np.ones(700), 'obs_eflux': np.full(700, 0.02),
             'convertair': False, 'modpoly': True, 'polyorder': 0} for s in range(len(ORDERS))]


def test_fitpayne_setup_with_lsf_vectors():
    """fixed Inst_R_<s> vectors leave the free parameters and the prior transform; a mix of vectors and scalars is a
    ValueError before any emulator is loaded"""
    from thepayne_b200.fitting.fitstar import FitPayne
    from thepayne_b200.fitting.multispec import MultiSpecLikelihood
    pri = {'Vrot': {'fixed': 3.0}, 'Inst_R_0': {'fixed': _order_lsf(0)[1]}, 'Inst_R_1': {'fixed': _order_lsf(1)[1]}}
    f = FitPayne()
    ind = f._setup(inputdict={'spec': _setup_specs(), 'specANNpath': None, 'priordict': pri}, verbose=False)
    f._prepare(ind)
    assert f.priorobj.fitpars_i == LABELS + ['Vrad', 'pc_0_0', 'pc_1_0'] and f.ndim == 7
    assert ind['fitargs']['fixedpars']['Inst_R_1'] is pri['Inst_R_1']['fixed']
    u = np.random.default_rng(0).random((5, 7))
    assert np.all(np.isfinite(f.priorobj.priortrans_batch(u)))
    assert np.all(f.priorobj.lnprior_batch(f.priorobj.priortrans_batch(u)) == 0.0)
    for inst1 in (32000.0, None):
        pri2 = dict(pri, Inst_R_1={'fixed': inst1}) if inst1 else {k: v for k, v in pri.items() if k != 'Inst_R_1'}
        ind = FitPayne()._setup(inputdict={'spec': _setup_specs(), 'specANNpath': None, 'priordict': pri2},
                                verbose=False)
        with pytest.raises(ValueError, match=r'spectra \[0\] have an LSF vector .* spectra \[1\] do not'):
            MultiSpecLikelihood(ind['fitargs'], ind['fitpars'], ind['runbools'])


@gpu
def test_multispec_likelihood_with_lsf_vectors():
    """lnlike_batch = -0.5 (sum of the single-spectrum chi2), each from a likelihood with that spectrum's LSF vector"""
    from thepayne_b200.fitting.fitstar import FitPayne
    from thepayne_b200.fitting.likelihood import likelihood
    from thepayne_b200.fitting.multispec import MultiSpecLikelihood
    spec = _emulator(12)
    specs = _two_orders(spec)
    lsfs = [_order_lsf(s)[1] for s in range(len(ORDERS))]
    pri = {'Vrot': {'fixed': 3.0}, 'Inst_R_0': {'fixed': lsfs[0]}, 'Inst_R_1': {'fixed': lsfs[1]}}
    ind = FitPayne()._setup(inputdict={'spec': specs, 'specANNpath': spec, 'priordict': pri}, verbose=False)
    L = MultiSpecLikelihood(ind['fitargs'], ind['fitpars'], ind['runbools'])
    assert L.fitpars_i == LABELS + ['Vrad', 'pc_0_0', 'pc_1_0'] and L.engine.query('lsf') == 1
    rng = np.random.default_rng(3)
    th = np.array([[TRUTH[p] for p in L.fitpars_i]] * 6)
    th[:, 0] += rng.uniform(-200, 200, 6)
    th[:, 4] += rng.uniform(-3, 3, 6)
    th[:, 5:] += rng.uniform(-0.05, 0.05, (6, 2))
    got = L.lnlike_batch(th)
    assert L.lnlikefn(list(th[2])) == got[2]
    c2 = []
    for s, sp in enumerate(specs):
        fa = {'obs_wave_fit': sp['obs_wave'], 'obs_flux_fit': sp['obs_flux'], 'obs_eflux_fit': sp['obs_eflux'],
              'specANNpath': spec, 'NNtype': 'LinNet', 'fixedpars': {'Vrot': 3.0, 'Inst_R': lsfs[s]}}
        names = LABELS + ['Vrad', 'Vrot', 'Inst_R', 'pc_0']
        one = likelihood(fa, [names, {n: n not in ('Vrot', 'Inst_R') for n in names}], [True, False, True, False, False],
                         verbose=False)
        cols = [L.fitpars_i.index(p) for p in LABELS + ['Vrad', 'pc_%d_0' % s]]
        c2.append(-2.0 * one.lnlike_batch(np.ascontiguousarray(th[:, cols])))
    assert np.all(np.isfinite(got))
    assert np.array_equal(got, -0.5 * (c2[0] + c2[1]))


@gpu
def test_fitpayne_two_orders_with_lsf_vectors(tmp_path):
    from thepayne_b200.fitting.fitstar import FitPayne
    spec = _emulator(12)
    pri = {'Teff': {'pv_uniform': [5400.0, 6100.0]}, 'log(g)': {'pv_uniform': [4.0, 4.8]},
           '[Fe/H]': {'pv_uniform': [-0.1, 0.1]}, '[a/Fe]': {'pv_uniform': [-0.1, 0.1]},
           'Vrad': {'pv_uniform': [-3.0, 3.0]}, 'Vrot': {'fixed': 3.0},
           'Inst_R_0': {'fixed': _order_lsf(0)[1]}, 'Inst_R_1': {'fixed': _order_lsf(1)[1]}}
    out = str(tmp_path / 'two_orders_lsf.dat')
    FitPayne().run(inputdict={'spec': _two_orders(spec), 'specANNpath': spec, 'NNtype': 'LinNet', 'priordict': pri,
                              'output': out, 'sampler': {'samplertype': 'Static', 'samplemethod': 'rwalk',
                                                         'npoints': 40, 'walks': 10, 'delta_logz_final': 0.5,
                                                         'seed': 5, 'maxiter': 6000}}, verbose=False)
    head = open(out).readline().split()
    assert head[1:9] == LABELS + ['Vrad', 'pc_0_0', 'pc_1_0', 'Vrot']
    assert not any(h.startswith('Inst_R') for h in head)
    d = np.loadtxt(out, skiprows=1)
    lw = d[:, head.index('log(wt)')] - d[:, head.index('log(z)')][-1]
    w = np.exp(lw - lw.max())
    w /= w.sum()
    for p in LABELS[:3] + ['Vrad', 'pc_0_0', 'pc_1_0']:
        x = d[:, head.index(p)]
        mean = np.sum(w * x)
        sd = np.sqrt(np.sum(w * (x - mean) ** 2))
        assert abs(mean - TRUTH[p]) <= 4.0 * sd + 1e-9 * abs(TRUTH[p]), (p, mean, sd, TRUTH[p])
