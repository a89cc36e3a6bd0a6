"""FitPayne with a list-valued ``spec`` (several spectra of one star): parameter names, fixed values, priors and the
refusals, without a GPU."""
import numpy as np
import pytest

from thepayne_b200.fitting.fitstar import FitPayne
from thepayne_b200.fitting.multispec import spectrum_name
from thepayne_b200.fitting.multistar import FitPayneMany


def _spec(lo, hi, n=50, **kw):
    w = np.linspace(lo, hi, n)
    return dict({'obs_wave': w, 'obs_flux': np.ones(n), 'obs_eflux': np.full(n, 0.01), 'convertair': False}, **kw)


def _setup(inputdict):
    f = FitPayne()
    ind = f._setup(inputdict=inputdict, verbose=False)
    f._prepare(ind)
    return f, ind


def test_list_spec_names_and_fixed_values():
    pri = {'Inst_R_1': {'fixed': 30000.0}, 'Inst_R_0': {'pv_uniform': [20000.0, 40000.0]},
           'blaze_coeff_1': [[0.0, 1.0], [0.1, 0.02]], 'Vrot': {'fixed': 2.0}}
    f, ind = _setup({'spec': [_spec(5150.0, 5160.0, modpoly=True, polyorder=2),
                              _spec(5170.0, 5180.0, modpoly=True, wave_minmax=[5171.0, 5179.0])],
                     'specANNpath': None, 'priordict': pri})
    fa = ind['fitargs']
    free = [p for p in ind['fitpars'][0] if ind['fitpars'][1][p]]
    assert free == ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Inst_R_0', 'pc_0_0', 'pc_0_1', 'pc_0_2',
                    'pc_1_0', 'pc_1_1']
    assert 'Inst_R' not in ind['fitpars'][0]
    assert fa['fixedpars'] == {'Inst_R_1': 30000.0, 'Vrot': 2.0}
    assert ind['runbools'][:3] == [True, False, True]
    assert len(fa['spectra']) == 2 and len(fa['spectra'][0]['obs_wave_fit']) == 50
    w1 = fa['spectra'][1]['obs_wave_fit']
    assert w1.min() >= 5171.0 and w1.max() <= 5179.0
    assert ind['priordict']['blaze_coeff_0'] == [[0.0, 1.0]] * 3
    # prior transforms: Inst_R_0 its own uniform prior, pc_<s>_0 in [0.75, 1.25], pc_<s>_k from blaze_coeff_<s>
    u = np.full((1, len(free)), 0.5)
    u[0, free.index('Inst_R_0')] = 0.25
    x = dict(zip(free, f.priorobj.priortrans_batch(u)[0]))
    assert x['Inst_R_0'] == 25000.0 and x['pc_0_0'] == 1.0 and x['pc_1_0'] == 1.0
    assert x['pc_0_1'] == 0.0 and np.isclose(x['pc_1_1'], 0.1)
    assert f.priorobj.priortrans([0.5] * len(free)) == list(f.priorobj.priortrans_batch(np.full((1, len(free)), 0.5))[0])


def test_list_spec_default_inst_r_range_and_additive_prior():
    pri = {'Inst_R_0': {'gaussian': [30000.0, 1000.0]}}
    f, ind = _setup({'spec': [_spec(5150.0, 5160.0), _spec(5170.0, 5180.0)], 'specANNpath': None, 'priordict': pri})
    free = f.priorobj.fitpars_i
    assert free == ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Inst_R_0', 'Inst_R_1']
    x = f.priorobj.priortrans([0.5] * len(free))
    assert x[free.index('Inst_R_1')] == 35000.0                   # the default range of Inst_R
    th = np.array([x, x])
    th[1, free.index('Inst_R_0')] = 31000.0
    assert np.allclose(f.priorobj.lnprior_batch(th), [-0.5 * 25.0, -0.5 * 1.0])


def test_spectrum_names():
    assert spectrum_name('Inst_R_1', 1) == 'Inst_R' and spectrum_name('Inst_R_1', 0) is None
    assert spectrum_name('pc_2_3', 2) == 'pc_3' and spectrum_name('pc_2_3', 1) is None
    assert spectrum_name('Vrad', 5) == 'Vrad'


def test_dict_spec_unchanged():
    _, ind = _setup({'spec': _spec(5150.0, 5160.0, modpoly=True), 'specANNpath': None})
    free = [p for p in ind['fitpars'][0] if ind['fitpars'][1][p]]
    assert free == ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Inst_R', 'pc_0', 'pc_1', 'pc_2']
    assert 'spectra' not in ind['fitargs']


def test_refusals():
    two = [_spec(5150.0, 5160.0), _spec(5170.0, 5180.0)]
    with pytest.raises(NotImplementedError):
        _setup({'spec': two, 'specANNpath': None, 'priordict': {'Vrad_1': {'pv_uniform': [-5.0, 5.0]}}})
    with pytest.raises(NotImplementedError):
        _setup({'spec': [_spec(5150.0, 5160.0, Vrad=1.0), two[1]], 'specANNpath': None})
    with pytest.raises(ValueError):
        _setup({'spec': [_spec(5150.0, 5160.0, modpoly=True), two[1]], 'specANNpath': None})
    with pytest.raises(NotImplementedError):
        FitPayneMany().run(inputdicts=[{'spec': two, 'specANNpath': None}], verbose=False)
