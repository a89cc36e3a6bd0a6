"""FitPayne's input dictionary with ``spec['modpoly_marginal']``: the continuum coefficients leave the sampled parameters,
their boxes follow the rule of a sampled ``pc_k`` (``prior.pc_box``), the output file keeps their columns, and the
errors for mixed lists of spectra and for ``modpoly_marginal`` without ``modpoly``.  No GPU needed."""
import numpy as np
import pytest

from thepayne_b200.fitting.fitstar import FitPayne
from thepayne_b200.fitting.prior import prior


def _spec(n=50, **kw):
    w = np.linspace(5150.0, 5180.0, n)
    d = {'obs_wave': w, 'obs_flux': np.ones(n), 'obs_eflux': np.full(n, 0.01), 'convertair': False}
    d.update(kw)
    return d


def _setup(inputdict):
    f = FitPayne()
    ind = f._setup(inputdict=inputdict, verbose=False)
    f._prepare(ind)
    return f, ind


def test_single_spectrum_parameters_and_boxes():
    blaze = [[1.0, 0.1], [0.02, 0.01], [-0.01, 0.004]]
    fs, ind_s = _setup({'spec': _spec(modpoly=True), 'priordict': {'blaze_coeff': blaze}})
    fm, ind_m = _setup({'spec': _spec(modpoly=True, modpoly_marginal=True), 'priordict': {'blaze_coeff': blaze}})
    sampled = [p for p in ind_s['fitpars'][0] if ind_s['fitpars'][1][p]]
    marginal = [p for p in ind_m['fitpars'][0] if ind_m['fitpars'][1][p]]
    assert sampled == marginal + ['pc_0', 'pc_1', 'pc_2']
    assert fm.ndim == fs.ndim - 3
    fa = ind_m['fitargs']
    assert fa['cont_names'] == ['pc_0', 'pc_1', 'pc_2']
    assert fa['cont_box'] == [prior.pc_box(k, blaze) for k in range(3)]
    assert np.allclose(fa['cont_box'], [(0.75, 1.25), (-0.03, 0.07), (-0.03, 0.01)], rtol=0, atol=1e-15)
    # the box is the range the sampled prior transform spans
    U = np.array([[0.0] * fs.ndim, [1.0] * fs.ndim])
    V = fs.priorobj.priortrans_batch(U)
    for k in range(3):
        i = fs.priorobj.fitpars_i.index('pc_%d' % k)
        assert np.allclose((V[0, i], V[1, i]), fa['cont_box'][k], rtol=0, atol=1e-15)
    assert prior.pc_box(0, blaze) == (0.75, 1.25)


def test_polyorder_default_boxes():
    _, ind = _setup({'spec': _spec(modpoly=True, modpoly_marginal=True, polyorder=2, polysigma=0.5)})
    assert ind['fitargs']['cont_box'] == [(0.75, 1.25), (-2.5, 2.5), (-2.5, 2.5)]


def test_output_columns(tmp_path):
    f, ind = _setup({'spec': _spec(modpoly=True, modpoly_marginal=True, polyorder=1),
                     'output': str(tmp_path / 'out.dat')})

    class Like:                                  # the columns come from the likelihood's parameters and fixedpars
        fitpars_i = [p for p in ind['fitpars'][0] if ind['fitpars'][1][p]]
        fixedpars = {}
    f.likeobj = Like()
    parnames = list(Like.fitpars_i) + list(ind['fitargs']['cont_names'])
    f._initoutput(parnames)
    f._writerow(0, [1.0] * len(Like.fitpars_i), parnames, (0, 0, 0, 0, 0, 0, 0), cont=[1.01, -0.02])
    f.outff.close()
    head, row = open(tmp_path / 'out.dat').read().splitlines()
    assert head.split()[-9:-7] == ['pc_0', 'pc_1']
    assert row.split()[len(Like.fitpars_i) + 1:len(Like.fitpars_i) + 3] == ['1.01', '-0.02']


def test_spectrum_list():
    specs = [_spec(modpoly=True, modpoly_marginal=True, polyorder=1), _spec(modpoly=True, modpoly_marginal=True)]
    f, ind = _setup({'spec': specs, 'priordict': {'blaze_coeff_1': [[1.0, 0.1], [0.0, 0.02], [0.0, 0.01], [0.0, 0.01]]}})
    free = [p for p in ind['fitpars'][0] if ind['fitpars'][1][p]]
    assert not any(p.startswith('pc_') for p in free)
    fa = ind['fitargs']
    assert fa['cont_names'] == ['pc_0_0', 'pc_0_1', 'pc_1_0', 'pc_1_1', 'pc_1_2', 'pc_1_3']
    assert fa['spectra'][0]['cont_box'] == [(0.75, 1.25), (-5.0, 5.0)]
    assert fa['spectra'][1]['cont_box'] == [(0.75, 1.25), (-0.1, 0.1), (-0.05, 0.05), (-0.05, 0.05)]


def test_errors():
    with pytest.raises(ValueError, match='modpoly_marginal or none'):
        _setup({'spec': [_spec(modpoly=True, modpoly_marginal=True), _spec(modpoly=True)]})
    with pytest.raises(ValueError, match='needs'):
        _setup({'spec': _spec(modpoly_marginal=True)})
    with pytest.raises(ValueError, match='needs'):
        _setup({'spec': [_spec(modpoly_marginal=True), _spec(modpoly_marginal=True)]})
