"""Double-lined binaries without a GPU: FitPayne's parameter names, order, defaults and priors with ``'binary': True``,
the refusals, the reference evaluation at Rratio = 0, and the PayneBinary ctypes mirror against the C header."""
import ctypes
import os
import subprocess
import types

import numpy as np
import pytest

from thepayne_b200 import _lib, synth
from thepayne_b200.fitting.fitstar import FitPayne
from thepayne_b200.fitting.multistar import FitPayneMany

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Inst_R']


def _spec(n=50, **kw):
    w = np.linspace(5150.0, 5160.0, n)
    return dict({'obs_wave': w, 'obs_flux': np.ones(n), 'obs_eflux': np.full(n, 0.01), 'convertair': False}, **kw)


def _setup(inputdict):
    f = FitPayne()
    ind = f._setup(inputdict=inputdict, verbose=False)
    f._prepare(ind)
    return f, ind


def _free(ind):
    return [p for p in ind['fitpars'][0] if ind['fitpars'][1][p]]


def test_binary_names_order_and_default_priors():
    f, ind = _setup({'spec': _spec(modpoly=True, polyorder=1), 'specANNpath': None, 'binary': True, 'priordict': {}})
    assert _free(ind) == REF + ['Teff_sec', 'log(g)_sec', 'Vrad_sec', 'Vrot_sec', 'Rratio', 'pc_0', 'pc_1']
    assert ind['fitargs']['binary'] is True and ind['fitargs']['fixedpars'] == {}
    pr = f.priorobj
    u = np.array([[0.0] * f.ndim, [1.0] * f.ndim])
    x = pr.priortrans_batch(u)
    lohi = {p: (x[0, i], x[1, i]) for i, p in enumerate(pr.fitpars_i)}
    # the _sec names take the primary's default ranges, Rratio uniform [0, 1]
    for p in ['Teff', 'log(g)', 'Vrad', 'Vrot']:
        assert lohi[p + '_sec'] == lohi[p] == tuple(pr.defaultpars[p])
    assert lohi['Rratio'] == (0.0, 1.0)


def test_binary_optional_parameters_fixed_values_and_priors():
    pri = {'[Fe/H]_sec': {'pv_uniform': [-0.5, 0.0]}, 'Vmic_sec': {'fixed': 1.2}, 'Vrot_sec': {'fixed': 4.0},
           'Rratio': {'pv_uniform': [0.2, 0.8]}, 'Teff_sec': {'pv_gaussian': [4500.0, 100.0]}}
    f, ind = _setup({'spec': _spec(), 'specANNpath': None, 'binary': True, 'priordict': pri})
    # [Fe/H]_sec gets a column because the prior names it; [a/Fe]_sec does not; Vmic_sec and Vrot_sec are fixed
    assert _free(ind) == REF + ['Teff_sec', 'log(g)_sec', '[Fe/H]_sec', 'Vrad_sec', 'Rratio']
    assert ind['fitargs']['fixedpars'] == {'Vmic_sec': 1.2, 'Vrot_sec': 4.0}
    x = f.priorobj.priortrans([0.5] * f.ndim)
    got = dict(zip(f.priorobj.fitpars_i, x))
    assert got['[Fe/H]_sec'] == -0.25 and got['Rratio'] == 0.5 and got['Teff_sec'] == 4500.0


def test_without_binary_nothing_changes():
    f, ind = _setup({'spec': _spec(), 'specANNpath': None, 'priordict': {}})
    assert _free(ind) == REF and 'binary' not in ind['fitargs']


def test_binary_refusals():
    with pytest.raises(NotImplementedError, match='list-valued'):
        FitPayne()._setup(inputdict={'spec': [_spec(), _spec()], 'binary': True}, verbose=False)
    with pytest.raises(NotImplementedError, match='photometry'):
        FitPayne()._setup(inputdict={'spec': _spec(), 'phot': {'GaiaEDR3_G': [10.0, 0.01]}, 'binary': True},
                          verbose=False)
    with pytest.raises(NotImplementedError, match='binaries'):
        FitPayneMany().run(inputdicts=[{'spec': _spec(), 'binary': True}], verbose=False)


def test_reference_at_rratio_zero_is_the_single_star_reference():
    from oracle import payne_oracle as O
    from binary_oracle import binary_lnlike_batch
    wave, rsig = synth.ann_wavegrid(5140.0, 5152.0, 50000.0)
    spec = synth.make_specnet(4, 16, wave, rsig, seed=0)
    w = np.linspace(wave[40], wave[-40], 300)
    rng = np.random.default_rng(2)
    fit = REF + ['Teff_sec', 'log(g)_sec', 'Vrad_sec', 'Vrot_sec', 'Rratio', 'pc_0', 'pc_1']
    cfg = types.SimpleNamespace(spec=spec, phot=None, runbools=[True, False, True, False, False], fitpars_i=fit,
                                fixedpars={}, obs_wave=w, obs_flux=1.0 + 0.02 * rng.standard_normal(len(w)),
                                obs_eflux=np.full(len(w), 0.02))
    th = np.array([[5800.0, 4.4, 0.0, 0.1, 3.0, 5.0, 30000.0, 4500.0, 4.7, -20.0, 2.0, 0.0, 1.01, 0.02],
                   [6200.0, 4.0, -0.3, 0.2, -8.0, 0.0, 36000.0, 5000.0, 4.5, 25.0, 0.0, 0.0, 0.98, -0.01]])
    lb, mb, cb = binary_lnlike_batch(cfg, th, return_model=True)
    ls, fs, _ = O.OracleLikelihood(cfg).lnlike_batch(th, return_model=True)
    assert np.array_equal(lb, ls) and np.array_equal(mb, fs)
    # and with a positive Rratio the secondary enters
    th[:, fit.index('Rratio')] = 0.6
    assert np.all(np.abs(binary_lnlike_batch(cfg, th) - ls) > 0)


def test_binary_struct_matches_header(tmp_path):
    src = tmp_path / 'b.c'
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "payne_b200.h"\n'
                   'int main(){printf("%zu %zu %zu %zu\\n", sizeof(PayneBinary), offsetof(PayneBinary, fixed),'
                   'offsetof(PayneBinary, rratio_col), offsetof(PayneBinary, rratio_fixed)); return 0;}\n')
    exe = tmp_path / 'b'
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    B = _lib.PayneBinary
    assert got == [ctypes.sizeof(B), B.fixed.offset, B.rratio_col.offset, B.rratio_fixed.offset]
