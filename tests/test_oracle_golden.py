"""CPU: pin the oracle (oracle/payne_oracle.py) against fixtures minted by the UNMODIFIED
reference (oracle/make_golden.py).  Same libraries on both sides, so agreement is to
round-off: 1e-9 relative on flux, 1e-9 relative on lnL."""
import numpy as np
import pytest

from conftest import load_case
from oracle import goldens, payne_oracle as O


@pytest.fixture(autouse=True, scope='module')
def _minting_threads():
    """The fixtures were minted with torch on 8 CPU threads of an AVX-512 host, and MKL's fp32 sgemm sums in an order
    that follows the thread count: pinned to 8, the oracle's emulator reproduces them bit for bit on AVX-512 hosts of
    any core count (16 threads differ by up to 1.5e-8 relative in flux, beyond the 1e-9 checked here)."""
    import torch
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize('name', list(goldens.CASES))
def test_oracle_matches_reference(name):
    cfg, g = load_case(name)
    L = O.OracleLikelihood(cfg)
    th = g['theta']
    n = min(len(th), 12 if name.startswith('c') else len(th))
    lnl = np.array([L.lnlikefn(t) for t in th[:n]])
    ref = g['lnl'][:n]
    assert np.array_equal(np.isnan(lnl), np.isnan(ref))
    ok = ~np.isnan(ref)
    np.testing.assert_allclose(lnl[ok], ref[ok], rtol=1e-9, atol=1e-9)
    nf = min(n, g['flux'].shape[0])
    _, fl, mg = L.lnlike_batch(th[:nf], return_model=True)
    np.testing.assert_allclose(fl, g['flux'][:nf], rtol=1e-9, atol=1e-12, equal_nan=True)
    if 'mags' in g:
        np.testing.assert_allclose(mg, g['mags'][:nf], rtol=1e-12, atol=1e-12)


def test_edge_rows_take_the_reference_branches():
    cfg, g = load_case('mini_spec')
    ix = {p: i for i, p in enumerate(cfg.fitpars_i)}
    th = g['theta']
    assert th[1, ix['Vrot']] == 0 and th[2, ix['Vrad']] == 0
    assert np.isnan(g['lnl'][4]) and np.isfinite(g['lnl'][[0, 1, 2, 3, 6, 7, 8, 9, 10, 11]]).all()
    cfg2, g2 = load_case('mini_edge')
    assert np.isnan(g2['lnl']).all()


def test_batched_mlp_noise_floor():
    """The reference's own fp32 emulator is only reproducible to ~1e-7 per pixel: running
    the same torch Linear stack at batch 1 (what the reference does) or batched changes
    the summation order.  This is the floor any re-implementation is measured against."""
    cfg, g = load_case('mini_spec')
    L = O.OracleLikelihood(cfg)
    th = g['theta'][:8]
    a, fa, _ = L.lnlike_batch(th, return_model=True)
    b, fb, _ = L.lnlike_batch(th, return_model=True, batched_mlp=True)
    ok = np.isfinite(a)
    rel = np.nanmax(np.abs(fa - fb) / np.abs(fa))
    assert rel < 1e-6
    assert np.max(np.abs(a[ok] - b[ok])) < 5e-3


def test_oracle_getspec_continuum_and_lsf_match_reference():
    """SURVEY §8 f3: the continuum-emulator multiply (predictspec.py:208-226) and the LSF-vector
    broadening (predictspec.py:265-286 -> smoothing.py:482-586) against the unmodified reference's getspec."""
    import os
    from conftest import GOLDEN
    g = np.load(os.path.join(GOLDEN, 'f3_getspec.npz'))
    spec, cont, calls = goldens.getspec_case()
    assert spec.digest() == str(g['digest']) and cont.digest() == str(g['cdigest'])
    net, cnet = O.make_net(spec), O.make_net(cont)
    for i, kw in enumerate(calls):
        w, f = O.getspec(net, spec, kw['Teff'], kw['log(g)'], kw['[Fe/H]'], kw['[a/Fe]'], np.nan, kw['rot_vel'],
                         kw['rad_vel'], kw.get('inst_R', np.nan), kw['outwave'],
                         cont=(cnet, cont) if kw['use_cont'] else None)
        np.testing.assert_array_equal(w, g['wave_%d' % i])
        np.testing.assert_allclose(f, g['flux_%d' % i], rtol=1e-9, atol=1e-12, equal_nan=True)
    assert np.isnan(g['flux_1']).sum() > 50          # plain-interp call: pixels beyond the continuum grid are NaN
