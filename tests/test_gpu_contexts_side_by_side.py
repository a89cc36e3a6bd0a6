"""Contexts of different sizes in one process.

The dynamic shared-memory opt-in (cudaFuncAttributeMaxDynamicSharedMemorySize) belongs to a kernel function on the
device, not to a context, and a launch that asks for more than it fails.  The LSF tail (both forms), the photometry
kernel (with and without band lists) and the general tail for grids of <= 1024 pixels share one instantiation between
contexts whose dynamic shared memory differs, so a context built later must not lower what an earlier one launches
with (raise_max_dyn_smem, launchers.h).

For each pair: build A and evaluate it (its reference); build B and evaluate it; A again must give the same bits with
status 0; destroy B, A again; then the same in the reverse creation order.  What the contexts report of their launch
grids must not depend on the order either.
"""
import numpy as np
import pytest

from thepayne_b200 import synth

pytestmark = pytest.mark.gpu
LABELS = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot']


def _log_grid(n):
    rsig = 50000.0 * synth.SIGMA_TO_FWHM_TRAIN
    w, _ = synth.ann_wavegrid(5000.0, 5000.0 * (1.0 + 1.0 / (3.0 * rsig)) ** (n - 1.0), 50000.0)
    return w, rsig


def _obs(w, n=300, seed=0):
    a, b = w[0], w[-1]
    ow = np.linspace(a + 0.3 * (b - a), a + 0.7 * (b - a), n)
    rng = np.random.default_rng(seed)
    return dict(wave=ow, flux=1.0 + 0.02 * rng.standard_normal(n), eflux=np.full(n, 0.02))


def _theta(fit, B, seed):
    rng = np.random.default_rng(seed)
    box = dict(synth._BOX)
    lo, hi = np.array([box[p][0] for p in fit]), np.array([box[p][1] for p in fit])
    return np.ascontiguousarray(lo + (hi - lo) * rng.random((B, len(fit))))


def _lsf_engine(n, targets):
    from thepayne_b200.engine import Engine
    w, rsig = _log_grid(n)
    spec = synth.make_specnet(4, 16, w, rsig, seed=n % 13)
    st = _obs(w)
    st['fixedpars'] = {'Inst_R': np.full(len(st['wave']), 0.1)}
    st['fitpars_i'] = LABELS
    eng = Engine(spec=spec, stars=[st], targets=[1] if targets else None)
    assert eng.query('lsf') == 1
    return eng, _theta(LABELS, 40, n)


def _phot_engine(H, nb, band_lists):
    from thepayne_b200.engine import Engine
    net = synth.make_photnet(synth.C1_BANDS[:nb], H=H, seed=H)
    fit = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'log(A)', 'Av']
    rb = [False, True, False, True, False]
    phot = {b: (5.0 + 0.1 * i, 0.05) for i, b in enumerate(net.bands)}
    if band_lists:                              # a subset in another order: the band-slot kernel
        bands = net.bands[::-2]
        eng = Engine(phot=net, stars=[{'phot': {b: phot[b] for b in bands}, 'bands': bands}], fitpars_i=fit, runbools=rb)
    else:
        eng = Engine(phot=net, obs_phot=phot, fitpars_i=fit, runbools=rb)
    return eng, _theta(fit, 40, H + nb)


def _general_engine(n):
    from thepayne_b200.engine import Engine
    _, rsig = _log_grid(16)
    w = np.linspace(5000.0, 5000.0 + 0.02 * n, n)
    spec = synth.make_specnet(4, 16, w, rsig, seed=n % 11)
    st = _obs(w, seed=n)
    fit = LABELS + ['Inst_R']
    eng = Engine(spec=spec, obs_wave=st['wave'], obs_flux=st['flux'], obs_eflux=st['eflux'], fitpars_i=fit)
    assert eng.query('fast_tail') == 0
    return eng, _theta(fit, 40, n)


def _eval(eng, th):
    import torch
    star = torch.zeros(len(th), dtype=torch.int32, device='cuda')
    thd = torch.from_numpy(th).cuda()
    if eng.n_targets:
        f, _, m, l = eng.model_batch_targets(thd, star)
        out = [l, eng.lnlike_batch_targets(thd, star)] + [x for x in (f, m) if x is not None]
    else:
        f, m, l = eng.model_batch(thd)
        out = [l, eng.lnlike_batch(thd)] + [x for x in (f, m) if x is not None]
    torch.cuda.synchronize()
    out = [x.cpu().numpy() for x in out]
    assert eng.query('status') == 0
    return out


def _same(a, b):
    return len(a) == len(b) and all(np.array_equal(x, y, equal_nan=True) for x, y in zip(a, b))


def _grids(eng):
    return {k: eng.query(k) for k in ('tail_grid', 'max_batch', 'lsf', 'fast_tail')}


PAIRS = {
    'lsf_star': (lambda: _lsf_engine(1 << 15, False), lambda: _lsf_engine(1 << 10, False)),
    'lsf_target': (lambda: _lsf_engine(1 << 15, True), lambda: _lsf_engine(1 << 10, True)),
    'phot': (lambda: _phot_engine(512, 7, False), lambda: _phot_engine(16, 7, False)),
    'phot_band_lists': (lambda: _phot_engine(64, 27, True), lambda: _phot_engine(64, 7, True)),
    'general_tail': (lambda: _general_engine(1024), lambda: _general_engine(300)),
}


@pytest.mark.parametrize('name', list(PAIRS))
def test_context_built_later_leaves_the_earlier_one_alone(name):
    mk_a, mk_b = PAIRS[name]
    a, th_a = mk_a()
    ref = _eval(a, th_a)
    assert np.isfinite(ref[0]).sum() > len(th_a) // 2
    grids_a = _grids(a)
    b, th_b = mk_b()
    ref_b = _eval(b, th_b)
    grids_b = _grids(b)
    assert _same(_eval(a, th_a), ref), name
    b.close()
    assert _same(_eval(a, th_a), ref), name
    a.close()
    # the reverse creation order
    b, _ = mk_b()
    assert _same(_eval(b, th_b), ref_b) and _grids(b) == grids_b, name
    a, _ = mk_a()
    assert _grids(a) == grids_a, name
    assert _same(_eval(a, th_a), ref), name
    b.close()
    assert _same(_eval(a, th_a), ref), name
    a.close()
