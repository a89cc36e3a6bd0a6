"""Per-star parameter layouts in an observation set (PayneStarOpts.layout, Engine(stars=[{'fitpars_i', 'runbools'}])):
each star's own free parameters and their order, continuum order, photometry and photscale in one batch.

The core check is bit-identity: every star's rows of an interleaved batch (with a run of one star's rows across a
slab boundary) give exactly (np.array_equal, NaN patterns included) what a single-star engine built from that star's
own layout gives when fed that star's own columns.  Then padding columns, layouts equal to the context's, the
refusals, the ABI struct against its ctypes mirror (no GPU), and FitPayneMany on heterogeneous input dictionaries.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from thepayne_b200 import _lib, synth
from thepayne_b200.engine import Engine, _layout, _specnet_struct
from test_gpu_star_opts import BANDS, FIXED, _apply, _lsf, _sampler, _spec, _stars, _subnet

gpu = pytest.mark.gpu
_INVALID, _UNSUPPORTED = -1, -4
LABELS = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]']

# name: (emulator, D_in, precision, settings, lsf, per-star (free spectral parameters, n_poly, photometry mode, permute))
A3 = ['Vrad', 'Vrot', 'Inst_R']
SETUPS = {
    'fast_poly_orders': ('mini', 4, 'parity', {'max_batch': 200}, False,
                         [(A3, 1, None, 0), (['Vrad', 'Inst_R'], 3, None, 0), (['Vrot'], 6, None, 0),
                          (A3, 16, None, 0), ([], 3, None, 0), (['Inst_R'], 1, None, 0)]),
    'fast_free_or_fixed': ('mini', 4, 'parity', {'max_batch': 200}, False,
                           [(A3, 0, None, 0), (['Vrad'], 0, None, 0), (['Vrot'], 0, None, 0), (['Inst_R'], 0, None, 0),
                            ([], 0, None, 0), (['Vrot', 'Inst_R'], 0, None, 0)]),
    'permuted_columns': ('mini', 4, 'parity', {'max_batch': 200}, False,
                         [(A3, 2, None, 1), (A3, 2, None, 2), (['Vrad'], 3, None, 3), (A3, 4, None, 4),
                          (['Vrot', 'Inst_R'], 2, None, 5), (A3, 5, None, 6)]),
    'cluster': ('mid', 4, 'parity', {'tail_cluster': 1, 'max_batch': 200}, False,
                [(A3, 1, None, 0), (['Vrad'], 3, None, 0), (['Inst_R'], 6, None, 3), (A3, 2, None, 0),
                 (['Vrot', 'Inst_R'], 1, None, 0), ([], 3, None, 0)]),
    'cluster_plain': ('mid', 4, 'parity', {'tail_cluster': 1, 'max_batch': 200}, False,
                      [(A3, 0, None, 0), (['Vrad'], 0, None, 0), (['Inst_R'], 0, None, 3), (A3, 0, None, 0),
                       (['Vrot', 'Inst_R'], 0, None, 0), ([], 0, None, 0)]),
    'multi_chunk': ('multi', 4, 'parity', {'max_batch': 200}, False,
                    [(A3, 2, None, 0), (['Vrad'], 1, None, 2), (['Vrot', 'Inst_R'], 4, None, 0), (A3, 3, None, 1),
                     ([], 2, None, 0), (['Inst_R'], 6, None, 0)]),
    'general': ('mini', 4, 'parity', {'fast_tail': 0, 'max_batch': 200}, False,
                [(A3, 2, None, 0), (['Vrad'], 4, None, 0), (['Inst_R'], 1, None, 1), (A3, 3, None, 0),
                 (['Vrot'], 2, None, 0), ([], 5, None, 0)]),
    'lsf': ('mini', 4, 'parity', {'max_batch': 200}, True,
            [(['Vrad', 'Vrot'], 2, None, 0), (['Vrad'], 3, None, 0), (['Vrot'], 2, None, 1), ([], 4, None, 0),
             (['Vrad', 'Vrot'], 1, None, 0), (['Vrot'], 2, None, 0)]),
    'continuum': ('mini', 4, 'parity', {'max_batch': 200, 'continuum': 1}, False,
                  [(A3, 1, None, 0), (['Vrad'], 2, None, 0), (['Inst_R'], 3, None, 1), (A3, 2, None, 0),
                   ([], 1, None, 0), (['Vrot', 'Inst_R'], 4, None, 0)]),
    'joint_mixed_phot': ('mini', 4, 'parity', {'max_batch': 200}, False,
                         [(A3, 2, None, 0), (A3, 3, 'scaled', 0), (['Vrad', 'Inst_R'], 2, 'dist', 1),
                          (['Inst_R'], 4, None, 0), (A3, 2, 'dist', 0), (['Vrot'], 3, 'scaled', 0)]),
    'phot_only_mixed': (None, 4, 'parity', {'max_batch': 200}, False,
                        [([], 0, 'scaled', 0), ([], 0, 'dist', 0), ([], 0, 'scaled', 1), ([], 0, 'dist', 2),
                         ([], 0, 'dist', 0), ([], 0, 'scaled', 0)]),
    'vmic': ('mini', 5, 'parity', {'max_batch': 200}, False,
             [(A3 + ['Vmic'], 2, None, 0), (A3, 2, None, 0), (['Vmic', 'Inst_R'], 3, None, 1), (['Inst_R'], 2, None, 0),
              (['Vmic'], 2, None, 0), (['Vrad', 'Vmic'], 4, None, 0)]),
    'simt': ('mini', 4, 'simt', {'max_batch': 200}, False,
             [(A3, 2, None, 0), (['Vrad'], 3, None, 0), (['Inst_R'], 2, None, 1), (A3, 6, None, 0),
              (['Vrot'], 2, None, 0), ([], 1, None, 0)]),
}


_MULTI = {}


def _emulator(emu, d_in):
    """'multi': a multi-chunk emulator on the 'mini' grid (chunks of 512 pixels); else test_gpu_star_opts' nets"""
    if emu != 'multi':
        return _spec(emu, d_in)
    if d_in not in _MULTI:
        w = _spec('mini', d_in).wavelength
        _MULTI[d_in] = synth.make_multinet(d_in, 64, w, _spec('mini', d_in).resolution, 512, seed=3)
    return _MULTI[d_in]


def _box(fit):
    box = dict(synth._BOX)
    for p in fit:
        if p.startswith('pc_'):
            box[p] = (0.75, 1.25) if p == 'pc_0' else (-0.1, 0.1)
    return box


def _build(name):
    """(engine keywords, stars with their own 'fitpars_i' / 'runbools' / 'fixedpars', nets)"""
    emu, d_in, prec, settings, lsf, per = SETUPS[name]
    spec = _emulator(emu or 'mini', d_in)
    any_phot = any(pm for _, _, pm, _ in per)
    net = synth.make_photnet(BANDS, H=16) if any_phot else None
    stars = _stars(spec, any_phot)
    for k, (free, npoly, pmode, perm) in enumerate(per):
        st = stars[k]
        fit = list(LABELS) + [p for p in (['Vmic'] if d_in == 5 else []) + A3 if p in free]
        if pmode == 'scaled':
            fit += ['log(A)', 'Av']
        elif pmode == 'dist':
            fit += ['log(R)', 'Av']
        fit += ['pc_%d' % i for i in range(npoly)]
        if perm:
            fit = [fit[i] for i in np.random.default_rng(perm).permutation(len(fit))]
        fx = {}
        if emu:
            for p in ['Vrad', 'Vrot', 'Inst_R'] + (['Vmic'] if d_in == 5 else []):
                if p not in fit:
                    fx[p] = FIXED[p][k]
            if lsf:
                fx['Inst_R'] = _lsf(st['wave'], k)
        if pmode == 'dist':
            fx['Dist'] = FIXED['Dist'][k]
        if pmode is None:
            st.pop('phot', None)
            st.pop('bands', None)
        st.update(fitpars_i=fit, fixedpars=fx, runbools=[emu is not None, pmode is not None, npoly > 0,
                                                           pmode == 'scaled'])
    kw = dict(spec=spec if emu else None, phot=net, precision=prec,
              runbools=[emu is not None, any_phot, per[0][1] > 0, False, False])
    return kw, stars, settings


def _single(kw, st, settings):
    """The single-star engine of star ``st``: its own layout, values, bands' net and LSF."""
    fx = dict(st['fixedpars'])
    lsf = fx.pop('Inst_R') if np.ndim(fx.get('Inst_R', 0.0)) == 1 else None
    obs_phot, phot = None, None
    if st['runbools'][1]:
        bands = st.get('bands') or [b for b in kw['phot'].bands if b in st['phot']]
        phot = _subnet(kw['phot'], bands)
        obs_phot = {b: st['phot'][b] for b in bands}
    spec_on = kw['spec'] is not None
    one = Engine(spec=kw['spec'], phot=phot, obs_wave=st['wave'] if spec_on else None,
                 obs_flux=st['flux'] if spec_on else None, obs_eflux=st['eflux'] if spec_on else None,
                 obs_phot=obs_phot, fitpars_i=st['fitpars_i'], fixedpars=fx, runbools=st['runbools'] + [False],
                 precision=kw['precision'])
    if lsf is not None:
        one.set_lsf(lsf)
    _apply(one, settings)
    return one


def _rows(stars, star, ndim, seed, pad):
    """Row p: star[p]'s parameters drawn from the prior box in its own order, then `pad` up to ndim."""
    rng = np.random.default_rng(seed)
    th = np.full((len(star), ndim), pad)
    for p, k in enumerate(star):
        fit = stars[k]['fitpars_i']
        box = _box(fit)
        lo = np.array([box[q][0] for q in fit])
        hi = np.array([box[q][1] for q in fit])
        th[p, :len(fit)] = lo + (hi - lo) * rng.random(len(fit))
        for q in ('Inst_R', 'Vrot'):
            if q in fit and rng.random() < 0.1:
                th[p, fit.index(q)] = 0.0
    return th


def _star_index(S, B):
    star = np.random.default_rng(17).integers(0, S, B).astype(np.int32)
    star[:250] = 1                      # a run of one star's rows across the 200-point slab boundary
    return star


def _eval(eng, th, star):
    tht = torch.from_numpy(np.ascontiguousarray(th)).cuda()
    stt = torch.from_numpy(star).cuda() if star is not None else None
    lnl_d = eng.lnlike_batch(tht, stt).cpu().numpy()
    flux, mags, lnl_m = eng.model_batch(tht, stt)
    lnl_h = eng.lnlike_batch(th, star)
    torch.cuda.synchronize()
    return (lnl_d, lnl_h, lnl_m.cpu().numpy(), flux.cpu().numpy() if flux is not None else None,
            mags.cpu().numpy() if mags is not None else None)


@gpu
@pytest.mark.parametrize('name', list(SETUPS))
def test_star_layouts_bit_identical_to_single_star_engines(name):
    kw, stars, settings = _build(name)
    S = len(stars)
    multi = Engine(stars=stars, **kw)
    _apply(multi, settings)
    assert multi.star_ndim == [len(st['fitpars_i']) for st in stars] and multi.ndim == max(multi.star_ndim)
    assert multi.star_fitpars_i == [st['fitpars_i'] for st in stars]
    if name.startswith('cluster'):
        assert multi.query('tail_cluster') == 1
    B = 520
    star = _star_index(S, B)
    th = _rows(stars, star, multi.ndim, sum(map(ord, name)), np.nan)
    lnl_d, lnl_h, lnl_m, flux, mags = _eval(multi, th, star)
    assert multi.query('status') == 0
    n_finite = 0
    for k in range(S):
        idx = np.flatnonzero(star == k)
        one = _single(kw, stars[k], settings)
        own = np.ascontiguousarray(th[idx, :len(stars[k]['fitpars_i'])])
        ref_d, ref_h, ref_m, rf, rm = _eval(one, own, None)
        assert np.array_equal(lnl_d[idx], ref_d, equal_nan=True), (name, k)
        assert np.array_equal(lnl_h[idx], ref_h, equal_nan=True), (name, k)
        assert np.array_equal(lnl_m[idx], ref_m, equal_nan=True), (name, k)
        if flux is not None:
            n = len(stars[k]['wave'])
            assert np.array_equal(flux[idx, :n], rf, equal_nan=True), (name, k)
        if mags is not None:
            nbk = len(multi.star_bands[k])
            if rm is not None:
                assert multi.star_bands[k] == one.bands
                assert np.array_equal(mags[idx, :nbk], rm, equal_nan=True), (name, k)
            else:
                assert nbk == 0                                          # a star without photometry
            assert np.isnan(mags[idx, nbk:]).all()
        n_finite += int(np.isfinite(ref_d).sum())
        one.close()
    assert n_finite > B // 4
    # what the padding columns hold is never read
    th2 = th.copy()
    for p, k in enumerate(star):
        th2[p, len(stars[k]['fitpars_i']):] = 1e300
    out2 = _eval(multi, th2, star)
    for a, b in zip((lnl_d, lnl_h, lnl_m, flux, mags), out2):
        assert (a is None and b is None) or np.array_equal(a, b, equal_nan=True), name
    multi.close()


@gpu
def test_layouts_equal_to_the_context_layout_change_nothing():
    """Every star given a layout equal to the context's gives the bits of the same context without layouts."""
    spec = _spec('mini')
    net = synth.make_photnet(BANDS, H=16)
    stars = _stars(spec, True)
    fit = LABELS + ['Vrad', 'Vrot', 'log(A)', 'Av', 'pc_0', 'pc_1']
    kw = dict(spec=spec, phot=net, fitpars_i=fit, fixedpars={'Inst_R': 33000.0},
              runbools=[True, True, True, True, False])
    star = _star_index(len(stars), 300)
    plain = [dict(st, fitpars_i=fit) for st in stars]
    th = _rows(plain, star, len(fit), 6, np.nan)
    a = Engine(stars=stars, **kw)
    b = Engine(stars=[dict(st, runbools=[True, True, True, True]) for st in stars], **kw)   # forces layouts
    ra, rb = _eval(a, th, star), _eval(b, th, star)
    assert np.isfinite(ra[0]).sum() > 100
    for x, y in zip(ra, rb):
        assert np.array_equal(x, y, equal_nan=True)


# ------------------------------------------------------------------ refusals

def _create(spec, phot, stars, ctx, lays, fixed=None):
    """payne_ctx_create_stars_opts with a context layout and per-star layouts (None: none); fixed: per-star
    PayneStarOpts.fixed arrays (None: none)."""
    lib = _lib.load()
    keep = []
    sp = _specnet_struct(spec, keep) if spec is not None else None
    ph = None
    if phot is not None:
        ph = _lib.PaynePhotNet()
        arrs = [np.ascontiguousarray(x, dtype=np.float32) for x in
                (phot.w1, phot.b1, phot.w2, phot.b2, np.asarray(phot.w3).reshape(len(phot.bands), -1),
                 np.asarray(phot.b3).reshape(-1))]
        keep += arrs
        ph.nb, ph.H = arrs[0].shape[0], arrs[0].shape[1]
        ph.w1, ph.b1, ph.w2, ph.b2, ph.w3, ph.b3 = [x.ctypes.data_as(ctypes.POINTER(ctypes.c_float)) for x in arrs]
        d = [np.ascontiguousarray(x, dtype=np.float64) for x in (phot.xmin, phot.xmax, phot.hiav)]
        keep += d
        ph.xmin, ph.xmax, ph.hiav = [x.ctypes.data_as(ctypes.POINTER(ctypes.c_double)) for x in d]
    S = len(stars)
    obs = (_lib.PayneObs * S)()
    opts = (_lib.PayneStarOpts * S)()
    dp = lambda x: x.ctypes.data_as(ctypes.POINTER(ctypes.c_double))        # noqa: E731
    for k, st in enumerate(stars):
        if spec is not None:
            ow, of, oe = [np.ascontiguousarray(st[x], dtype=np.float64) for x in ('wave', 'flux', 'eflux')]
            keep += [ow, of, oe]
            obs[k].n_obs, obs[k].wave, obs[k].flux, obs[k].eflux = len(ow), dp(ow), dp(of), dp(oe)
        if st.get('mag') is not None:
            mag = np.ascontiguousarray(st['mag'], dtype=np.float64)
            err = np.full(len(mag), 0.05)
            keep += [mag, err]
            obs[k].nb, obs[k].phot_mag, obs[k].phot_err = len(mag), dp(mag), dp(err)
        if lays[k] is not None:
            opts[k].layout = ctypes.pointer(lays[k])
        if fixed is not None and fixed[k] is not None:
            v = np.ascontiguousarray(fixed[k], dtype=np.float64)
            keep.append(v)
            opts[k].fixed = dp(v)
    ctx_out = ctypes.c_void_p()
    rc = lib.payne_ctx_create_stars_opts(ctypes.byref(sp) if sp else None, ctypes.byref(ph) if ph else None, obs,
                                         opts, S, ctypes.byref(ctx), 0, ctypes.byref(ctx_out))
    return rc, ctx_out


@gpu
def test_refusals():
    lib = _lib.load()
    spec = _spec('mini')
    net = synth.make_photnet(BANDS, H=16)
    stars = _stars(spec, False)[:2]
    nan = np.full(_lib.NPAR, np.nan)
    fit = LABELS + ['Vrad', 'Vrot', 'pc_0', 'pc_1']
    rb = [True, False, True, False]
    ctx = _layout(fit, nan, rb, 'parity')

    def check(lay1, code, what, ctx_lay=ctx, st=stars, phot=None, fixed=None):
        rc, c = _create(spec if ctx_lay.spec_bool else None, phot, st, ctx_lay, [None, lay1], fixed)
        msg = lib.payne_last_error()
        if rc == 0:
            lib.payne_ctx_destroy(c)
        assert rc == code and what in msg, (what, rc, msg)

    ok = _layout(LABELS + ['Vrot', 'pc_0', 'pc_1', 'pc_2'], nan, rb, 'parity')
    check(ok, 0, b'')
    bad = _layout(fit, nan, rb, 'parity')
    bad.col[_lib.PAR_INDEX['Vrad']] = len(fit)
    check(bad, _INVALID, b'outside')
    bad = _layout(fit, nan, rb, 'parity')
    bad.col[_lib.PAR_INDEX['Vrad']] = 0
    check(bad, _INVALID, b'twice')
    bad = _layout(fit, nan, rb, 'parity')
    bad.poly_col[1] = -3
    check(bad, _INVALID, b'outside')
    bad = _layout(fit, nan, rb, 'parity')
    bad.poly_col[1] = bad.col[0]
    check(bad, _INVALID, b'twice')
    bad = _layout(fit, nan, rb, 'parity')
    bad.n_poly = _lib.MAX_POLY + 1
    check(bad, _INVALID, b'n_poly')
    check(_layout(fit, nan, rb, 'simt'), _INVALID, b'precision')
    check(_layout(fit, nan, [False, True, True, False], 'parity'), _INVALID, b'spec_bool')
    check(_layout(fit, nan, [True, True, True, False], 'parity'), _INVALID, b'photometry')
    check(_layout(fit, nan, rb, 'parity'), _INVALID, b'not both', fixed=[None, nan])
    # stars with and without a continuum polynomial
    check(_layout(LABELS + ['Vrad'], nan, [True, False, False, False], 'parity'), _UNSUPPORTED, b'polynomial')
    check(_layout(LABELS + ['Vrad'], nan, [True, False, True, False], 'parity'), _UNSUPPORTED, b'polynomial')
    # a star below the set's largest continuum order whose abscissae are not finite (one pixel); equal orders are fine
    one_px = [stars[0], dict(stars[1], wave=stars[1]['wave'][:1], flux=stars[1]['flux'][:1], eflux=stars[1]['eflux'][:1])]
    check(_layout(LABELS + ['Vrad', 'pc_0'], nan, rb, 'parity'), _UNSUPPORTED, b'abscissae', st=one_px)
    check(_layout(LABELS + ['Vrad', 'pc_0', 'pc_1'], nan, rb, 'parity'), 0, b'', st=one_px)
    # photometry-only context: a star with nothing to fit, a star without photometry that has magnitudes
    pctx = _layout(LABELS + ['log(A)', 'Av'], nan, [False, True, False, True], 'parity')
    two = [{'mag': [5.0, 6.0, 7.0, 8.0]}, {'mag': [5.0, 6.0, 7.0, 8.0]}]
    check(_layout(LABELS, nan, [False, False, False, False], 'parity'), _INVALID, b'nothing to fit', ctx_lay=pctx,
          st=two, phot=net)
    jctx = _layout(fit + ['log(A)', 'Av'], nan, [True, True, True, True], 'parity')
    jst = [dict(s, mag=[5.0, 6.0, 7.0, 8.0]) for s in stars]
    check(_layout(fit, nan, rb, 'parity'), _INVALID, b'nb', ctx_lay=jctx, st=jst, phot=net)
    # ld below the largest ndim
    eng = Engine(stars=[dict(stars[0], fitpars_i=fit), dict(stars[1], fitpars_i=fit + ['Vmic', 'Inst_R'])],
                 spec=spec, runbools=rb + [False])
    th = np.zeros((4, len(fit)))
    star = np.array([0, 1, 0, 1], dtype=np.int32)
    out = np.empty(4)
    assert lib.payne_lnlike_batch_stars_host(eng._ctx, th.ctypes.data, star.ctypes.data, 4, len(fit),
                                             out.ctypes.data) == _INVALID
    assert b'ld' in lib.payne_last_error()
    with pytest.raises(ValueError, match='columns|must be'):
        eng.lnlike_batch(th, star)
    eng.close()


@gpu
def test_layout_with_free_inst_r_after_switching_the_lsf_off():
    """A one-star context with a layout that samples Inst_R and an LSF vector: with the vector its rows give what the
    LSF engine gives, and after set_lsf(None) the Inst_R column is read again, as without a layout."""
    spec = _spec('mini')
    st = _stars(spec, False)[0]
    lsf = _lsf(st['wave'], 0)
    fit = LABELS + ['Vrad', 'Vrot', 'Inst_R', 'pc_0', 'pc_1']
    kw = dict(spec=spec, fitpars_i=fit, runbools=[True, False, True, False, False])
    eng = Engine(stars=[dict(st, fixedpars={'Inst_R': lsf}, runbools=[True, False, True, False])], **kw)
    assert eng.query('lsf') == 1
    th = _rows([{'fitpars_i': fit}], np.zeros(300, dtype=np.int32), len(fit), 9, np.nan)
    ref = Engine(obs_wave=st['wave'], obs_flux=st['flux'], obs_eflux=st['eflux'], **kw)
    ref.set_lsf(lsf)
    assert np.array_equal(eng.lnlike_batch(th, np.zeros(300, np.int32)), ref.lnlike_batch(th), equal_nan=True)
    eng.set_lsf(None)
    ref.set_lsf(None)
    got, want = eng.lnlike_batch(th, np.zeros(300, np.int32)), ref.lnlike_batch(th)
    assert np.isfinite(want).sum() > 100 and np.array_equal(got, want, equal_nan=True)
    eng.close()
    ref.close()


def test_star_opts_struct_matches_the_ctypes_mirror(tmp_path):
    """sizeof(PayneStarOpts) and the offset of its layout pointer, from the header compiled with the host C
    compiler, against the ctypes mirror (no GPU)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / 'opts.c'
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "payne_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu\\n", sizeof(PayneStarOpts), offsetof(PayneStarOpts, layout),'
                   ' sizeof(PayneLayout)); return 0; }\n')
    exe = tmp_path / 'opts'
    subprocess.run(['gcc', '-I', os.path.join(root, 'include'), '-o', str(exe), str(src)], check=True)
    size, off, lsize = map(int, subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split())
    assert size == ctypes.sizeof(_lib.PayneStarOpts)
    assert off == _lib.PayneStarOpts.layout.offset
    assert lsize == ctypes.sizeof(_lib.PayneLayout)
    assert _lib.ABI_VERSION == 8


# ------------------------------------------------------------------ FitPayneMany

@gpu
def test_fitpaynemany_heterogeneous_input_dicts(tmp_path):
    """Four input dictionaries with different continuum orders, photometry for some stars only, both photscale
    kinds and a fixed Vrad or Vrot on some: each output file is byte-identical to a separate FitPayne run."""
    from conftest import load_case
    from test_gpu_star_opts import _run_many
    cfg, _ = load_case('mini_joint')
    n = len(cfg.obs_wave)
    sels = [slice(0, n), slice(n // 5, n - n // 7), slice(0, n // 2), slice(n // 3, n)]
    polyorder = [1, 3, 2, 4]
    phot = [list(cfg.obs_phot), None, ['2MASS_J', 'Bessell_V'], None]
    photscale = [True, False, False, False]
    fixed = [{}, {'Vrad': 12.0}, {'Vrot': 4.0}, {'Vrad': -3.0, 'Vrot': 0.0}]
    dicts = []
    box = dict(synth._BOX, **cfg.box)
    for k in range(4):
        free = LABELS + ['Vrad', 'Vrot']
        if phot[k] is not None:
            free += ['log(A)', 'Av'] if photscale[k] else ['log(R)', 'Dist', 'Av']
        pri = {p: {'pv_uniform': list(box[p])} for p in free}
        pri['Inst_R'] = {'fixed': 32000.0 + 1000.0 * k}
        for p, v in fixed[k].items():
            pri[p] = {'fixed': v}
        d = {'spec': {'obs_wave': cfg.obs_wave[sels[k]], 'obs_flux': cfg.obs_flux[sels[k]],
                      'obs_eflux': cfg.obs_eflux[sels[k]], 'convertair': False, 'modpoly': True,
                      'polyorder': polyorder[k], 'polysigma': 0.05},
             'specANNpath': cfg.spec, 'NNtype': 'LinNet', 'sampler': _sampler(400 + k, [50, 35, 45, 30][k]),
             'priordict': pri}
        if phot[k] is not None:
            d.update(phot={b: cfg.obs_phot[b] for b in phot[k]}, photANNpath=cfg.phot, photscale=photscale[k])
        dicts.append(d)
    many = _run_many(tmp_path, dicts)
    eng = many.likeobj.engine
    assert eng.star_ndim == [len(f.likeobj.fitpars_i) for f in many.fits]
    assert len(set(eng.star_ndim)) > 1 and eng.star_bands[1] == [] and eng.star_bands[3] == []
