"""Measurement: continuum marginalisation (payne_ctx_set_cont_marg) against sampled continuum coefficients.

1. Tail time on the C2 emulator (LinNet 4-256-256-256-14172, 7000 observed pixels), B = 4096: a context that
   integrates K coefficients out against one that samples the same K, fed the same theta (the sampled one with the
   marginal c-hat appended), K in {1, 3, 5, 8, 16}.  payne_ctx_last_ms(tail) medians over --reps calls, alternating.
2. An 8-member target (8 orders splitting the 7000 pixels), K = 4 per member, the same comparison through the target
   entries.
3. FitPayne on a mock problem (one spectrum, polyorder 3) and on the same pixels as an 8-order echelle spectrum
   (polyorder 3 per order, Inst_R fixed; three sampler settings), sampled against marginal coefficients with the same
   seed: ndim, iterations, likelihood calls, wall time and log Z +- its error.

The GPU name and power limit are read in the same run.

usage: python tools/gpu_cont_marg.py [--out DIR] [--reps 30] [--no-fit]
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from thepayne_b200 import synth  # noqa: E402
from thepayne_b200.engine import Engine  # noqa: E402
from gpu_multistar import gpu_info  # noqa: E402

FIT = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Inst_R']
BOX = dict(synth._BOX, Vrad=(-30.0, 30.0), Vrot=(0.5, 12.0))


def draw(B, seed):
    rng = np.random.default_rng(seed)
    return np.stack([BOX[p][0] + (BOX[p][1] - BOX[p][0]) * rng.random(B) for p in FIT], axis=1)


def cbox(K):
    return [(0.75, 1.25)] + [(-0.5, 0.5)] * (K - 1)


def tail_ms(eng, fn, reps):
    eng.set('timing', 1)
    out = []
    for _ in range(reps):
        fn()
        torch.cuda.synchronize()
        out.append(eng.last_ms('tail'))
    return out


def compare(marg, samp, call_m, call_s, reps):
    call_m(), call_s()                                        # warm-up
    mm, ms = [], []
    for _ in range(reps):
        mm += tail_ms(marg, call_m, 1)
        ms += tail_ms(samp, call_s, 1)
    return float(np.median(mm)), float(np.median(ms))


def star_rows(spec, w, f, e, B, reps):
    rows = []
    th = torch.from_numpy(draw(B, 1)).cuda()
    for K in (1, 3, 5, 8, 16):
        marg = Engine(spec=spec, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=FIT, cont_box=cbox(K))
        samp = Engine(spec=spec, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=FIT + ['pc_%d' % k for k in range(K)],
                      runbools=[True, False, True, False, False])
        for eng in (marg, samp):
            eng.set('max_batch', B)
        coef = marg.cont_batch(th)[0]
        ths = torch.cat([th, coef], dim=1).contiguous()
        tm, ts = compare(marg, samp, lambda: marg.lnlike_batch(th), lambda: samp.lnlike_batch(ths), reps)
        rows.append({'K': K, 'marginal_tail_ms': tm, 'sampled_tail_ms': ts, 'ratio': tm / ts})
        print('K=%2d  marginal tail %.3f ms  sampled tail %.3f ms  (x%.3f)' % (K, tm, ts, tm / ts), flush=True)
        marg.close(), samp.close()
    return rows


def target_row(spec, w, f, e, B, reps, K=4, n=8):
    fit = FIT[:6]
    edges = np.linspace(0, len(w), n + 1).astype(int)
    stars = []
    for s in range(n):
        sl = slice(edges[s], edges[s + 1])
        stars.append({'wave': w[sl], 'flux': f[sl], 'eflux': e[sl], 'fitpars_i': fit + ['Inst_R'],
                      'runbools': [True, False, False, False]})
    marg = Engine(spec=spec, stars=[dict(st, cont_box=cbox(K)) for st in stars], targets=[n])
    sfit = fit + ['Inst_R'] + ['pc_%d' % k for k in range(K)]
    samp = Engine(spec=spec, stars=[dict(st, fitpars_i=sfit, runbools=[True, False, True, False]) for st in stars],
                  targets=[n])
    for eng in (marg, samp):
        eng.set('max_batch', B)
    th = torch.from_numpy(draw(B, 2)).cuda()
    tg = torch.zeros(B, dtype=torch.int32, device='cuda')
    tm, ts = compare(marg, samp, lambda: marg.lnlike_batch_targets(th, tg), lambda: samp.lnlike_batch_targets(
        torch.cat([th, torch.full((B, K), 0.0, dtype=torch.float64, device='cuda')], dim=1), tg), reps)
    print('target of %d members, K=%d: marginal tail %.3f ms  sampled tail %.3f ms  (x%.3f)' % (n, K, tm, ts, tm / ts),
          flush=True)
    return {'members': n, 'K': K, 'marginal_tail_ms': tm, 'sampled_tail_ms': ts, 'ratio': tm / ts}


def fit_rows():
    from thepayne_b200.fitting.fitstar import FitPayne
    wave, rsig = synth.ann_wavegrid(5140.0, 5190.0, 50000.0)
    spec = synth.make_specnet(4, 64, wave, rsig, seed=0)
    truth = [5770.0, 4.44, 0.0, 0.0, 0.5, 3.0, 32000.0]
    w = np.linspace(5150.0, 5180.0, 1500)
    one = Engine(spec=spec, obs_wave=w, obs_flux=np.ones(len(w)), obs_eflux=np.ones(len(w)), fitpars_i=FIT)
    f = one.model_batch(np.array([truth]), want_mags=False)[0].cpu().numpy()[0]
    one.close()
    x = 2.0 * (w - w[0]) / (w[-1] - w[0]) - 1.0
    f = f * np.polynomial.chebyshev.chebval(x, [1.0, 0.02, -0.01, 0.005])
    e = np.abs(f) / 50.0
    obs = f + e * np.random.default_rng(3).standard_normal(len(w))
    pri = {'Teff': {'pv_uniform': [5400.0, 6100.0]}, 'log(g)': {'pv_uniform': [4.0, 4.8]},
           '[Fe/H]': {'pv_uniform': [-0.1, 0.1]}, '[a/Fe]': {'pv_uniform': [-0.1, 0.1]},
           'Vrad': {'pv_uniform': [-3.0, 3.0]}, 'Vrot': {'fixed': 3.0}, 'Inst_R': {'pv_uniform': [24000.0, 40000.0]}}
    rows = []
    for marginal in (False, True):
        sp = {'obs_wave': w, 'obs_flux': obs, 'obs_eflux': e, 'convertair': False, 'modpoly': True, 'polyorder': 3,
              'polysigma': 0.1, 'modpoly_marginal': marginal}
        with tempfile.TemporaryDirectory() as d:
            fp = FitPayne()
            t0 = time.time()
            smp = fp.run(inputdict={'spec': sp, 'specANNpath': spec, 'priordict': dict(pri),
                                    'output': os.path.join(d, 'o.dat'),
                                    'sampler': {'npoints': 200, 'walks': 25, 'delta_logz_final': 0.1, 'seed': 7}},
                         verbose=False)
            wall = time.time() - t0
        row = {'marginal': marginal, 'ndim': fp.ndim, 'iterations': int(smp.it), 'lnl_calls': int(smp.ncall),
               'wall_s': wall, 'logz': float(smp.logz), 'logz_err': float(np.sqrt(max(smp.logzvar, 0.0)))}
        rows.append(row)
        print('FitPayne %s: %s' % ('marginal' if marginal else 'sampled', json.dumps(row)), flush=True)
    # an 8-order echelle spectrum (list-valued spec), polyorder 3 in every order: 32 continuum coefficients
    orders = np.linspace(5150.0, 5180.0, 9)
    specs = []
    for s_ in range(8):
        sel = (w >= orders[s_]) & (w < orders[s_ + 1])
        specs.append({'obs_wave': w[sel], 'obs_flux': obs[sel], 'obs_eflux': e[sel], 'convertair': False,
                      'modpoly': True, 'polyorder': 3, 'polysigma': 0.1})
    pri8 = {k: v for k, v in pri.items() if k != 'Inst_R'}
    pri8.update({'Inst_R_%d' % s_: {'fixed': 32000.0} for s_ in range(8)})
    # rwalk in 37 dimensions needs many walks before the sampled run's log Z settles: three sampler settings
    for walks, npoints in ((25, 100), (100, 200), (400, 200)):
        for marginal in (False, True):
            for sp in specs:
                sp['modpoly_marginal'] = marginal
            with tempfile.TemporaryDirectory() as d:
                fp = FitPayne()
                t0 = time.time()
                smp = fp.run(inputdict={'spec': specs, 'specANNpath': spec, 'priordict': dict(pri8),
                                        'output': os.path.join(d, 'o.dat'),
                                        'sampler': {'npoints': npoints, 'walks': walks, 'delta_logz_final': 0.5,
                                                    'seed': 7}},
                             verbose=False)
                wall = time.time() - t0
            row = {'echelle_orders': 8, 'walks': walks, 'npoints': npoints, 'marginal': marginal, 'ndim': fp.ndim,
                   'iterations': int(smp.it), 'lnl_calls': int(smp.ncall), 'wall_s': wall, 'logz': float(smp.logz),
                   'logz_err': float(np.sqrt(max(smp.logzvar, 0.0)))}
            rows.append(row)
            print('FitPayne 8 orders %s: %s' % ('marginal' if marginal else 'sampled', json.dumps(row)), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--reps', type=int, default=30)
    ap.add_argument('--no-fit', action='store_true')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('gpu_cont_marg.py needs a CUDA device')
    info = gpu_info()
    print('gpu:', json.dumps(info))
    wave, rsig = synth.ann_wavegrid(5130.0, 5340.0, 50000.0)              # C2 (synth.config_c2)
    spec = synth.make_specnet(4, 256, wave, rsig, seed=0)
    a, b = wave[0], wave[-1]
    w = np.linspace(a + 0.04 * (b - a), b - 0.04 * (b - a), 7000)
    rng = np.random.default_rng(1)
    x = 2.0 * (w - w[0]) / (w[-1] - w[0]) - 1.0
    f, e = (1.0 + 0.02 * x) * (1.0 + 0.02 * rng.standard_normal(len(w))), np.full(len(w), 0.02)
    res = {'gpu': info, 'stars': star_rows(spec, w, f, e, 4096, args.reps),
           'target': target_row(spec, w, f, e, 4096, args.reps)}
    if not args.no_fit:
        res['fit'] = fit_rows()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'cont_marg.json'), 'w') as fo:
            json.dump(res, fo, indent=1)


if __name__ == '__main__':
    main()
