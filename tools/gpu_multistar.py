"""Measurement: one multi-star call against K single-star calls (observation sets, payne_ctx_create_stars).

Workload: the C2 emulator (LinNet 4-256-256-256-14172, SURVEY §8d) with K stars.  Each star has its own observed
grid inside the emulator coverage; the grids differ in range and n_obs (3000 .. 7000 pixels).  For every K and
per-star batch b three cases are timed:

  multi    one payne_lnlike_batch_stars call of K*b points (stars concatenated, as FitPayneMany makes them);
  singles  K payne_lnlike_batch calls of b points each, on K single-star contexts, one stream;
  ceiling  one single-star call of K*b points (star 0's context): the rate the GPU reaches at that size.

Device time: CUDA events around the case, median over --reps repetitions.  Host-entry time: a host clock around
the case and a device synchronise (what a sampler waiting for its lnL sees), median.  Inputs are drawn once per
(K, b); every case is warmed up before it is timed.  The GPU name and power limit are read in the same run.

--lsf: every star brings its own LSF vector (a fixed Inst_R array, payne_ctx_create_stars_opts), the single-star
contexts too; every row then also records the LSF tail's device time per point (payne_ctx_last_ms(..., 1) of one
multi-star call over its points).

--layouts: every star has its own parameter layout (PayneStarOpts.layout), on the C2 emulator plus the C3 photometry
net (7 bands, H = 128): continuum polynomials of 2 to 6 coefficients (star k: 2 + k % 5), photometry for every third
star (alternately log(A) and log(R) + Dist), Vrad fixed on stars k % 4 == 1 and Vrot on k % 4 == 2; every single-star
context has its star's own layout and theta rows its own columns.  A second set is the same with star 0's polynomial
raised to 16 coefficients (every star's polynomial is evaluated to the set's largest order).  Besides the three cases,
each row records the per-kernel device time (payne_ctx_last_ms: emulator, tail, photometry; median over --reps calls)
of the mixed call and of calls of the same size on one context whose stars all have one layout (every spectral
parameter free, no photometry, 2, 6 and 16 coefficients).

usage: python tools/gpu_multistar.py [--out DIR] [--ks 1,4,16,64] [--bs 64,128,256,512] [--reps 30] [--lsf | --layouts]
Prints one line per (K, b) and the GPU record; with --out DIR it also writes every row to DIR/multistar.json.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from thepayne_b200 import synth  # noqa: E402
from thepayne_b200.engine import Engine  # noqa: E402

FIT = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Inst_R']


def gpu_info():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().split('\n')[0]
        info['nvidia_smi'] = out
    except Exception as e:                              # noqa: BLE001 -- recorded, not fatal
        info['nvidia_smi'] = 'unavailable: %s' % e
    return info


def make_stars(spec, K, seed=1):
    w = spec.wavelength
    a, b = w[0], w[-1]
    span = b - a
    rng = np.random.default_rng(seed)
    stars = []
    for k in range(K):
        lo = a + span * (0.04 + 0.10 * rng.random())
        hi = b - span * (0.04 + 0.10 * rng.random())
        n = int(rng.integers(3000, 7001))
        g = np.linspace(lo, hi, n)
        stars.append({'wave': g, 'flux': 1.0 + 0.02 * rng.standard_normal(n), 'eflux': np.full(n, 0.02), 'phot': None})
    return stars


def draw(B, seed):
    box = synth._BOX
    rng = np.random.default_rng(seed)
    lo = np.array([box[p][0] for p in FIT])
    hi = np.array([box[p][1] for p in FIT])
    return lo + (hi - lo) * rng.random((B, len(FIT)))


def draw_fit(fit, B, rng):
    box = dict(synth._BOX, **{p: ((0.75, 1.25) if p == 'pc_0' else (-0.05, 0.05)) for p in fit if p.startswith('pc_')})
    lo = np.array([box[p][0] for p in fit])
    hi = np.array([box[p][1] for p in fit])
    return lo + (hi - lo) * rng.random((B, len(fit)))


def star_layout(k, npoly):
    """--layouts: star k's free parameters, run booleans and fixed values"""
    fit = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]'] + [p for i, p in ((1, 'Vrad'), (2, 'Vrot')) if k % 4 != i] + ['Inst_R']
    fixed = {'Vrad': 5.0} if k % 4 == 1 else {'Vrot': 3.0} if k % 4 == 2 else {}
    phot = k % 3 == 0
    scaled = phot and (k // 3) % 2 == 0
    if phot:
        fit += ['log(A)', 'Av'] if scaled else ['log(R)', 'Dist', 'Av']
    fit += ['pc_%d' % i for i in range(npoly)]
    return fit, [True, phot, True, scaled], fixed


def kernel_ms(eng, th, star, reps):
    """median per-kernel device time (emulator, tail, photometry) of one call"""
    eng.set('timing', 1)
    rows = []
    for _ in range(reps):
        eng.lnlike_batch(th, star)
        torch.cuda.synchronize()
        rows.append([max(0.0, eng.last_ms(w)) for w in ('mlp', 'tail', 'phot')])
    eng.set('timing', 0)
    return [float(v) for v in np.median(np.array(rows), axis=0)]


def run_layouts(args, spec, ks, bs):
    phot = synth.make_photnet(synth.PROCYON_BANDS, H=128)                   # C3 (synth.config_c3)
    kmax = max(ks)
    base = make_stars(spec, kmax)
    obs_phot = {b: (6.0 + 0.1 * i, 0.03) for i, b in enumerate(synth.PROCYON_BANDS)}
    rows = []
    for label, high in (('mixed n_poly 2-6', False), ('mixed n_poly 2-6, star 0 at 16', True)):
        stars = []
        for k, s in enumerate(base):
            fit, rb, fixed = star_layout(k, 16 if (high and k == 0) else 2 + k % 5)
            stars.append(dict(s, fitpars_i=fit, runbools=rb, fixedpars=fixed, phot=obs_phot if rb[1] else None))
        singles = [Engine(obs_wave=s['wave'], obs_flux=s['flux'], obs_eflux=s['eflux'], obs_phot=s['phot'],
                          spec=spec, phot=phot if s['runbools'][1] else None, fitpars_i=s['fitpars_i'],
                          fixedpars=s['fixedpars'], runbools=s['runbools'] + [False], precision='parity')
                   for s in stars]
        for K in ks:
            multi = Engine(stars=stars[:K], spec=spec, phot=phot, runbools=[True, True, True, False, False],
                           precision='parity')
            for b in bs:
                rng = np.random.default_rng(K * 1000 + b)
                parts_np = [draw_fit(stars[k]['fitpars_i'], b, rng) for k in range(K)]
                th_np = np.full((K * b, multi.ndim), np.nan)
                for k in range(K):
                    th_np[k * b:(k + 1) * b, :parts_np[k].shape[1]] = parts_np[k]
                th = torch.from_numpy(th_np).cuda()
                parts = [torch.from_numpy(p).cuda() for p in parts_np]
                star = torch.repeat_interleave(torch.arange(K, dtype=torch.int32), b).cuda()
                th0 = torch.from_numpy(draw_fit(stars[0]['fitpars_i'], K * b, rng)).cuda()
                res = {'set': label, 'K': K, 'b': b, 'points': K * b}
                res['multi_dev_ms'], res['multi_host_ms'], res['multi_dev_min_ms'] = time_case(
                    lambda: multi.lnlike_batch(th, star), args.reps)
                res['singles_dev_ms'], res['singles_host_ms'], res['singles_dev_min_ms'] = time_case(
                    lambda: [singles[k].lnlike_batch(parts[k]) for k in range(K)], args.reps)
                res['ceiling_dev_ms'], res['ceiling_host_ms'], res['ceiling_dev_min_ms'] = time_case(
                    lambda: singles[0].lnlike_batch(th0), args.reps)
                got = multi.lnlike_batch(th, star)
                ref = torch.cat([singles[k].lnlike_batch(parts[k]) for k in range(K)])
                torch.cuda.synchronize()
                res['bit_identical'] = bool(torch.equal(torch.nan_to_num(got, nan=1.5), torch.nan_to_num(ref, nan=1.5)))
                res['kernel_ms_mixed'] = kernel_ms(multi, th, star, args.reps)
                for npoly in (2, 6, 16):                       # one layout for every star, same size
                    fit = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Inst_R'] + ['pc_%d' % i for i in range(npoly)]
                    uni = Engine(stars=[{x: s[x] for x in ('wave', 'flux', 'eflux')} for s in stars[:K]], spec=spec, fitpars_i=fit,
                                 runbools=[True, False, True, False, False], precision='parity')
                    thu = torch.from_numpy(draw_fit(fit, K * b, rng)).cuda()
                    res['kernel_ms_uniform_%d' % npoly] = kernel_ms(uni, thu, star, args.reps)
                    uni.close()
                rows.append(res)
                km = res['kernel_ms_mixed']
                print('%s K=%3d b=%4d  multi %.3f ms dev / %.3f host | %d singles %.3f / %.3f | ceiling %.3f / %.3f | '
                      'x%.2f host  %s | kernels mlp/tail/phot ms: mixed %.3f/%.3f/%.3f  uniform 2: %.3f/%.3f  '
                      '6: %.3f/%.3f  16: %.3f/%.3f' % (
                          label, K, b, res['multi_dev_ms'], res['multi_host_ms'], K, res['singles_dev_ms'],
                          res['singles_host_ms'], res['ceiling_dev_ms'], res['ceiling_host_ms'],
                          res['singles_host_ms'] / res['multi_host_ms'],
                          'bit-identical' if res['bit_identical'] else 'DIFFERENT', km[0], km[1], km[2],
                          *res['kernel_ms_uniform_2'][:2], *res['kernel_ms_uniform_6'][:2],
                          *res['kernel_ms_uniform_16'][:2]), flush=True)
            multi.close()
        for e in singles:
            e.close()
    return rows


def time_case(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    dev, host = [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        host.append((time.perf_counter() - t0) * 1e3)
        dev.append(e0.elapsed_time(e1))
    return float(np.median(dev)), float(np.median(host)), float(np.min(dev))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None, help='directory for multistar.json (default: print only)')
    ap.add_argument('--ks', default='1,4,16,64')
    ap.add_argument('--bs', default='64,128,256,512')
    ap.add_argument('--reps', type=int, default=30)
    ap.add_argument('--lsf', action='store_true', help='per-star LSF vectors (the LSF tail)')
    ap.add_argument('--layouts', action='store_true', help='per-star parameter layouts, C2 + C3 photometry net')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('gpu_multistar.py measures on the GPU: no CUDA device')
    ks = [int(v) for v in args.ks.split(',')]
    bs = [int(v) for v in args.bs.split(',')]
    wave, rsig = synth.ann_wavegrid(5130.0, 5340.0, 50000.0)              # C2 (synth.config_c2)
    spec = synth.make_specnet(4, 256, wave, rsig, seed=0)
    if args.layouts:
        rows = run_layouts(args, spec, ks, bs)
        doc = {'gpu': gpu_info(), 'workload': 'C2 emulator + C3 photometry net, per-star layouts, parity',
               'reps': args.reps, 'rows': rows}
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, 'multistar_layouts.json'), 'w') as f:
                json.dump(doc, f, indent=1)
        print(json.dumps(doc['gpu']))
        return
    kw = dict(spec=spec, fitpars_i=FIT, fixedpars={}, runbools=[True, False, False, False, False], precision='parity')
    Kmax = max(ks)
    all_stars = make_stars(spec, Kmax)
    if args.lsf:
        for k, s in enumerate(all_stars):
            g = s['wave']
            s['fixedpars'] = {'Inst_R': 0.04 + 0.002 * (k % 5) + 0.01 * (g - g[0]) / (g[-1] - g[0])}
    singles = [Engine(obs_wave=s['wave'], obs_flux=s['flux'], obs_eflux=s['eflux'],
                      **dict(kw, fixedpars=s.get('fixedpars', {}))) for s in all_stars]
    rows = []
    for K in ks:
        multi = Engine(stars=all_stars[:K], **kw)
        for b in bs:
            th = torch.from_numpy(draw(K * b, seed=K * 1000 + b)).cuda()
            star = torch.repeat_interleave(torch.arange(K, dtype=torch.int32), b).cuda()
            parts = [th[k * b:(k + 1) * b] for k in range(K)]
            res = {'K': K, 'b': b, 'points': K * b}
            res['multi_dev_ms'], res['multi_host_ms'], res['multi_dev_min_ms'] = time_case(
                lambda: multi.lnlike_batch(th, star), args.reps)
            res['singles_dev_ms'], res['singles_host_ms'], res['singles_dev_min_ms'] = time_case(
                lambda: [singles[k].lnlike_batch(parts[k]) for k in range(K)], args.reps)
            res['ceiling_dev_ms'], res['ceiling_host_ms'], res['ceiling_dev_min_ms'] = time_case(
                lambda: singles[0].lnlike_batch(th), args.reps)
            # same answers: the multi-star call against the K single-star calls
            got = multi.lnlike_batch(th, star)
            ref = torch.cat([singles[k].lnlike_batch(parts[k]) for k in range(K)])
            torch.cuda.synchronize()
            res['bit_identical'] = bool(torch.equal(torch.nan_to_num(got, nan=1.5), torch.nan_to_num(ref, nan=1.5)))
            res['speedup_host'] = res['singles_host_ms'] / res['multi_host_ms']
            res['speedup_dev'] = res['singles_dev_ms'] / res['multi_dev_ms']
            res['multi_over_ceiling_dev'] = res['multi_dev_ms'] / res['ceiling_dev_ms']
            res['multi_Mevals_s'] = K * b / res['multi_host_ms'] / 1e3
            if args.lsf:
                multi.set('timing', 1)
                multi.lnlike_batch(th, star)
                res['lsf_tail_us_per_point'] = 1e3 * multi.last_ms('tail') / (K * b)
                multi.set('timing', 0)
                print('K=%3d b=%4d  LSF tail %.1f us per point' % (K, b, res['lsf_tail_us_per_point']), flush=True)
            rows.append(res)
            print('K=%3d b=%4d  multi %.3f ms dev / %.3f ms host | %d singles %.3f / %.3f | ceiling %.3f / %.3f | '
                  'x%.2f host  x%.2f dev  multi/ceiling %.3f  %s' % (
                      K, b, res['multi_dev_ms'], res['multi_host_ms'], K, res['singles_dev_ms'], res['singles_host_ms'],
                      res['ceiling_dev_ms'], res['ceiling_host_ms'], res['speedup_host'], res['speedup_dev'],
                      res['multi_over_ceiling_dev'], 'bit-identical' if res['bit_identical'] else 'DIFFERENT'),
                  flush=True)
        multi.close()
    for e in singles:
        e.close()
    doc = {'gpu': gpu_info(), 'workload': 'C2 emulator LinNet 4-256-256-256-14172, per-star n_obs 3000-7000, parity' +
           (', per-star LSF vectors' if args.lsf else ''),
           'reps': args.reps, 'rows': rows}
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'multistar.json'), 'w') as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc['gpu']))


if __name__ == '__main__':
    main()
