"""Measurement: double-lined binaries (payne_lnlike_batch_binary) against one star and against the host workaround.

Workload: the C2 emulator (LinNet 4-256-256-256-14172, SURVEY §8d) and 7000 observed pixels across its coverage; the
primary samples Teff, log(g), [Fe/H], [a/Fe], Vrad, Vrot and Inst_R, the secondary its own Teff, log(g), Vrad and Vrot,
and Rratio.  For B points three calls are timed on one context:

  binary      one payne_lnlike_batch_binary call of B rows (2 B emulator rows, two tail passes per point);
  single      one payne_lnlike_batch call of B rows (the primary alone);
  workaround  what a user had to do before: two payne_model_batch calls (the primary's and the secondary's parameters),
              both model arrays copied to the host, the components combined and chi2 summed in numpy.

CUDA events around every call (for the workaround the end event is recorded after the host work, so it spans it),
median over --reps rounds with the three calls alternating within a round, after a warm-up of each.  The binary and
workaround lnL must agree to 1e-9 relative.  The GPU name and power limit are read in the same run.

usage: python tools/gpu_binary.py [--out DIR] [--bs 512,4096] [--reps 20]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from thepayne_b200 import synth  # noqa: E402
from thepayne_b200.engine import Engine  # noqa: E402
from gpu_multistar import gpu_info  # noqa: E402

PRIM = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot', 'Inst_R']
SEC = {'Teff_sec': 'Teff', 'log(g)_sec': 'log(g)', 'Vrad_sec': 'Vrad', 'Vrot_sec': 'Vrot'}
FIT = PRIM + list(SEC) + ['Rratio']
C2_RAD = 1.438776877e8
BOX = dict(synth._BOX, Vrad=(-30.0, 30.0), Teff_sec=(3800.0, 5500.0), Vrad_sec=(-60.0, 60.0), Vrot_sec=(0.0, 5.0),
           Rratio=(0.3, 0.9), **{'log(g)_sec': (4.3, 5.0)})


def draw(B, seed):
    rng = np.random.default_rng(seed)
    th = np.empty((B, len(FIT)))
    for i, p in enumerate(FIT):
        th[:, i] = BOX[p][0] + (BOX[p][1] - BOX[p][0]) * rng.random(B)
    return th


def secondary_rows(th):
    out = th.clone()
    for s, p in SEC.items():
        out[:, FIT.index(p)] = th[:, FIT.index(s)]
    return out


def workaround(eng, th, th2, w, f, e):
    """two model calls, the copies to the host, the combination and chi2 there"""
    a1 = eng.model_batch(th, want_mags=False)[0].cpu().numpy()
    a2 = eng.model_batch(th2, want_mags=False)[0].cpu().numpy()
    t = th.cpu().numpy()
    t1, t2, rr = t[:, FIT.index('Teff'), None], t[:, FIT.index('Teff_sec'), None], t[:, FIT.index('Rratio'), None]
    k = rr ** 2 * np.expm1(C2_RAD / (w * t1)) / np.expm1(C2_RAD / (w * t2))
    m = (a1 + k * a2) / (1.0 + k)
    return -0.5 * np.sum(((m - f) ** 2) / (e ** 2), axis=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--bs', default='512,4096')
    ap.add_argument('--reps', type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('gpu_binary.py needs a CUDA device')
    wave, rsig = synth.ann_wavegrid(5130.0, 5340.0, 50000.0)              # C2 (synth.config_c2)
    spec = synth.make_specnet(4, 256, wave, rsig, seed=0)
    info = gpu_info()
    print('gpu:', json.dumps(info))
    a, b = wave[0], wave[-1]
    w = np.linspace(a + 0.04 * (b - a), b - 0.04 * (b - a), 7000)
    rng = np.random.default_rng(1)
    f, e = 1.0 + 0.02 * rng.standard_normal(len(w)), np.full(len(w), 0.02)
    eng = Engine(spec=spec, obs_wave=w, obs_flux=f, obs_eflux=e, fitpars_i=FIT, precision='parity', binary=True)
    rows = []
    for B in [int(v) for v in args.bs.split(',')]:
        eng.set('max_batch', max(8192, 2 * B))                   # one slab for every call
        th = torch.from_numpy(draw(B, B)).cuda()
        th2 = secondary_rows(th)
        out = {}
        calls = {'binary': lambda: out.__setitem__('b', eng.lnlike_batch_binary(th)),
                 'single': lambda: out.__setitem__('s', eng.lnlike_batch(th)),
                 'workaround': lambda: out.__setitem__('w', workaround(eng, th, th2, w, f, e))}
        for fn in list(calls.values()) * 2:
            fn()
        torch.cuda.synchronize()
        lb, lw = out['b'].cpu().numpy(), out['w']
        agree = bool(np.all(np.abs(lb - lw) <= 1e-9 * np.abs(lw)))
        ms = {k: [] for k in calls}
        for _ in range(args.reps):
            for k, fn in calls.items():
                s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                fn()
                t.record()
                torch.cuda.synchronize()
                ms[k].append(s.elapsed_time(t))
        row = {'B': B, 'agree_1e-9': agree, 'max_rel_dlnl': float(np.max(np.abs(lb - lw) / np.abs(lw)))}
        row.update({k + '_ms': float(np.median(v)) for k, v in ms.items()})
        row['binary_over_single'] = row['binary_ms'] / row['single_ms']
        row['workaround_over_binary'] = row['workaround_ms'] / row['binary_ms']
        rows.append(row)
        print('B=%5d  binary %.3f ms  single %.3f ms (x%.2f)  workaround %.3f ms (x%.2f of binary)  lnL agree: %s '
              '(max rel %.1e)' % (B, row['binary_ms'], row['single_ms'], row['binary_over_single'],
                                  row['workaround_ms'], row['workaround_over_binary'], agree, row['max_rel_dlnl']),
              flush=True)
    eng.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'binary.json'), 'w') as fo:
            json.dump({'gpu': info, 'rows': rows}, fo, indent=1)
    if not all(r['agree_1e-9'] for r in rows):
        sys.exit('binary and workaround lnL differ')


if __name__ == '__main__':
    main()
