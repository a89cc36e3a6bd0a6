"""Measurement: targets (one star observed in K spectra, payne_ctx_set_targets) against the duplicated-row workaround.

Workload: the C2 emulator (LinNet 4-256-256-256-14172, SURVEY §8d) and one target of K spectra (K = 1, 2, 4, 8), the
echelle-order case: member m observes the m-th of K consecutive slices of the emulator's coverage, 7000 / K pixels
each, with its own Inst_R column; the labels, Vrad and Vrot are shared.  For B points two cases of the same work are
timed on one context (the K members as the stars of an observation set):

  targets     one payne_lnlike_batch_targets call of B rows (one emulator row and one rotation stage per row, then
              stage 2, the final pass and chi2 once per member);
  duplicated  one payne_lnlike_batch_stars call of K*B rows: every theta row repeated K times, row p*K + m naming member m,
              the K lnL of a point summed on the host in member order -- what a user had to do before targets.

Per kernel: payne_ctx_last_ms (device events around the emulator -- the continuum emulator
included -- and around the tail), median over --reps calls.  Per call: CUDA events around the call, median.  The two
cases must give the same lnL bits (checked on every (K, B)).  Inputs are drawn once per (K, B) and every case is
warmed up before it is timed.  The GPU name and power limit are read in the same run.

--lsf: every member has its own LSF vector (a fixed Inst_R array, the shape of test_gpu_star_opts._lsf) and its own
Vrad column in place of the Inst_R column; the labels and Vrot are shared.  Each member's LSF mask reaches 2000 AA past
its pixels, so its LSF stage spans about the whole emulator grid whatever its slice: targets save the K-1 emulator
rows and rotation stages per point, not LSF work.

usage: python tools/gpu_targets.py [--out DIR] [--ks 1,2,4,8] [--bs 512,4096] [--reps 30] [--lsf]
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

SHARED = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrad', 'Vrot']
SHARED_LSF = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]', 'Vrot']


def lsf_vector(wave, k):
    return 0.035 + 0.004 * k + 0.01 * (wave - wave.min()) / (wave.max() - wave.min()) + 0.003 * np.sin(wave / 2.0)


def members(spec, K, lsf=False, seed=1):
    w = spec.wavelength
    a, b = w[0], w[-1]
    lo, hi = a + 0.04 * (b - a), b - 0.04 * (b - a)
    edges = np.linspace(lo, hi, K + 1)
    rng = np.random.default_rng(seed)
    n = 7000 // K
    out = []
    for m in range(K):
        g = np.linspace(edges[m], edges[m + 1], n)
        st = {'wave': g, 'flux': 1.0 + 0.02 * rng.standard_normal(n), 'eflux': np.full(n, 0.02),
              'runbools': [True, False, False, False]}
        if lsf:                                           # member m's Vrad in column 5 + m
            st['fitpars_i'] = SHARED_LSF + ['pad'] * m + ['Vrad']
            st['fixedpars'] = {'Inst_R': lsf_vector(g, m)}
        else:                                             # member m's Inst_R in column 6 + m
            st['fitpars_i'] = SHARED + ['pad'] * m + ['Inst_R']
        out.append(st)
    return out


def draw(K, B, seed, lsf=False):
    rng = np.random.default_rng(seed)
    box = synth._BOX
    cols = SHARED_LSF + ['Vrad'] * K if lsf else SHARED + ['Inst_R'] * K
    th = np.empty((B, len(cols)))
    for i, p in enumerate(cols):
        th[:, i] = box[p][0] + (box[p][1] - box[p][0]) * rng.random(B)
    return th


def timed(fn, reps):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in ev]))


def kernels(eng, fn, reps):
    eng.set('timing', 1)
    rows = []
    for _ in range(reps):
        fn()
        torch.cuda.synchronize()
        rows.append([max(0.0, eng.last_ms(w)) for w in ('mlp', 'tail')])
    eng.set('timing', 0)
    return [float(v) for v in np.median(np.array(rows), axis=0)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--ks', default='1,2,4,8')
    ap.add_argument('--bs', default='512,4096')
    ap.add_argument('--reps', type=int, default=30)
    ap.add_argument('--lsf', action='store_true', help='members with their own LSF vectors and Vrad columns')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('gpu_targets.py needs a CUDA device')
    wave, rsig = synth.ann_wavegrid(5130.0, 5340.0, 50000.0)              # C2 (synth.config_c2)
    spec = synth.make_specnet(4, 256, wave, rsig, seed=0)
    info = gpu_info()
    print('gpu:', json.dumps(info))
    rows = []
    for K in [int(v) for v in args.ks.split(',')]:
        mem = members(spec, K, args.lsf)
        eng = Engine(spec=spec, stars=mem, targets=[K], precision='parity')
        for B in [int(v) for v in args.bs.split(',')]:
            eng.set('max_batch', max(8192, K * B))           # one slab for either case
            th = torch.from_numpy(draw(K, B, K * 100 + B, args.lsf)).cuda()
            tgt = torch.zeros(B, dtype=torch.int32, device='cuda')
            th_dup = th.repeat_interleave(K, dim=0).contiguous()   # row p*K + m: point p, member m
            star = torch.arange(K, dtype=torch.int32, device='cuda').repeat(B).contiguous()
            out = {}
            f_t = lambda: out.__setitem__('t', eng.lnlike_batch_targets(th, tgt))        # noqa: E731
            f_d = lambda: out.__setitem__('d', eng.lnlike_batch(th_dup, star))            # noqa: E731
            for f in (f_t, f_d, f_t, f_d):
                f()
            torch.cuda.synchronize()
            c2 = (-2.0 * out['d'].cpu().numpy()).reshape(B, K)
            tot = c2[:, 0].copy()
            for m in range(1, K):
                tot = tot + c2[:, m]
            same = bool(np.array_equal(-0.5 * tot, out['t'].cpu().numpy(), equal_nan=True))
            row = {'K': K, 'B': B, 'lsf': args.lsf, 'identical_lnl': same,
                   'targets_ms': timed(f_t, args.reps), 'duplicated_ms': timed(f_d, args.reps),
                   'targets_kernels_ms': kernels(eng, f_t, args.reps),
                   'duplicated_kernels_ms': kernels(eng, f_d, args.reps)}
            row['speedup'] = row['duplicated_ms'] / row['targets_ms']
            rows.append(row)
            print('K=%d B=%5d  targets %.3f ms (emulator %.3f, tail %.3f)  duplicated %.3f ms (emulator %.3f, tail '
                  '%.3f)  x%.2f  identical lnL: %s' % (K, B, row['targets_ms'], *row['targets_kernels_ms'],
                                                       row['duplicated_ms'], *row['duplicated_kernels_ms'],
                                                       row['speedup'], same), flush=True)
        eng.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'targets_lsf.json' if args.lsf else 'targets.json'), 'w') as f:
            json.dump({'gpu': info, 'rows': rows}, f, indent=1)
    if not all(r['identical_lnl'] for r in rows):
        sys.exit('lnL of the two cases differ')


if __name__ == '__main__':
    main()
