"""Every emulator shape path against a float64 evaluation of the same network.

The emulator's kernels are chosen by shape (run_mlp in payne_b200.cu, tc_run_layers_mode / tc_run_multinet_mode /
tc_run_scaled_layer in mlp_tc.cuh):

  * LinNet, parity: lin2..lin5 as one cluster launch of H/64 CTAs (mlp_stack.cuh) when every hidden layer is H -> H with
    H in {64, 128, 256, 512}; one tensor-core launch per layer otherwise (H below 64, off the powers of two, or layers of
    different widths); refused above 512.  simt: CUDA-core layers.  3xtf32 / tf32: per-layer tensor-core launches.
  * multi-chunk (G nets of `chunk` pixels), parity: grouped GEMMs for lin2, lin3 and, when the chunk is a multiple of 32
    pixels (or G = 1), lin4; one lin4 launch per chunk otherwise; refused when the chunk is not a multiple of 4.
  * SMLP / YST1, parity: CUDA-core hidden layers and the output layer on the tensor cores with row-scaled slices when its
    contraction K satisfies 8 <= K <= 512, CUDA cores otherwise.

CONFIGS is that matrix as plain data; every row names the parity path it is meant for.  `test_table_covers_every_path`
(no GPU) rebuilds each row's network, recomputes the path from its weights and asserts the union still reaches every
branch, every hidden width, label count, output width, batch edge and chunk layout listed below, so a change of the
synthetic defaults cannot silently empty one.

The GPU test evaluates every row with `ann_eval` at B = 1, 127, 128, 129 and 300 and compares with the oracle's network
in float64 (`make_net(spec, ideal=True)`) and in float32 (`make_net(spec)`; YST1's reference is float64 numpy, so its
float32 yardstick is the same stack in torch float32):
  parity: max relative error <= 5e-7; rms distance from float64 over all of a row's evaluations <= 1.25 x the float32
          network's own; |mean signed relative error| <= 2e-9, or 4 standard errors on narrow nets (see Errors);
  simt: <= 1e-6;  3xtf32: <= 3e-6;  tf32: <= 5e-4.
`query('launches')` around each call pins the path that ran.  For rows with at most five labels the likelihood path runs
too: `model_batch` with Vrot = 0, Vrad = 0 and no Inst_R on observed pixels that are interior emulator pixels, so the
model spectrum is the emulator row at those pixels (line-depth emission with the bias shifted by -1, the flux slab with
its padded pitch, the output map sized to the workspace rows).  Labels 6 to 8 have no likelihood parameter
(payne_b200.cu leaves them NaN): there the library returns NaN spectra and NaN lnL without a status bit, which the test
pins.

Also here: PDL off (PAYNE_GEMM_PDL=0), read once per process, runs in a subprocess and must match the default bit for
bit; and the tensor-map caches across a workspace that grows between two calls.
"""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import payne_oracle as O  # noqa: E402
from thepayne_b200 import synth  # noqa: E402

W0 = 5000.0
R_FWHM = 50000.0
BATCHES = [1, 127, 128, 129, 300]
BARS = {'parity': 5e-7, 'simt': 1e-6, '3xtf32': 3e-6, 'tf32': 5e-4}
RMS_FACTOR = 1.25
MEAN_BAR = 2e-9
PS = ['parity', 'simt']
TF = ['parity', 'simt', '3xtf32', 'tf32']


def _lin(name, H, D_in, D_out, path, precs=PS, **kw):
    H = (H, H, H) if isinstance(H, int) else H
    return dict(name=name, kind='LinNet', H=H, D_in=D_in, D_out=D_out, path=path, precs=precs, **kw)


# kind, hidden widths (H1, H2, H3; SMLP uses all three, YST1 two), labels, pixels, intended parity path
CONFIGS = [
    _lin('lin_h8', 8, 4, 33, 'layers'),
    _lin('lin_h16', 16, 1, 127, 'layers'),
    _lin('lin_h40', 40, 2, 32, 'layers', TF),
    _lin('lin_h64', 64, 3, 129, 'stack1', TF),
    _lin('lin_h100', 100, 5, 100, 'layers', TF),
    _lin('lin_h128', 128, 6, 255, 'stack2'),
    _lin('lin_h192', 192, 7, 128, 'layers'),
    _lin('lin_h256', 256, 8, 257, 'stack4'),
    _lin('lin_h320', 320, 4, 131, 'layers'),
    _lin('lin_h512', 512, 5, 4097, 'stack8'),
    _lin('lin_64_128_256', (64, 128, 256), 4, 257, 'layers', TF),
    _lin('lin_256_100_512', (256, 100, 512), 4, 129, 'layers'),
    _lin('lin_h520', 520, 4, 64, 'refused'),
    _lin('lin_slab200', 64, 4, 130, 'stack1', max_batch=200),
    _lin('lin_large', 256, 4, 4097, 'stack4', batches=[4096]),
]
# multi-chunk: G = ceil(D_out / chunk); the last chunk is D_out - (G - 1) chunk pixels wide
for _n, _H, _c, _D in [('multi_g1', 16, 100, 100),          # G = 1 (grouped launch of one chunk, any width)
                       ('multi_c32_g2', 40, 32, 33),        # last chunk 1 pixel: narrower by chunk - 1
                       ('multi_c64_g13', 64, 64, 831),      # last chunk narrower by 1
                       ('multi_c96_g64', 16, 96, 6068),     # G = 64, last chunk 20 pixels (< 32)
                       ('multi_c36', 128, 36, 179),         # one launch per chunk, last narrower by 1
                       ('multi_c100', 64, 100, 250),        # last chunk 50 pixels
                       ('multi_c500', 512, 500, 1001),      # last chunk 1 pixel
                       ('multi_c33', 40, 33, 99),           # chunk % 4 != 0: simt only
                       ('multi_c50', 16, 50, 120)]:
    CONFIGS.append(dict(name=_n, kind='MultiNet', H=(_H, _H, _H), D_in=4 if _H != 64 else 5, D_out=_D, chunk=_c,
                        path=('multi-grouped' if _c % 32 == 0 or _c >= _D else
                              'refused' if _c % 4 else 'multi-per-chunk'), precs=PS))
CONFIGS += [
    dict(name='smlp_k4', kind='SMLP', H=(16, 16, 4), D_in=4, D_out=129, path='legacy-cuda', precs=PS),
    dict(name='smlp_k48', kind='SMLP', H=(64, 64, 48), D_in=4, D_out=200, path='legacy-tc', precs=PS),
    dict(name='smlp_k512', kind='SMLP', H=(128, 128, 512), D_in=5, D_out=257, path='legacy-tc', precs=PS),
    dict(name='yst_k8', kind='YST1', H=(32, 8, 8), D_in=4, D_out=33, path='legacy-tc', precs=PS),
    dict(name='yst_k100', kind='YST1', H=(64, 100, 100), D_in=4, D_out=300, path='legacy-tc', precs=PS),
    dict(name='yst_k600', kind='YST1', H=(64, 600, 600), D_in=4, D_out=129, path='legacy-cuda', precs=PS),
    # the output layer's activations span 1e-3 .. 1e3 within every row: the row scale of x3_split_rows_kernel
    dict(name='yst_scaled', kind='YST1', H=(64, 256, 256), D_in=4, D_out=131, path='legacy-tc', precs=PS,
         scaled=True),
]
BY_NAME = {c['name']: c for c in CONFIGS}
LABELS = ['teff', 'logg', 'feh', 'afe', 'vmic', 'x5', 'x6', 'x7']
XMIN = np.array([3500.0, 0.0, -2.5, -0.2, 0.5, -1.0, 0.0, 10.0])
XMAX = np.array([8000.0, 5.5, 0.5, 0.6, 3.0, 1.0, 2.0, 20.0])


def wave_grid(n):
    """Log-uniform emulator grid of exactly n pixels (ann_wavegrid's own recurrence ends on the last one)."""
    rsig = R_FWHM * synth.SIGMA_TO_FWHM_TRAIN
    w, _ = synth.ann_wavegrid(W0, W0 * (1.0 + 1.0 / (3.0 * rsig)) ** (n - 1.0), R_FWHM)
    assert len(w) == n
    return w


_built = {}


def build(name):
    """The row's SpecNet (deterministic, cached)."""
    if name in _built:
        return _built[name]
    c = BY_NAME[name]
    w = wave_grid(c['D_out'])
    rsig = R_FWHM * synth.SIGMA_TO_FWHM_TRAIN
    H1, H2, H3 = c['H']
    seed = CONFIGS.index(c) + 11
    if c['kind'] == 'MultiNet':
        spec = synth.make_multinet(c['D_in'], H1, w, rsig, c['chunk'], seed=seed)
    else:
        spec = synth.make_specnet(c['D_in'], H1, w, rsig, seed=seed, H2=H2, H3=H3, nntype=c['kind'])
    # labels beyond the five synth knows: the struct reads D_in bounds
    spec.xmin, spec.xmax, spec.inlabels = XMIN[:c['D_in']].copy(), XMAX[:c['D_in']].copy(), LABELS[:c['D_in']]
    if c.get('scaled'):
        rng = np.random.default_rng(5)
        s = 10.0 ** rng.permutation(np.linspace(-3.0, 3.0, spec.weights[1].shape[0]))
        spec.weights[1] = (spec.weights[1] * s[:, None]).astype(np.float32)     # leaky ReLU is positively homogeneous
        spec.biases[1] = (spec.biases[1] * s).astype(np.float32)
        spec.weights[2] = (spec.weights[2] * 1e-3).astype(np.float32)           # keeps the flux near 1
    _built[name] = spec
    return spec


def route(spec, prec):
    """(path, launches per ann_eval slab) run_mlp takes for this network and precision."""
    W = spec.weights
    if spec.nntype == 'MultiNet':
        G, P, H = spec.n_groups, spec.chunk, W[1].shape[-1]
        if prec == 'simt':
            return 'multi-simt', 4 * G
        if P % 4 or H > 512 or prec != 'parity':
            return 'refused', None
        return ('multi-grouped', 4) if (P % 32 == 0 or G == 1) else ('multi-per-chunk', 3 + G)
    if spec.nntype in ('SMLP', 'YST1'):
        K, nl = W[-1].shape[1], len(W)
        if prec == 'parity' and 8 <= K <= 512:
            return 'legacy-tc', nl + 1          # encode, hidden layers, row split + GEMM
        return ('legacy-cuda' if prec == 'parity' else 'legacy-simt'), nl
    din = [w.shape[1] for w in W]
    dout = [w.shape[0] for w in W]
    if prec == 'simt':
        return 'simt', 6
    if prec == 'parity' and max(din[1:]) > 512:
        return 'refused', None
    if prec != 'parity':
        return prec + '-layers', 7             # encode, operand split, five GEMMs
    H = din[1]
    if all(din[k] == H and dout[k] == H for k in range(1, 5)) and H in (64, 128, 256, 512):
        return 'stack%d' % (H // 64), 3        # encode + slicing, the stack, lin6
    return 'layers', 6


def labels(spec, B, seed):
    rng = np.random.default_rng(seed)
    return spec.xmin + (spec.xmax - spec.xmin) * rng.uniform(0.02, 0.98, (B, spec.D_in))


# ------------------------------------------------------------------ CPU: the table reaches every path
def test_table_covers_every_path():
    seen = set()
    lin_h, lin_din, lin_dout, layer_h = set(), set(), set(), set()
    multi_g, last_short = set(), set()
    legacy_k = set()
    for c in CONFIGS:
        spec = build(c['name'])
        assert spec.D_in == c['D_in'] and spec.D_out == c['D_out'] and spec.nntype == c['kind'], c['name']
        got = route(spec, 'parity')[0]
        assert got == c['path'], (c['name'], got)
        for p in c['precs']:
            seen.add(route(spec, p)[0])
        if c['kind'] == 'LinNet':
            hs = tuple(w.shape[0] for w in spec.weights[1:5])
            lin_h.add(hs[0]) if len(set(hs)) == 1 else lin_h.add(hs)
            lin_din.add(spec.D_in)
            lin_dout.add(spec.D_out)
            if got == 'layers':
                layer_h.add(hs)
        elif c['kind'] == 'MultiNet':
            G, P = spec.n_groups, spec.chunk
            multi_g.add(G)
            last = spec.D_out - (G - 1) * P
            assert spec.weights[0].shape[0] == G and spec.weights[3].shape[0] == spec.D_out
            if G > 1:
                last_short.update(k for k, ok in [('by1', last == P - 1), ('to1', last == 1), ('lt32', last < 32)] if ok)
        else:
            legacy_k.add(spec.weights[-1].shape[1])
    assert seen >= {'stack1', 'stack2', 'stack4', 'stack8', 'layers', 'refused', 'simt', '3xtf32-layers',
                    'tf32-layers', 'multi-grouped', 'multi-per-chunk', 'multi-simt', 'legacy-tc', 'legacy-cuda',
                    'legacy-simt'}, seen
    assert {8, 16, 40, 64, 100, 128, 192, 256, 320, 512} <= lin_h and (64, 128, 128, 256) in lin_h
    assert (256, 100, 100, 512) in lin_h
    assert any(h[0] < 64 for h in layer_h) and {(192,) * 4, (320,) * 4} <= layer_h
    assert lin_din == set(range(1, 9))
    assert {32, 33, 100, 127, 128, 129, 255, 257, 4097} <= lin_dout and any(d % 4 for d in lin_dout)
    assert {1, 2, 13, 64} <= multi_g and last_short == {'by1', 'to1', 'lt32'}
    chunks = {c['chunk']: c['path'] for c in CONFIGS if c['kind'] == 'MultiNet'}
    assert all(chunks[k] == 'multi-grouped' for k in (32, 64, 96))
    assert all(chunks[k] == 'multi-per-chunk' for k in (36, 100, 500))
    assert all(chunks[k] == 'refused' for k in (33, 50))
    assert {c['H'][0] for c in CONFIGS if c['kind'] == 'MultiNet'} >= {16, 40, 64, 128, 512}
    assert legacy_k >= {4, 8, 48, 100, 512, 600} and any(c.get('scaled') for c in CONFIGS)
    assert {'SMLP', 'YST1'} <= {c['kind'] for c in CONFIGS if c['path'].startswith('legacy')}
    # the scaled row's output-layer activations do span 1e-3 .. 1e3 within a row
    spec = build('yst_scaled')
    x = labels(spec, 4, 0)
    h = (x - spec.xmin) / (spec.xmax - spec.xmin) - 0.5
    for k in range(2):
        z = h @ spec.weights[k].T.astype(np.float64) + spec.biases[k]
        h = np.where(z > 0, z, 0.01 * z)
    h = np.abs(h)
    assert np.all(h.max(1) > 1e2) and np.all(np.median(h, 1) < 1.0) and np.all(h.min(1) < 1e-3)
    # batches: the tile edges, a slab that is not a multiple of 128, and lin6 with more than 1000 output tiles
    assert set(BATCHES) == {1, 127, 128, 129, 300}
    c = BY_NAME['lin_slab200']
    assert c['max_batch'] % 128 and max(BATCHES) > c['max_batch']
    c = BY_NAME['lin_large']
    assert c['D_out'] >= 4097 and math.ceil(c['batches'][0] / 128) * math.ceil(c['D_out'] / 128) > 1000


# ------------------------------------------------------------------ GPU helpers
class Fp32Yst:
    """YST1 (float64 numpy in the reference) evaluated in torch float32: the yardstick for the rms bar."""

    def __init__(self, spec):
        self.spec = spec

    def __call__(self, x):
        sp = self.spec
        h = torch.from_numpy((np.asarray(x) - sp.xmin) / (sp.xmax - sp.xmin) - 0.5).float()
        lin = torch.nn.functional.linear
        for k in range(2):
            h = torch.nn.functional.leaky_relu(lin(h, torch.from_numpy(sp.weights[k]), torch.from_numpy(sp.biases[k])))
        return lin(h, torch.from_numpy(sp.weights[2]), torch.from_numpy(sp.biases[2])).numpy()


def fp32_net(spec):
    return Fp32Yst(spec) if spec.nntype == 'YST1' else O.make_net(spec)


def fitpars(spec):
    lab = ['Teff', 'log(g)', '[Fe/H]', '[a/Fe]'] + (['Vmic'] if spec.D_in >= 5 else [])
    return lab + ['Vrad', 'Vrot']


def obs_index(spec):
    n = spec.D_out
    return np.unique(np.linspace(2, n - 3, min(n - 4, 2000)).astype(int))


def engine(spec, prec):
    from thepayne_b200.engine import Engine
    ix = obs_index(spec)
    one = np.ones(len(ix))
    return Engine(spec=spec, obs_wave=spec.wavelength[ix], obs_flux=one, obs_eflux=0.01 * one,
                  fitpars_i=fitpars(spec), runbools=(True, False, False, False, False), precision=prec)


class Errors:
    """Relative errors of one row against float64, and the float32 network's own.

    The mean signed error is taken over the largest batch (the smaller ones repeat its first points).  A point's
    outputs share its rounded hidden activations, and a pixel's output weights are the same for every point, so the
    errors are correlated along both axes and a narrow net's mean is a mean over few independent values:
    multi_c32_g2 (29 observed pixels, H = 40, 300 points) measured +2.3e-9 on the model path at an rms of 1.1e-8, with
    a standard error of 8.7e-11 between points but the same sign at every point.  The bar is therefore
    max(2e-9, 4 standard errors of the mean), the standard error taken as the larger of the spread of the per-point
    and of the per-pixel means; on the wide rows 2e-9 is what decides.
    """

    def __init__(self):
        self.d, self.d32, self.worst, self.last = [], [], 0.0, None

    def add(self, y, ref64, ref32):
        y = np.asarray(y, dtype=np.float64)
        assert np.all(np.isfinite(y))
        rel = (y - ref64) / np.abs(ref64)
        self.worst = max(self.worst, float(np.abs(rel).max()))
        self.d.append((y - ref64).ravel())
        self.d32.append((np.asarray(ref32, dtype=np.float64) - ref64).ravel())
        self.last = rel

    def check(self, prec, what):
        d, d32 = np.concatenate(self.d), np.concatenate(self.d32)
        rms, rms32 = np.sqrt(np.mean(d ** 2)), np.sqrt(np.mean(d32 ** 2))
        mean = float(self.last.mean())
        sem = 0.0
        for ax in (1, 0):          # per-point means, then per-pixel means: the larger standard error counts
            m = self.last.mean(axis=ax)
            sem = max(sem, float(m.std() / np.sqrt(len(m))) if len(m) > 1 else float('inf'))
        print('  %-7s %-10s max rel %.2e  rms %.2e (fp32 net %.2e, ratio %.2f)  mean rel %+.1e (s.e. %.1e)'
              % (prec, what, self.worst, rms, rms32, rms / rms32 if rms32 else float('nan'), mean, sem))
        assert self.worst <= BARS[prec], (prec, what, self.worst)
        if prec == 'parity':
            assert rms <= RMS_FACTOR * rms32, (what, rms, rms32)
            assert abs(mean) <= max(MEAN_BAR, 4.0 * sem), (what, mean, sem)


def _refuses(spec, prec):
    from thepayne_b200 import _lib
    with pytest.raises(_lib.PayneError) as e:
        engine(spec, prec)
    return str(e.value)


# ------------------------------------------------------------------ GPU: every row
@pytest.mark.gpu
@pytest.mark.parametrize('name', [c['name'] for c in CONFIGS])
def test_emulator_shape(name):
    c = BY_NAME[name]
    spec = build(name)
    batches = c.get('batches', BATCHES)
    x = labels(spec, max(batches), seed=len(name))
    ref64 = O.make_net(spec, ideal=True)(x)
    ref32 = fp32_net(spec)(x)
    ix = obs_index(spec)
    Bm = min(max(batches), 300)
    th = np.zeros((Bm, len(fitpars(spec))))
    th[:, :min(spec.D_in, 5)] = x[:Bm, :5]
    print(name)
    for prec in c['precs']:
        path, per_slab = route(spec, prec)
        if path == 'refused':
            msg = _refuses(spec, prec)
            assert ('hidden widths up to 512' in msg) if spec.nntype == 'LinNet' else ('multiple of 4' in msg), msg
            continue
        eng = engine(spec, prec)
        if 'max_batch' in c:
            eng.set('max_batch', c['max_batch'])
        slab = eng.query('max_batch')
        assert eng.query('gemm_stack') == 1 and eng.query('precision') == _prec_id(prec)
        assert eng.query('legacy_tc') == (1 if path == 'legacy-tc' else 0)
        err = Errors()
        for B in batches:
            l0 = eng.query('launches')
            y = eng.ann_eval(torch.from_numpy(x[:B]).cuda()).cpu().numpy()
            assert eng.query('launches') - l0 == per_slab * math.ceil(B / slab), (prec, B, path)
            err.add(y, ref64[:B], ref32[:B])
        err.check(prec, 'ann_eval')
        # the likelihood path: model spectrum = emulator row at interior emulator pixels
        flux, _, lnl = eng.model_batch(torch.from_numpy(th).cuda())
        f, lnl = flux.cpu().numpy(), lnl.cpu().numpy()
        if spec.D_in > 5:
            assert np.all(np.isnan(f)) and np.all(np.isnan(lnl))
        else:
            e2 = Errors()
            e2.add(f, ref64[:Bm, ix].astype(np.float64), ref32[:Bm, ix])
            e2.check(prec, 'model')
            assert np.all(np.isfinite(lnl))
        assert eng.query('status') == 0
        eng.close()


def _prec_id(prec):
    from thepayne_b200._lib import PREC
    return PREC[prec]


# ------------------------------------------------------------------ env-selected variants, in a subprocess
VARIANT_ROWS = [('lin_large', 4096), ('multi_c36', 300), ('multi_c64_g13', 300), ('yst_k100', 300)]


def variant_outputs():
    """Outputs the environment variants must reproduce: lin6 with > 1000 tiles, the per-chunk and grouped multi-chunk
    launches, a legacy row and the GEMM hook at M > 128."""
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_gpu_gemm import gemm, random_inputs
    out = {}
    for name, B in VARIANT_ROWS:
        spec = build(name)
        eng = engine(spec, 'parity')
        x = torch.from_numpy(labels(spec, B, seed=1)).cuda()
        out[name] = eng.ann_eval(x).cpu().numpy()
        th = torch.zeros((min(B, 300), len(fitpars(spec))), dtype=torch.float64, device='cuda')
        th[:, :min(spec.D_in, 5)] = x[:min(B, 300), :5]
        out[name + '_model'] = eng.model_batch(th)[0].cpu().numpy()
        eng.close()
    for M, N, K in [(300, 260, 256), (2560, 4096, 512)]:
        out['gemm_%d' % M] = gemm(*random_inputs(M, N, K, seed=3), 'parity')
    return out


def _run_variant(tmp_path, env_key, env_val):
    path = str(tmp_path / ('%s.npz' % env_key))
    env = dict(os.environ)
    env[env_key] = env_val
    cmd = [sys.executable] + (['-s'] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), path]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return dict(np.load(path))


@pytest.mark.gpu
@pytest.mark.parametrize('env_key,env_val', [('PAYNE_GEMM_PDL', '0')])
def test_env_variants_are_bit_identical(tmp_path, env_key, env_val):
    """Same MMAs in the same K order: launching without PDL changes no bit."""
    got = _run_variant(tmp_path, env_key, env_val)
    ref = variant_outputs()
    assert sorted(got) == sorted(ref)
    for k in ref:
        assert np.array_equal(got[k], ref[k], equal_nan=True), (env_key, k, np.nanmax(np.abs(got[k] - ref[k])))


# ------------------------------------------------------------------ tensor-map caches across workspace growth
def _ann_eval_into(eng, x, y):
    from thepayne_b200 import _lib
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(eng.lib.payne_ann_eval(eng._ctx, x.data_ptr(), x.shape[0], y.data_ptr(), y.shape[1], st))
    torch.cuda.synchronize()
    return y[:x.shape[0], :eng.D_out].cpu().numpy().copy()


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['lin_h64', 'lin_h100'])
def test_map_caches_survive_workspace_growth(name):
    """One engine, one output buffer: ann_eval(100), a 9000-point likelihood call that grows the workspace past the
    8192-row slab (every activation plane is freed and reallocated), ann_eval(100) again, then the stack and the
    precision toggled back and forth.  Every result must be the bits a fresh engine gives."""
    spec = build(name)
    x = torch.from_numpy(labels(spec, 100, seed=2)).cuda()
    th_np = np.zeros((9000, len(fitpars(spec))))
    th_np[:, :spec.D_in] = labels(spec, 9000, seed=4)
    th = torch.from_numpy(th_np).cuda()
    ldy = (spec.D_out + 3) // 4 * 4

    def fresh(prec, stack=1):
        e = engine(spec, prec)
        e.set('gemm_stack', stack)
        y = torch.empty((100, ldy), dtype=torch.float32, device='cuda')
        r = _ann_eval_into(e, x, y)
        e.close()
        return r

    want = {p: fresh(p) for p in ('parity', 'simt', '3xtf32')}
    assert np.array_equal(fresh('parity', 0), want['parity'])
    e = engine(spec, 'parity')
    lnl_want = e.lnlike_batch(th).cpu().numpy()
    e.close()

    eng = engine(spec, 'parity')
    y = torch.empty((100, ldy), dtype=torch.float32, device='cuda')
    assert np.array_equal(_ann_eval_into(eng, x, y), want['parity'])
    lnl = eng.lnlike_batch(th).cpu().numpy()
    assert np.array_equal(lnl, lnl_want)
    assert np.array_equal(_ann_eval_into(eng, x, y), want['parity'])
    for stack in (0, 1, 0, 1):
        eng.set('gemm_stack', stack)
        assert np.array_equal(_ann_eval_into(eng, x, y), want['parity']), stack
    for prec in ('simt', 'parity', '3xtf32', 'parity'):
        eng.set('precision', prec)
        assert np.array_equal(_ann_eval_into(eng, x, y), want[prec]), prec
    assert np.array_equal(eng.lnlike_batch(th).cpu().numpy(), lnl_want)
    assert np.array_equal(_ann_eval_into(eng, x, y), want['parity'])
    assert eng.query('status') == 0
    eng.close()


if __name__ == '__main__':
    # subprocess of test_env_variants_are_bit_identical: the variants read their environment once per process
    np.savez(sys.argv[1], **variant_outputs())
