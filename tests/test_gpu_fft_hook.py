"""GPU: the runtime-planned shared-memory FFT convolution of the fused tails (csrc/fft.cuh: FftPlan, strided_pass<1..4>,
contiguous16, filter_pairs) alone, through the payne_fft_test hook, against irfft(rfft(x) * H) in float64.

Every transform size the tails can plan at run time is checked (N = 2^5 .. 2^15 real samples; plans of one, two and
three strided passes of radix 2, 4, 8 and 16).  Inputs: random normal data, unit impulses at both ends, the Nyquist tone,
a constant and a spectrum of Gaussian absorption lines (line depths, what the tails convolve).  Transfer functions: the
identity, the instrumental Gaussian taper of smoothing.py:604-606 and the rotational kernel sb(u) of smoothing.py:612-619.

Bars, from what B200 measures:
  * rms error / rms(x) <= 5e-8 sqrt(log2 N).  The rounding of a float32 transform pair grows with the number of passes;
    measured 4.3e-8 .. 4.6e-8 sqrt(log2 N) (9.7e-8 at N = 32, 1.42e-7 at 1024, 1.78e-7 at 32768, worst case random
    normal data with H = 1), so a flat 1.5e-7 would fail every N >= 2048 with correct code;
  * max error <= 1e-6 max|x| (measured at most 1.8e-7 up to N = 1024);
  * with H = 1 the amplitude bias sum((y - x) x) / sum(x^2) of DESIGN §3.3 (hi+lo radix constants, modulus-optimised
    twiddles) within 1e-8 (measured -5e-10 .. 5.2e-9), pooled over enough random vectors per size (8192 .. 1048576
    samples) that its noise is about 1e-9.
"""
import numpy as np
import pytest
from scipy.special import j1

pytestmark = pytest.mark.gpu

SIZES = list(range(5, 16))


def _fft_conv(x, H):
    from thepayne_b200 import _lib
    lib = _lib.load()
    x = np.ascontiguousarray(x, dtype=np.float32)
    H = np.ascontiguousarray(H, dtype=np.float32)
    y = np.empty_like(x)
    _lib.check(lib.payne_fft_test(x.ctypes.data, int(np.log2(len(x))), H.ctypes.data, 0, y.ctypes.data))
    return y


def _reference(x, H):
    x = np.asarray(x, dtype=np.float32).astype(np.float64)
    H = np.asarray(H, dtype=np.float32).astype(np.float64)
    return np.fft.irfft(np.fft.rfft(x) * H, n=len(x))


def _inputs(N):
    n = np.arange(N)
    rng = np.random.default_rng(N)
    lines = np.zeros(N)
    for _ in range(max(2, N // 64)):
        c, w, d = rng.uniform(0, N), rng.uniform(0.7, 6.0), rng.uniform(0.05, 0.8)
        lines -= d * np.exp(-0.5 * ((n - c) / w) ** 2)
    imp0, imp1 = np.zeros(N), np.zeros(N)
    imp0[0], imp1[-1] = 1.0, 1.0
    return {'normal': rng.standard_normal(N), 'impulse0': imp0, 'impulseN-1': imp1, 'nyquist': (-1.0) ** n,
            'constant': np.full(N, 0.73), 'lines': lines}


def _transfers(N):
    f = np.arange(N // 2 + 1) / N                     # cycles per sample
    out = {'one': np.ones(N // 2 + 1)}
    for s in (0.6, 2.5, 9.0):                          # Gaussian sigma in samples (smoothing.py:604-606)
        out['gauss%.1f' % s] = np.exp(-2.0 * np.pi ** 2 * s ** 2 * f ** 2)
    for s in (1.5, 12.0):                              # vsini in samples (smoothing.py:612-619, as the oracle)
        ss = f.copy()
        ss[0] = 0.01
        u = 2.0 * np.pi * s * ss
        sb = j1(u) / u - 3 * np.cos(u) / (2 * u ** 2) + 3.0 * np.sin(u) / (2 * u ** 3)
        sb[0] = 1.0
        out['rot%.1f' % s] = sb
    return out


def test_fft_hook_rejects_sizes_it_does_not_plan():
    from thepayne_b200 import _lib
    lib = _lib.load()
    buf = np.zeros(1 << 16, dtype=np.float32)
    for l2 in (4, 16):
        assert lib.payne_fft_test(buf.ctypes.data, l2, buf.ctypes.data, 0, buf.ctypes.data) == -1


@pytest.mark.parametrize('log2N', SIZES)
def test_fft_convolution_against_float64(log2N):
    N = 1 << log2N
    worst_rms = worst_max = 0.0
    for xname, x in _inputs(N).items():
        for hname, H in _transfers(N).items():
            y = _fft_conv(x, H).astype(np.float64)
            ref = _reference(x, H)
            xs = np.asarray(x, dtype=np.float32).astype(np.float64)
            rms_x, max_x = np.sqrt(np.mean(xs ** 2)), np.max(np.abs(xs))
            err = y - ref
            rms, mx = np.sqrt(np.mean(err ** 2)) / rms_x, np.max(np.abs(err)) / max_x
            worst_rms, worst_max = max(worst_rms, rms), max(worst_max, mx)
            assert rms <= 5e-8 * np.sqrt(log2N), (xname, hname, rms)
            assert mx <= 1e-6, (xname, hname, mx)
    print('fft log2N=%d: rms err / rms(x) %.2e, max err / max|x| %.2e' % (log2N, worst_rms, worst_max))


@pytest.mark.parametrize('log2N', SIZES)
def test_fft_amplitude_bias(log2N):
    """With H = 1 the convolution is the identity: sum((y - x) x) / sum(x^2) measures a coherent gain error."""
    N = 1 << log2N
    calls = min(256, max(4, (1 << 20) >> log2N))
    rng = np.random.default_rng(1000 + log2N)
    H = np.ones(N // 2 + 1)
    num = den = 0.0
    for _ in range(calls):
        x = rng.standard_normal(N).astype(np.float32)
        y = _fft_conv(x, H).astype(np.float64)
        xd = x.astype(np.float64)
        num += np.dot(y - xd, xd)
        den += np.dot(xd, xd)
    bias = num / den
    print('fft log2N=%d: amplitude bias %.2e over %d samples' % (log2N, bias, calls * N))
    assert abs(bias) <= 1e-8, bias
