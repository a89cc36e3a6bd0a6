"""CPU: host-side logic that does not need the device -- the FFT-convolution index model the
CUDA kernels implement, shard arithmetic, container I/O, the reference-interface mirrors'
parameter plumbing."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))


@pytest.mark.parametrize('N', [512, 2048, 16384, 32768])
def test_fft_convolution_model_matches_numpy(N):
    """tools/fft_model.py mirrors csrc/fft.cuh: in-place DIF -> digit-reversed pair filter -> DIT
    must equal irfft(rfft(x) * H) (smoothing.py:588-629)."""
    import fft_model as fm
    rng = np.random.default_rng(N)
    s = rng.standard_normal(N)
    k = np.arange(N // 2 + 1)
    H = np.exp(-3e-7 * k ** 2) * np.cos(0.003 * k)
    ref = np.fft.irfft(np.fft.rfft(s) * H)
    assert np.abs(fm.conv_real(s, H) - ref).max() < 1e-12


def test_radix_plan_covers_all_bits():
    import fft_model as fm
    for m in range(8, 16):
        plan = fm.radix_plan(m)
        assert sum(plan) == m and plan[-1] == 4 and all(1 <= r <= 4 for r in plan)


def test_shard_bounds_partition():
    from thepayne_b200.dist import shard_bounds
    for B in [0, 1, 7, 4096, 1000003]:
        for world in [1, 2, 3, 8]:
            spans = [shard_bounds(B, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == B
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [h - l for l, h in spans]
            assert max(sizes) - min(sizes) <= 1


def test_ann_container_roundtrip(tmp_path):
    from thepayne_b200 import annio, synth
    w, rs = synth.ann_wavegrid(5140.0, 5150.0, 50000.0)
    net = synth.make_specnet(4, 16, w, rs)
    p = str(tmp_path / 'ann.npz')
    annio.save_specnet(p, net)
    back = annio.load_specnet(p)
    assert back.digest() == net.digest() and back.inlabels == net.inlabels
    assert back.resolution == net.resolution and np.array_equal(back.xmin, net.xmin)
    ph = synth.make_photnet(synth.PROCYON_BANDS[:3], H=8)
    annio.save_photnet(str(tmp_path / 'phot'), ph)
    pb = annio.load_photnet(str(tmp_path / 'phot'), ph.bands, hiav=ph.hiav)
    assert np.array_equal(pb.w2, ph.w2) and np.array_equal(pb.b3, ph.b3)


def test_wavegrid_is_the_trainer_grid():
    """readc3k.py:441-451: w0*(1+1/(3 R))**i while <= w1."""
    from thepayne_b200 import synth
    w, rs = synth.ann_wavegrid(5130.0, 5340.0, 50000.0)
    assert len(w) == 14172 and abs(rs - 50000 * 2.35482) < 1e-9
    ref, i = [], 1
    while True:
        x = 5130.0 * (1.0 + 1.0 / (3.0 * rs)) ** (i - 1.0)
        if x > 5340.0:
            break
        ref.append(x)
        i += 1
    assert np.array_equal(w, np.array(ref))


def test_free_parameters_and_highav():
    from thepayne_b200.fitting.likelihood import free_parameters
    from thepayne_b200.predict.highred import highAv
    names = ['Teff', 'log(g)', 'Vrad', 'pc_0']
    flags = {'Teff': True, 'log(g)': False, 'Vrad': True, 'pc_0': True}
    assert free_parameters([names, flags]) == ['Teff', 'Vrad', 'pc_0']
    h = highAv(['2MASS_J', 'Nope'])
    assert np.isnan(h.Avlist[1]).all() and np.isfinite(h.Avlist[0]).all()
    bc = h.calc(np.array([1.0, 1.0]), 6.0, 3.1)
    a1, b1, a2, b2, c2 = h.Avlist[0]
    assert bc[0] == 1.0 - (a1 + b1 * 6.0 * (a2 + b2 * 3.1 + c2 * 3.1 ** 2.0)) and np.isnan(bc[1])


def test_polycalc_is_chebval_on_normalised_grid():
    from thepayne_b200.fitting.fitutils import polycalc
    from oracle import payne_oracle as O
    w = np.linspace(5150, 5320, 50)
    c = np.array([1.0, 0.02, -0.01])
    assert np.array_equal(polycalc(c, w), O.polycalc(c, w))


def test_legacy_network_containers_round_trip(tmp_path):
    """SMLP (model/features.*) and YST1 (w_array_* / x_min / wavelength) layouts of the reference's
    files (NNmodels.py:51-63, ystpred.py:25-37) through both containers; the type is inferred from the
    dataset names when not given."""
    from thepayne_b200 import annio, synth
    w = synth.ann_wavegrid(5150.0, 5160.0, 1e5)[0][:300]
    for nntype, H, nl in [('LinNet', 32, 6), ('SMLP', 24, 4), ('YST1', 16, 3)]:
        net = synth.make_specnet(4, H, w, 1e5, seed=1, nntype=nntype)
        assert net.n_layers == nl and net.activation == ('sigmoid' if nl == 6 else 'leaky')
        for ext in ['npz', 'h5']:
            p = str(tmp_path / ('%s.%s' % (nntype, ext)))
            annio.save_specnet(p, net)
            back = annio.load_specnet(p)
            assert back.nntype == nntype and back.n_layers == nl and back.resolution == net.resolution
            assert all(np.array_equal(a, b) for a, b in zip(net.weights + net.biases, back.weights + back.biases))
            assert np.array_equal(back.wavelength, net.wavelength) and np.array_equal(back.xmax, net.xmax)
            assert annio.load_specnet(p, NNtype=nntype).D_out == net.D_out


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float64 .npy files; an output over the size cap becomes the same seeded sample on every
    run, so that two builds compare the same positions."""
    import bench
    a = np.linspace(-5.0, 5.0, 100, dtype=np.float32)
    bench.dump_outputs(str(tmp_path / 'a'), {'lnl': a[:10]})
    got = np.load(tmp_path / 'a' / 'lnl.npy')
    assert got.dtype == np.float64 and np.array_equal(got, a[:10])
    monkeypatch.setattr(bench, 'DUMP_MAX_BYTES', 8 * 64)
    for d in 'bc':
        bench.dump_outputs(str(tmp_path / d), {'lnl': a, 'flux': a})
    b = [np.load(tmp_path / 'b' / n) for n in ('lnl.npy', 'flux.npy')]
    assert all(x.size == 32 for x in b) and np.all(np.diff(b[0]) > 0) and np.isin(b[0], a).all()
    assert np.array_equal(b[0], np.load(tmp_path / 'c' / 'lnl.npy'))
