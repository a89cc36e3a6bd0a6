"""Pure-Python HDF5 reader (SURVEY §8 f2: the reference's network files without h5py)."""
import os

import numpy as np
import pytest

from thepayne_b200 import annio, h5lite, synth


def _sample():
    rng = np.random.default_rng(3)
    return {'xmin': rng.normal(size=4), 'resolution': np.array(32000.0),
            'label_i': np.array([b'teff', b'logg', b'feh', b'afe']),
            'model/lin1.weight': rng.normal(size=(64, 4)).astype(np.float32),
            'model/lin6.weight': rng.normal(size=(1417, 64)).astype(np.float32),     # 23 chunks, ragged last one
            'model/lin6.bias': rng.normal(size=1417).astype(np.float32),
            'a/b/c/ints': np.arange(10, dtype=np.int32), 'u8': np.arange(7, dtype=np.uint8),
            'wavelengths': np.linspace(5000, 5100, 777), 'empty': np.zeros(0)}


@pytest.mark.parametrize('gzip', [(), ('lin',), True])
def test_round_trip(tmp_path, gzip):
    d = _sample()
    p = h5lite.write(str(tmp_path / 't.h5'), d, gzip=gzip)
    r = h5lite.read(p)
    assert sorted(r) == sorted(d)
    for k in d:
        assert r[k].dtype == d[k].dtype and r[k].shape == d[k].shape, k
        assert np.array_equal(r[k], d[k]), k


def test_compressed_is_chunked_and_smaller(tmp_path):
    d = {'model/w': np.zeros((4096, 64), np.float32)}
    a = os.path.getsize(h5lite.write(str(tmp_path / 'a.h5'), d))
    b = os.path.getsize(h5lite.write(str(tmp_path / 'b.h5'), d, gzip=True))
    assert b < a / 5
    assert np.array_equal(h5lite.read(str(tmp_path / 'b.h5'))['model/w'], d['model/w'])


def test_rejects_what_it_cannot_read(tmp_path):
    p = tmp_path / 'x.h5'
    p.write_bytes(b'not hdf5 at all' * 10)
    with pytest.raises(IOError):
        h5lite.read(str(p))
    good = bytearray(open(h5lite.write(str(tmp_path / 'g.h5'), {'a': np.ones(3)}), 'rb').read())
    good[8] = 2                                     # pretend libver='latest'
    p.write_bytes(bytes(good))
    with pytest.raises(IOError, match='superblock version 2'):
        h5lite.read(str(p))


def test_specnet_and_photnet_through_h5(tmp_path):
    """annio falls back to h5lite when h5py is missing: .h5 in the reference's layout -> same networks."""
    net = synth.make_specnet(4, 32, synth.ann_wavegrid(5150.0, 5160.0, 100000.0)[0][:300], 100000.0, seed=5)
    p = str(tmp_path / 'spec.h5')
    annio.save_specnet(p, net)
    back = annio.load_specnet(p)
    assert back.inlabels == net.inlabels and back.resolution == net.resolution
    for a, b in zip(net.weights + net.biases, back.weights + back.biases):
        assert a.dtype == b.dtype and np.array_equal(a, b)
    assert np.array_equal(back.wavelength, net.wavelength) and np.array_equal(back.xmin, net.xmin)
    ph = synth.make_photnet(['2MASS_J', 'GaiaEDR3_G'], H=16, seed=2)
    annio.save_photnet(str(tmp_path / 'phot'), ph, fmt='h5')
    pb = annio.load_photnet(str(tmp_path / 'phot'), ph.bands, hiav=ph.hiav)
    assert np.array_equal(pb.w2, ph.w2) and np.array_equal(pb.xmax, ph.xmax)


def test_multichunk_files_round_trip(tmp_path):
    """The multi-chunk trainer's per-chunk files (train/old/trainspec_multi.py:300-313): written in its
    layout, read back in any order, chunks re-assembled by wavelength."""
    from thepayne_b200 import annio, synth
    wave, rsig = synth.ann_wavegrid(5140.0, 5150.0, 50000.0)
    net = synth.make_multinet(4, 24, wave, rsig, chunk=200, seed=3)
    assert net.n_groups == (len(wave) + 199) // 200 and net.D_out == len(wave) and net.D_in == 4
    paths = annio.save_multinet(str(tmp_path / 'ann'), net)
    assert len(paths) == net.n_groups and all('_w' in p for p in paths)
    d = h5lite.read(paths[1])
    assert sorted(k.split('/')[-1] for k in d if 'model/' in k) == sorted(
        ['lin%d.%s' % (k, w) for k in range(1, 5) for w in ('weight', 'bias')])
    back = annio.load_multinet(list(reversed(paths)), net.xmin, net.xmax, net.resolution)
    assert back.nntype == 'MultiNet' and back.chunk == 200 and back.encode_offset == 0.0
    for a, b in zip(net.weights + net.biases, back.weights + back.biases):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(net.wavelength, back.wavelength)
    assert back.digest() == net.digest()
    back2 = annio.load_multinet(str(tmp_path / 'ann_w*.h5'), net.xmin, net.xmax, net.resolution)
    assert back2.digest() == net.digest()
