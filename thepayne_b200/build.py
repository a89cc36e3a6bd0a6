"""Build libpayne_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

The library is six translation units compiled in parallel (csrc/launchers.h says which kernel family
lives where); objects go to csrc/_build/ (git-ignored) and only the ones whose sources changed are redone.
"""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
OBJ = os.path.join(CSRC, '_build')
OUT = os.path.join(HERE, 'libpayne_b200.so')
HDR = os.path.join(os.path.dirname(HERE), 'include', 'payne_b200.h')

_GEMM = ['mlp_tc.cuh', 'mlp_simt.cuh', 'obs_star.cuh']
_FFT = ['fft.cuh', 'fft_ct.cuh', 'tail.cuh', 'obs_star.cuh']
_FAST = _FFT + ['tail_fast.cuh', 'tail_general.cuh']
# translation unit -> the headers whose change alters its object code
UNITS = {
    'payne_b200.cu': ['mlp_simt.cuh', 'mlp_tc_types.h'] + _FAST + ['launchers.h', 'phot.cuh', 'continuum.cuh', 'tail_lsf.cuh'],
    'gemm_tu.cu': _GEMM + ['mlp_tc_types.h', 'launchers.h'],
    'tail_fast_tu.cu': _FAST + ['launchers.h', 'tail_fast_tu.inl'],
    'tail_fast_poly_tu.cu': _FAST + ['launchers.h', 'tail_fast_tu.inl'],
    'tail_cluster_tu.cu': _FAST + ['tail_cluster.cuh', 'launchers.h'],
    'tail_general_tu.cu': _FFT + ['tail_general.cuh', 'tail_lsf.cuh', 'continuum.cuh', 'launchers.h'],
}


def nvcc_path():
    for c in [os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc']:
        if c and os.path.exists(c):
            return c
    raise RuntimeError('nvcc not found')


def _deps(unit):
    return [os.path.join(CSRC, unit), HDR, os.path.abspath(__file__)] + \
           [os.path.join(CSRC, h) for h in UNITS[unit] if os.path.exists(os.path.join(CSRC, h))]


# Development switch: PAYNE_FAST_ONLY=14 compiles the fast tail for that transform size only (every other
# size then reports "unsupported"); the object gets its own name so a full build never picks it up.
FAST_ONLY = os.environ.get('PAYNE_FAST_ONLY', '')
_FAST_UNITS = ('tail_fast_tu.cu', 'tail_fast_poly_tu.cu')


def _obj(unit):
    tag = ('_only' + FAST_ONLY) if (FAST_ONLY and unit in _FAST_UNITS) else ''
    return os.path.join(OBJ, unit[:-3] + tag + '.o')


def _stale(unit):
    o = _obj(unit)
    return not os.path.exists(o) or any(os.path.getmtime(d) > os.path.getmtime(o) for d in _deps(unit))


FLAVOR = os.path.join(OBJ, 'flavor')      # which tail_fast object the current .so was linked from


def _flavor():
    try:
        return open(FLAVOR).read().strip()
    except OSError:
        return '?'


def needs_build():
    if not os.path.exists(OUT) or _flavor() != ('only' + FAST_ONLY if FAST_ONLY else 'full'):
        return True
    t = os.path.getmtime(OUT)
    if FAST_ONLY and any(_stale(u) or os.path.getmtime(_obj(u)) > t for u in _FAST_UNITS):
        return True
    return any(os.path.getmtime(d) > t for u in UNITS for d in _deps(u))


def _compile(unit, verbose):
    # (-split-compile would shorten the tail units further, but the tail kernel it produces is 39 % slower
    # on B200 -- measured -- so each unit keeps the single-threaded optimiser)
    cmd = [nvcc_path(), '-O3', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo',
           '-Xcompiler', '-fPIC', '-c', '-o', _obj(unit), os.path.join(CSRC, unit)]
    if verbose:
        cmd[1:1] = ['-Xptxas', '-v']
    if FAST_ONLY and unit in _FAST_UNITS:
        cmd[1:1] = ['-DPAYNE_FAST_ONLY=' + FAST_ONLY]
    r = subprocess.run(cmd, capture_output=True, text=True)
    return unit, r


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    os.makedirs(OBJ, exist_ok=True)
    todo = [u for u in UNITS if force or _stale(u)]
    with ThreadPoolExecutor(max_workers=max(1, min(len(todo), os.cpu_count() or 1))) as ex:
        results = list(ex.map(lambda u: _compile(u, verbose), todo))
    for unit, r in results:
        if verbose or r.returncode != 0:
            sys.stderr.write('== %s\n%s%s' % (unit, r.stdout, r.stderr))
        if r.returncode != 0:
            raise RuntimeError('nvcc failed on %s:\n%s' % (unit, r.stderr[-4000:]))
    link = [nvcc_path(), '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', OUT] + [_obj(u) for u in UNITS]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('link failed:\n' + r.stderr[-4000:])
    with open(FLAVOR, 'w') as f:
        f.write('only' + FAST_ONLY if FAST_ONLY else 'full')
    return OUT


if __name__ == '__main__':
    print(build(force='-f' in sys.argv or '-v' in sys.argv, verbose='-v' in sys.argv))
