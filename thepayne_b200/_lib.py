"""ctypes binding of libpayne_b200.so (the C ABI declared in include/payne_b200.h).

There is deliberately no fallback: if the CUDA library is missing or fails to load, every
entry point raises.  The product never imports ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# PAYNE_LIB_PATH: development override (an instrumented build of the same sources)
LIB_PATH = os.environ.get('PAYNE_LIB_PATH') or os.path.join(HERE, 'libpayne_b200.so')

ABI_VERSION = 8          # PAYNE_ABI_VERSION of include/payne_b200.h the ctypes structs below mirror
NPAR = 13
MAX_POLY = 16
PAR_INDEX = {
    'Teff': 0, 'log(g)': 1, '[Fe/H]': 2, '[a/Fe]': 3, 'Vrad': 4, 'Vrot': 5, 'Vmic': 6,
    'Inst_R': 7, 'log(R)': 8, 'Dist': 9, 'log(A)': 10, 'Av': 11, 'Rv': 12,
}
PREC = {'parity': 0, 'x3': 0, 'tf32': 1, 'bf16': 2, 'simt': 3, 'fp32': 3, '3xtf32': 4}

EXPORTS = ['payne_abi_version', 'payne_last_error', 'payne_ctx_create', 'payne_ctx_destroy',
           'payne_lnlike_batch', 'payne_lnlike_batch_host', 'payne_model_batch', 'payne_ann_eval',
           'payne_ctx_query', 'payne_ctx_set', 'payne_ctx_last_ms', 'payne_gemm_test', 'payne_fft_test',
           'payne_ctx_attach_continuum', 'payne_ctx_set_lsf',
           'payne_gather_create', 'payne_gather_connect', 'payne_lnlike_batch_gather', 'payne_gather_flush',
           'payne_ctx_create_stars', 'payne_lnlike_batch_stars', 'payne_lnlike_batch_stars_host',
           'payne_model_batch_stars', 'payne_ctx_create_stars_opts',
           'payne_ctx_set_targets', 'payne_lnlike_batch_targets', 'payne_lnlike_batch_targets_host',
           'payne_model_batch_targets',
           'payne_ctx_set_binary', 'payne_lnlike_batch_binary', 'payne_lnlike_batch_binary_host',
           'payne_model_batch_binary',
           'payne_ctx_set_cont_marg', 'payne_cont_batch_stars', 'payne_cont_batch_targets']
GATHER_HANDLE_BYTES = 128

_f = C.POINTER(C.c_float)
_d = C.POINTER(C.c_double)


class PayneSpecNet(C.Structure):
    _fields_ = [('D_in', C.c_int32), ('H1', C.c_int32), ('H2', C.c_int32), ('H3', C.c_int32),
                ('D_out', C.c_int32), ('W', _f * 6), ('b', _f * 6), ('xmin', _d), ('xmax', _d),
                ('wavelength', _d), ('resolution', C.c_double), ('encode_offset', C.c_double),
                ('n_layers', C.c_int32), ('activation', C.c_int32), ('label_fp32_cast', C.c_int32),
                ('n_groups', C.c_int32), ('group_size', C.c_int32), ('reserved_', C.c_int32)]


class PaynePhotNet(C.Structure):
    _fields_ = [('nb', C.c_int32), ('H', C.c_int32), ('w1', _f), ('b1', _f), ('w2', _f), ('b2', _f),
                ('w3', _f), ('b3', _f), ('xmin', _d), ('xmax', _d), ('hiav', _d)]


class PayneObs(C.Structure):
    _fields_ = [('n_obs', C.c_int32), ('wave', _d), ('flux', _d), ('eflux', _d),
                ('nb', C.c_int32), ('phot_mag', _d), ('phot_err', _d)]


class PayneLayout(C.Structure):
    _fields_ = [('ndim', C.c_int32), ('col', C.c_int32 * NPAR), ('fixed', C.c_double * NPAR),
                ('n_poly', C.c_int32), ('poly_col', C.c_int32 * MAX_POLY),
                ('spec_bool', C.c_int32), ('phot_bool', C.c_int32), ('modpoly_bool', C.c_int32),
                ('photscale_bool', C.c_int32), ('precision', C.c_int32)]


class PayneStarOpts(C.Structure):
    _fields_ = [('fixed', _d), ('band', C.POINTER(C.c_int32)), ('lsf', _d), ('layout', C.POINTER(PayneLayout))]


class PayneBinary(C.Structure):
    _fields_ = [('col', C.c_int32 * NPAR), ('fixed', C.c_double * NPAR), ('rratio_col', C.c_int32),
                ('rratio_fixed', C.c_double)]


class PayneContMarg(C.Structure):
    _fields_ = [('n_coef', C.c_int32), ('lo', C.c_double * MAX_POLY), ('hi', C.c_double * MAX_POLY)]


class PayneError(RuntimeError):
    pass


_lib = None


def load():
    """Load the CUDA library (built in-tree by ``thepayne_b200/build.py``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PayneError(
            'libpayne_b200.so is missing (%s). Build it with `python -m thepayne_b200.build`; '
            'there is no CPU fallback.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.payne_abi_version.restype = C.c_int
    got = lib.payne_abi_version()
    if got != ABI_VERSION:
        raise PayneError('%s has ABI version %d, these bindings expect %d: rebuild it with '
                         '`python -m thepayne_b200.build`' % (LIB_PATH, got, ABI_VERSION))
    lib.payne_last_error.restype = C.c_char_p
    lib.payne_ctx_create.restype = C.c_int
    lib.payne_ctx_create.argtypes = [C.POINTER(PayneSpecNet), C.POINTER(PaynePhotNet), C.POINTER(PayneObs),
                                     C.POINTER(PayneLayout), C.c_int, C.POINTER(vp)]
    lib.payne_ctx_create_stars.restype = C.c_int
    lib.payne_ctx_create_stars.argtypes = [C.POINTER(PayneSpecNet), C.POINTER(PaynePhotNet), C.POINTER(PayneObs),
                                           C.c_int32, C.POINTER(PayneLayout), C.c_int, C.POINTER(vp)]
    lib.payne_ctx_create_stars_opts.restype = C.c_int
    lib.payne_ctx_create_stars_opts.argtypes = [C.POINTER(PayneSpecNet), C.POINTER(PaynePhotNet), C.POINTER(PayneObs),
                                                C.POINTER(PayneStarOpts), C.c_int32, C.POINTER(PayneLayout), C.c_int,
                                                C.POINTER(vp)]
    lib.payne_lnlike_batch_stars.restype = C.c_int
    lib.payne_lnlike_batch_stars.argtypes = [vp, vp, vp, C.c_int64, C.c_int64, vp, vp]
    lib.payne_lnlike_batch_stars_host.restype = C.c_int
    lib.payne_lnlike_batch_stars_host.argtypes = [vp, vp, vp, C.c_int64, C.c_int64, vp]
    lib.payne_model_batch_stars.restype = C.c_int
    lib.payne_model_batch_stars.argtypes = [vp, vp, vp, C.c_int64, C.c_int64, vp, C.c_int64, vp, vp, vp]
    lib.payne_ctx_set_targets.restype = C.c_int
    lib.payne_ctx_set_targets.argtypes = [vp, vp, C.c_int32]
    lib.payne_lnlike_batch_targets.restype = C.c_int
    lib.payne_lnlike_batch_targets.argtypes = [vp, vp, vp, C.c_int64, C.c_int64, vp, vp]
    lib.payne_lnlike_batch_targets_host.restype = C.c_int
    lib.payne_lnlike_batch_targets_host.argtypes = [vp, vp, vp, C.c_int64, C.c_int64, vp]
    lib.payne_model_batch_targets.restype = C.c_int
    lib.payne_model_batch_targets.argtypes = [vp, vp, vp, C.c_int64, C.c_int64, vp, C.c_int64, vp, C.c_int64, vp, vp, vp]
    lib.payne_ctx_set_binary.restype = C.c_int
    lib.payne_ctx_set_binary.argtypes = [vp, C.POINTER(PayneBinary)]
    lib.payne_lnlike_batch_binary.restype = C.c_int
    lib.payne_lnlike_batch_binary.argtypes = [vp, vp, vp, C.c_int64, C.c_int64, vp, vp]
    lib.payne_lnlike_batch_binary_host.restype = C.c_int
    lib.payne_lnlike_batch_binary_host.argtypes = [vp, vp, vp, C.c_int64, C.c_int64, vp]
    lib.payne_model_batch_binary.restype = C.c_int
    lib.payne_model_batch_binary.argtypes = [vp, vp, vp, C.c_int64, C.c_int64, vp, C.c_int64, vp, vp, vp]
    lib.payne_ctx_set_cont_marg.restype = C.c_int
    lib.payne_ctx_set_cont_marg.argtypes = [vp, C.POINTER(PayneContMarg)]
    lib.payne_cont_batch_stars.restype = C.c_int
    lib.payne_cont_batch_stars.argtypes = [vp, vp, vp, C.c_int64, C.c_int64, vp, C.c_int64, vp, C.c_int64, vp, vp, vp]
    lib.payne_cont_batch_targets.restype = C.c_int
    lib.payne_cont_batch_targets.argtypes = [vp, vp, vp, C.c_int64, C.c_int64, vp, C.c_int64, vp, C.c_int64, vp,
                                             C.c_int64, vp, vp]
    lib.payne_ctx_destroy.restype = None
    lib.payne_ctx_destroy.argtypes = [vp]
    lib.payne_lnlike_batch.restype = C.c_int
    lib.payne_lnlike_batch.argtypes = [vp, vp, C.c_int64, C.c_int64, vp, vp]
    lib.payne_lnlike_batch_host.restype = C.c_int
    lib.payne_lnlike_batch_host.argtypes = [vp, vp, C.c_int64, C.c_int64, vp]
    lib.payne_model_batch.restype = C.c_int
    lib.payne_model_batch.argtypes = [vp, vp, C.c_int64, C.c_int64, vp, vp, vp, vp]
    lib.payne_ann_eval.restype = C.c_int
    lib.payne_ann_eval.argtypes = [vp, vp, C.c_int64, vp, C.c_int64, vp]
    lib.payne_ctx_attach_continuum.restype = C.c_int
    lib.payne_ctx_attach_continuum.argtypes = [vp, C.POINTER(PayneSpecNet)]
    lib.payne_ctx_set_lsf.restype = C.c_int
    lib.payne_ctx_set_lsf.argtypes = [vp, vp, C.c_int64]
    lib.payne_gather_create.restype = C.c_int
    lib.payne_gather_create.argtypes = [vp, C.c_int, C.c_int, C.c_int64, vp]
    lib.payne_gather_connect.restype = C.c_int
    lib.payne_gather_connect.argtypes = [vp, vp]
    lib.payne_lnlike_batch_gather.restype = C.c_int
    lib.payne_lnlike_batch_gather.argtypes = [vp, vp, C.c_int64, C.c_int64, vp, C.POINTER(vp)]
    lib.payne_gather_flush.restype = C.c_int
    lib.payne_gather_flush.argtypes = [vp, vp, C.POINTER(vp)]
    lib.payne_ctx_query.restype = C.c_int64
    lib.payne_ctx_query.argtypes = [vp, C.c_char_p]
    lib.payne_ctx_set.restype = C.c_int
    lib.payne_ctx_set.argtypes = [vp, C.c_char_p, C.c_int64]
    lib.payne_ctx_last_ms.restype = C.c_double
    lib.payne_ctx_last_ms.argtypes = [vp, C.c_int]
    lib.payne_gemm_test.restype = C.c_int
    lib.payne_gemm_test.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.payne_fft_test.restype = C.c_int
    lib.payne_fft_test.argtypes = [vp, C.c_int, vp, C.c_int, vp]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().payne_last_error()
        raise PayneError('payne_b200 error %d: %s' % (rc, msg.decode() if msg else '?'))
