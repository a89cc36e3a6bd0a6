"""The tcgen05 GEMM kernel alone (payne_gemm_test hook) against float64 matmul and a bit-level model of parity mode.

The parity mode ("X3": three 8-bit fixed-point bf16 slices per operand, mlp_tc.cuh) must be EXACT whenever
the dominant slice products sum to an fp32-representable integer -- that is the property the
whole scheme rests on (the TMEM accumulator never rounds) -- and correctly rounded to fp32
accuracy on random data.

`x3_model` restates what the code computes, in float64:
  * weights (tc_prepare_weights): per row the power of two s_n = 2^e, max|w_n| = m 2^e with 0.5 <= m < 1 (1 for an
    all-zero row), and u = w / s_n cut into q1, q2, q3 on the 2^-7 / 2^-15 / 2^-23 grids;
  * activations (x3_split_act): p1, p2, p3 on the 2^-8 / 2^-16 / 2^-24 grids;
  every cut rounds to nearest, ties to even (np.rint);
  * the leading sum v = sum p1 q1 and the five kept cross terms c = sum p1q2 + p2q1 + p1q3 + p2q2 + p3q1, both exact in
    float64 (grids 2^-15 and 2^-31, magnitudes below 2^10 for K <= 512);
  * the epilogue (epi_store_block): fl32(fl32(v + c) s_n + b).
The tensor core sums the cross terms in its fp32 accumulator, whose rounding is ~2^-32 of the result.  That can tip the
first rounding, fl32(v + c), by one ulp of v + c, and where the bias cancels part of the product the second rounding
magnifies it: measured on B200, one element at (M, N, K) = (127, 260, 512) was 4 ulps of the output from the model,
v s = -0.632 against b = 0.840.  So the kernel may differ from the model by one ulp at either rounding,
ulp(y) + s_n ulp(v + c), and at least 97 % of all elements must be bit-identical to it (measured: 99.99 % at K = 8,
99.4 % at K = 256, 98.9 % at K = 384; the share falls with K as the cross-term sums grow).

The CPU tests check the model itself: it stays within the dropped terms of the float64 product and reproduces the
integer-exactness property.  The GPU tests run a matrix of shapes that includes K below one 64-element stage and off
its multiples, M and N ragged against the 128-row / 128-column tiles and the 32-column store box, and two shapes with
more than 3 x 148 output tiles, so every CTA of the persistent grid works through several tiles (ring-phase wrap,
double-buffered accumulator handover, epilogue under the next tile's MMAs).
"""
import numpy as np
import pytest

KS = [8, 16, 24, 56, 64, 72, 100, 128, 200, 256, 384, 512]
MS = [1, 2, 127, 128, 129, 255]
NS = [4, 28, 32, 36, 124, 128, 132, 260]     # the hook writes with pitch N: the TMA-store map needs N % 4 == 0
LARGE = [(4096, 2048, 256), (2560, 4096, 512)]   # 512 and 640 output tiles of 128 x 128


def gemm(A, W, b, prec):
    from thepayne_b200 import _lib
    lib = _lib.load()
    A, W, b = [np.ascontiguousarray(x, dtype=np.float32) for x in (A, W, b)]
    M, K = A.shape
    N = W.shape[0]
    C = np.empty((M, N), dtype=np.float32)
    _lib.check(lib.payne_gemm_test(A.ctypes.data, W.ctypes.data, b.ctypes.data, M, N, K, _lib.PREC[prec], 0,
                                   C.ctypes.data))
    return C


# ------------------------------------------------------------------ the model
def x3_act_slices(A):
    h = np.asarray(A, dtype=np.float32).astype(np.float64)
    p1 = np.rint(h * 2.0 ** 8) / 2.0 ** 8
    r1 = h - p1
    p2 = np.rint(r1 * 2.0 ** 16) / 2.0 ** 16
    p3 = np.rint((r1 - p2) * 2.0 ** 24) / 2.0 ** 24
    return p1, p2, p3


def x3_weight_slices(W):
    w = np.asarray(W, dtype=np.float32).astype(np.float64)
    _, e = np.frexp(np.abs(w).max(axis=1))       # frexp(0) = (0, 0): an all-zero row gets s = 1, as on the host
    s = np.ldexp(1.0, e)
    u = w / s[:, None]
    q1 = np.rint(u * 2.0 ** 7) / 2.0 ** 7
    r1 = u - q1
    q2 = np.rint(r1 * 2.0 ** 15) / 2.0 ** 15
    q3 = np.rint((r1 - q2) * 2.0 ** 23) / 2.0 ** 23
    return s, q1, q2, q3


def x3_parts(A, W):
    """(v, c, s): leading sum, kept cross terms (both exact in float64, [M, N]) and the row scales [N]."""
    p1, p2, p3 = x3_act_slices(A)
    s, q1, q2, q3 = x3_weight_slices(W)
    v = p1 @ q1.T
    c = p1 @ (q2 + q3).T + p2 @ (q1 + q2).T + p3 @ q1.T      # p1q2 + p1q3 + p2q1 + p2q2 + p3q1, all on the 2^-31 grid
    return v, c, s


def x3_model(A, W, b, slack=False):
    """fl32(fl32(v + c) s_n + b); slack=True also returns the allowance ulp(y) + s_n ulp(v + c)."""
    v, c, s = x3_parts(A, W)
    t = (v + c).astype(np.float32)
    y = (t.astype(np.float64) * s[None, :] + np.asarray(b, dtype=np.float32).astype(np.float64)[None, :])
    y = y.astype(np.float32)
    if not slack:
        return y
    return y, np.spacing(np.abs(y)).astype(np.float64) + np.spacing(np.abs(t)).astype(np.float64) * s[None, :]


def ulp_distance(a, b):
    """Distance in units in the last place between two float32 arrays (sign-aware, 0 for equal values)."""
    def ordered(x):
        i = np.ascontiguousarray(x, dtype=np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.abs(ordered(a) - ordered(b))


# ------------------------------------------------------------------ inputs
def random_inputs(M, N, K, seed):
    """Sigmoid-like activations with the edge values of the slicing, weight rows with the edges of the row scale."""
    rng = np.random.default_rng(seed)
    A = 1.0 / (1.0 + np.exp(-2.0 * rng.standard_normal((M, K))))
    edges = [0.0, 1.0, 1.0 - 2.0 ** -24, 2.0 ** -30]        # 1.0 is a saturated sigmoid: slice k1 = 256
    idx = rng.integers(0, M * K, size=(len(edges), max(1, M * K // 16)))
    for v, ii in zip(edges, idx):
        A.flat[ii] = v
    A[0, :] = np.array(edges)[np.arange(K) % 4]
    W = (rng.random((N, K)) - 0.5) * 0.04
    W[0] = 0.0                                              # all-zero row: s_n = 1
    W[1, 0] = 0.03125                                       # row maximum exactly a power of two
    W[1, 1:] = np.clip(W[1, 1:], -0.03, 0.03)
    W[2] *= 10.0 ** rng.uniform(-6.0, 0.0, K)               # 1e6 dynamic range within the row
    W[2, 0] = 0.02
    if N > 4:
        W[N // 2] = 0.0
    b = rng.standard_normal(N) * 0.1 + 1.0
    return A.astype(np.float32), W.astype(np.float32), b.astype(np.float32)


def integer_inputs(M, N, K, seed):
    """One activation slice and one weight slice: the products sum to fp32-exact values (p1 q1 only)."""
    rng = np.random.default_rng(seed)
    A = rng.integers(0, 257, (M, K)).astype(np.float64) / 256.0              # includes 1.0 (k1 = 256)
    W = rng.integers(-128, 129, (N, K)).astype(np.float64) / 128.0 * 0.125
    W[:, 0] = 0.125 * (1 - 2.0 ** -7)                 # pins every row scale to 2^-3
    return A.astype(np.float32), W.astype(np.float32), np.zeros(N, dtype=np.float32)


def reference(A, W, b):
    return A.astype(np.float64) @ W.astype(np.float64).T + b.astype(np.float64)[None, :]


# ------------------------------------------------------------------ CPU: the model itself
@pytest.mark.parametrize('K', [8, 72, 256, 512])
def test_x3_model_within_the_dropped_terms(K):
    """The kept slice products differ from the float64 product only by p2q3 + p3q2 + p3q3 and the slicing residues of
    h and w: per product at most (3 * 2^-25 + 2^-32 + |h| 2^-24) s_n, and with random signs their sum stays within a
    random walk of 2^-24 s_n steps."""
    M, N = 96, 80
    A, W, b = random_inputs(M, N, K, seed=K)
    v, c, s = x3_parts(A, W)
    exact = A.astype(np.float64) @ W.astype(np.float64).T
    err = np.abs((v + c) * s[None, :] - exact)
    bound = (np.abs(A.astype(np.float64)).sum(1)[:, None] * 2.0 ** -24 + K * (3 * 2.0 ** -25 + 2.0 ** -32)) * s[None, :]
    assert np.all(err <= bound), np.max(err / bound)
    assert np.all(err <= 6.0 * np.sqrt(K) * 2.0 ** -24 * s[None, :])
    # the slices are what the kernel stores: bf16-exact (at most 8 significant bits) and on their grids
    p1, p2, p3 = x3_act_slices(A)
    for p, g in [(p1, 8), (p2, 16), (p3, 24)]:
        k = p * 2.0 ** g
        assert np.array_equal(k, np.rint(k)) and np.abs(k).max() <= 256
    sw, q1, q2, q3 = x3_weight_slices(W)
    for q, g in [(q1, 7), (q2, 15), (q3, 23)]:
        k = q * 2.0 ** g
        assert np.array_equal(k, np.rint(k)) and np.abs(k).max() <= 128
    assert sw[0] == 1.0 and sw[1] == 0.0625           # zero row; max exactly 2^-5 -> s = 2^-4 (frexp convention)
    # after the epilogue's two roundings the model is within one fp32 ulp of the float64 result (plus the dropped terms)
    y = x3_model(A, W, b)
    ref = reference(A, W, b)
    assert np.all(np.abs(y - ref) <= 2.0 ** -24 * (np.abs(exact) + np.abs(ref)) * (1 + 1e-6) + bound)


@pytest.mark.parametrize('K', [8, 64, 100, 512])
def test_x3_model_integer_sums_are_exact(K):
    A, W, b = integer_inputs(70, 50, K, seed=K)
    assert np.array_equal(x3_model(A, W, b).astype(np.float64), reference(A, W, b))


def test_ulp_distance():
    a = np.array([1.0, -1.0, 0.0, 0.0, 1.0], dtype=np.float32)
    b = np.array([np.nextafter(np.float32(1), np.float32(2)), -1.0, -0.0, np.float32(1.4e-45), 1.0], dtype=np.float32)
    assert list(ulp_distance(a, b)) == [1, 0, 0, 1, 0]


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize('K', [64, 256, 512])
def test_x3_integer_sums_are_exact(K):
    M, N = 300, 700                                   # ragged in M and N on purpose
    A, W, b = integer_inputs(M, N, K, seed=K)
    C = gemm(A, W, b, 'parity')
    assert np.array_equal(C.astype(np.float64), reference(A, W, b))   # exact in float64 (integers < 2^53)


def _shapes(K):
    out = [(M, N, K) for M in MS for N in NS]
    return out + [s for s in LARGE if s[2] == K]


@pytest.mark.gpu
@pytest.mark.parametrize('K', KS)
def test_x3_shape_matrix_against_the_model(K):
    """Parity mode at every (M, N) of the matrix: within one rounding of the model, integer inputs bit-exact, no bias."""
    n_el = n_same = worst = 0
    rel = []
    for M, N, KK in _shapes(K):
        A, W, b = random_inputs(M, N, K, seed=M * 7919 + N * 31 + K)
        C = gemm(A, W, b, 'parity')
        y, slack = x3_model(A, W, b, slack=True)
        d = ulp_distance(C, y)
        worst = max(worst, int(d.max()))
        n_el += d.size
        n_same += int((d == 0).sum())
        bad = np.abs(C.astype(np.float64) - y) > slack
        assert not bad.any(), (M, N, K, int(d.max()), np.argwhere(bad)[:5])
        ref = reference(A, W, b)
        rel.append(((C - ref) / np.abs(ref)).ravel())
        Ai, Wi, bi = integer_inputs(M, N, K, seed=M + N + K)
        assert np.array_equal(gemm(Ai, Wi, bi, 'parity').astype(np.float64), reference(Ai, Wi, bi)), (M, N, K)
    rel = np.concatenate(rel)
    print('K=%d: %d elements, max %d ulp from the model, %.5f%% bit-identical; max rel err %.2e, mean %.2e'
          % (K, n_el, worst, 100.0 * n_same / n_el, np.abs(rel).max(), rel.mean()))
    assert n_same >= 0.97 * n_el
    assert abs(rel.mean()) <= 2e-9


@pytest.mark.gpu
@pytest.mark.parametrize('prec,bar', [('3xtf32', 3e-6), ('tf32', 3e-3)])
@pytest.mark.parametrize('K', KS)
def test_tf32_modes_shape_matrix(K, prec, bar):
    """The kModeT3 / kModeT1 instantiations at the same shapes (a shape check, not a parity claim).

    The error is taken relative to the sum of magnitudes |A| |W|^T + |b|: these inputs include outputs where the bias
    cancels most of the product, and relative to |C| alone 3xtf32 measured 3.6e-6 there (K = 384), tf32 above 3e-3."""
    for M, N, KK in _shapes(K):
        A, W, b = random_inputs(M, N, K, seed=M * 7919 + N * 31 + K)
        C = gemm(A, W, b, prec)
        ref = reference(A, W, b)
        mag = np.abs(A.astype(np.float64)) @ np.abs(W.astype(np.float64)).T + np.abs(b.astype(np.float64))[None, :]
        err = np.abs(C - ref) / mag
        assert err.max() <= bar, (M, N, K, err.max())


@pytest.mark.gpu
@pytest.mark.parametrize('prec,bar', [('parity', 1.5e-7), ('3xtf32', 3e-6), ('tf32', 3e-3)])
def test_gemm_accuracy_random(prec, bar):
    rng = np.random.default_rng(7)
    M, N, K = 513, 1000, 256
    A = 1.0 / (1.0 + np.exp(-rng.standard_normal((M, K))))               # sigmoid-like activations
    W = (rng.random((N, K)) - 0.5) * 0.04
    b = rng.standard_normal(N) * 0.1 + 1.0
    A32, W32, b32 = A.astype(np.float32), W.astype(np.float32), b.astype(np.float32)
    ref = A32.astype(np.float64) @ W32.astype(np.float64).T + b32.astype(np.float64)
    C = gemm(A32, W32, b32, prec)
    err = np.abs(C - ref) / np.abs(ref)
    assert err.max() <= bar, err.max()
    if prec == 'parity':
        # no coherent bias: the mean signed error is far below one fp32 ulp
        assert abs(np.mean((C - ref) / np.abs(ref))) < 2e-9
        y, slack = x3_model(A32, W32, b32, slack=True)
        assert np.all(np.abs(C.astype(np.float64) - y) <= slack)
