"""GPU: the operator-level drop-in (`compute_Z_q_expectations` with host buffers, zigap.py:79-95 /
gap.py:67-80) against the reference's numba output (golden) and the sequential C loop oracle."""
import ctypes

import numpy as np
import pytest

from conftest import GOLDEN_CASES, golden_state, load_golden, relerr

pytestmark = pytest.mark.gpu


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def z_op(lib, lU, lV, X, D=None, quirk=True, third=False):
    from oriana_b200 import _lib
    n, K = lU.shape; p = lV.shape[0]
    Zi = np.full((n, K), np.nan, np.float32); Zj = np.full((p, K), np.nan, np.float32)
    Z3 = np.full((p, K), np.nan, np.float32) if third else None
    arrs = [np.ascontiguousarray(a, dtype=np.float32) for a in (lU, lV, X)]
    if D is None:
        _lib.check(lib.ori_gap_compute_Z_q_expectations_host(_ptr(Zi), _ptr(Zj), _ptr(arrs[0]), _ptr(arrs[1]),
                                                             _ptr(arrs[2]), n, p, K))
    else:
        D = np.ascontiguousarray(D, dtype=np.float32)
        _lib.check(lib.ori_zigap_compute_Z_q_expectations_host(_ptr(Zi), _ptr(Zj), _ptr(Z3), _ptr(arrs[0]),
                                                               _ptr(arrs[1]), _ptr(D), _ptr(arrs[2]), n, p, K,
                                                               int(quirk)))
    return (Zi, Zj, Z3) if third else (Zi, Zj)


@pytest.mark.parametrize('name', GOLDEN_CASES)
def test_against_reference_numba_kernel(cuda_lib, name):
    from oracle import cavi_numpy as cn
    g = load_golden(name)
    s = golden_state(g, 0)
    D = cn.expectations(s).get('D_hat')
    Zi, Zj = z_op(cuda_lib, g['z_log_U_hat'], g['z_log_V_hat'], s['X'], D, quirk=True)
    assert relerr(Zi, g['z_Zi']) < 1e-5, relerr(Zi, g['z_Zi'])
    assert relerr(Zj, g['z_Zj']) < 1e-5, relerr(Zj, g['z_Zj'])


@pytest.mark.parametrize('quirk', [True, False])
@pytest.mark.parametrize('shape', [(1, 3, 1), (5, 7, 3), (129, 33, 8), (260, 517, 9), (300, 140, 17), (70, 90, 40)])
def test_against_c_loop_with_soft_dropout(cuda_lib, shape, quirk):
    """Arbitrary D_hat in (0,1) (not just the indicator), ragged shapes, every padded-K bucket, third output."""
    from oracle import zloop
    n, p, K = shape
    if quirk and p < K:
        pytest.skip('zigap.py:94 indexes D_hat[i, k]: needs p >= K')
    rng = np.random.default_rng(n * 1000 + p)
    lU = rng.normal(-0.5, 1.0, (n, K)).astype(np.float32)
    lV = rng.normal(-0.5, 1.0, (p, K)).astype(np.float32)
    X = (rng.poisson(3.0, (n, p)) * (rng.random((n, p)) < 0.6)).astype(np.float32)
    D = np.where(X != 0, 1.0, rng.random((n, p))).astype(np.float32)
    Zi, Zj, Z3 = z_op(cuda_lib, lU, lV, X, D, quirk=quirk, third=True)
    rZi, rZj, rZ3 = zloop.zigap_z(lU, lV, D, X, quirk=quirk, third=True)
    assert relerr(Zi, rZi) < 1e-5 and relerr(Zj, rZj) < 1e-5
    # signed terms cancel in zigap.py:95: judge the absolute error against the array's scale
    assert np.max(np.abs(Z3 - rZ3)) < 3e-6 * np.max(np.abs(rZ3))
    gZi, gZj = z_op(cuda_lib, lU, lV, X)
    rZi, rZj = zloop.gap_z(lU, lV, X)
    assert relerr(gZi, rZi) < 1e-5 and relerr(gZj, rZj) < 1e-5


def test_underflow_guard_and_empty(cuda_lib):
    """zigap.py:88-90: den <= 0 -> 1 when every exp underflows; n = 0 leaves zero gene sums.

    The log-expectations are centred per row before the exp (csrc/special.cuh), so the centred denominators stay
    positive where the reference's float32 exp(lU + lV) is 0 for every component; the operator carries the reference's
    underflow thresholds (underflow_thr_f32) and assigns such counts to nobody, like the reference."""
    from oracle import zloop
    X = np.arange(24, dtype=np.float32).reshape(4, 6)
    lU = np.full((4, 2), -3e4, np.float32); lV = np.full((6, 2), -1.5, np.float32)
    Zi, Zj = z_op(cuda_lib, lU, lV, X)
    rZi, rZj = zloop.gap_z(lU, lV, X)
    assert np.array_equal(Zi, rZi) and np.array_equal(Zj, rZj) and not Zi.any() and not Zj.any()
    lU = np.full((4, 2), -200., np.float32); lV = np.full((6, 2), -200., np.float32)
    Zi, Zj = z_op(cuda_lib, lU, lV, X)
    assert not zloop.gap_z(lU, lV, X)[0].any()                    # the reference: all zero
    assert not Zi.any() and not Zj.any()
    # -60 and -60: exp(-120) is 0 in float32 although neither factor is out of range on its own
    lU = np.full((4, 2), -60., np.float32); lV = np.full((6, 2), -60., np.float32)
    Zi, Zj = z_op(cuda_lib, lU, lV, X)
    assert not zloop.gap_z(lU, lV, X)[0].any() and not Zi.any() and not Zj.any()
    # -60 and -20: a normal float32 number (e^-80): the ratios (1/2 each) are kept
    lV = np.full((6, 2), -20., np.float32)
    Zi, Zj = z_op(cuda_lib, lU, lV, X)
    rZi, rZj = zloop.gap_z(lU, lV, X)
    np.testing.assert_allclose(Zi, rZi, rtol=1e-5); np.testing.assert_allclose(Zj, rZj, rtol=1e-5)
    np.testing.assert_allclose(Zi, np.repeat(X.sum(1, keepdims=True) / 2, 2, axis=1), rtol=1e-5)
    # one component 150 below the other: flushed (the reference's exp underflows for it as well)
    lU = np.tile(np.asarray([[-1., -151.]], np.float32), (4, 1)); lV = np.tile(np.asarray([[-0.5, -0.5]], np.float32), (6, 1))
    Zi, Zj = z_op(cuda_lib, lU, lV, X)
    rZi, rZj = zloop.gap_z(lU, lV, X)
    np.testing.assert_allclose(Zi, rZi, rtol=1e-6, atol=1e-30); np.testing.assert_allclose(Zj, rZj, rtol=1e-6, atol=1e-30)
    assert not Zi[:, 1].any()
    Zi, Zj = z_op(cuda_lib, np.zeros((0, 3), np.float32), np.zeros((5, 3), np.float32), np.zeros((0, 5), np.float32))
    assert Zi.shape == (0, 3) and not Zj.any()


def test_bad_arguments_raise(cuda_lib):
    from oriana_b200 import _lib
    with pytest.raises(_lib.OrianaB200Error):
        z_op(cuda_lib, np.zeros((2, 70), np.float32), np.zeros((80, 70), np.float32), np.zeros((2, 80), np.float32))
    with pytest.raises(_lib.OrianaB200Error):   # quirk needs p >= K
        z_op(cuda_lib, np.zeros((2, 5), np.float32), np.zeros((3, 5), np.float32), np.zeros((2, 3), np.float32),
             np.ones((2, 3), np.float32), quirk=True)
    # the third gene sum (eUl) belongs to the sparse model: a ZIGaP problem that asks for it is refused
    from oriana.models import ZIGaP
    P = _lib.OriProblem.from_buffer_copy(ZIGaP(np.ones((4, 6)), k=2, use_factors=False)._P)
    _lib.check(cuda_lib.ori_problem_check(ctypes.byref(P)))
    P.eUl[0] = P.eU[0]
    with pytest.raises(_lib.OrianaB200Error):
        _lib.check(cuda_lib.ori_problem_check(ctypes.byref(P)))


def _stats(lib, ctx=None):
    c = [ctypes.c_uint64(0) for _ in range(4)]
    from oriana_b200 import _lib
    _lib.check(lib.ori_ctx_stats(ctx, *[ctypes.byref(x) for x in c]))
    return dict(zip(('calls', 'allocs', 'tensor_slabs', 'simt_slabs'), (int(x.value) for x in c)))


@pytest.mark.parametrize('quirk', [True, False])
@pytest.mark.parametrize('K', [10, 40])
def test_tensor_sized_slabs_take_the_tcgen05_passes(cuda_lib, K, quirk):
    """Slabs of >= 2^21 entries go through the tcgen05 / TMA kernels (TF32 operands: 1e-3 against the sequential float32
    loop of the reference, restated in C), through an explicit context with three ragged slabs; a second call of the
    same shape allocates nothing and gives the same answer up to the order of the float atomics.  K = 10 runs the
    KP = 32 plan, K = 40 the KP = 64 one."""
    from oracle import zloop
    from oriana_b200 import _lib
    n, p = 2900, 1500
    rng = np.random.default_rng(5)
    lU = rng.normal(-0.5, 1.0, (n, K)).astype(np.float32)
    lV = rng.normal(-0.5, 1.0, (p, K)).astype(np.float32)
    X = (rng.poisson(3.0, (n, p)) * (rng.random((n, p)) < 0.6)).astype(np.float32)
    D = np.where(X != 0, 1.0, rng.random((n, p))).astype(np.float32)
    ctx = ctypes.c_void_p()
    _lib.check(cuda_lib.ori_ctx_create(ctypes.byref(ctx), 1408))          # 1408 x 1500 = 2.1e6 entries per slab
    try:
        outs = []
        for rep in range(2):
            Zi = np.full((n, K), np.nan, np.float32); Zj = np.full((p, K), np.nan, np.float32)
            Z3 = np.full((p, K), np.nan, np.float32)
            _lib.check(cuda_lib.ori_zigap_compute_Z_q_expectations_ctx(ctx, _ptr(Zi), _ptr(Zj), _ptr(Z3), _ptr(lU), _ptr(lV),
                                                                       _ptr(D), _ptr(X), n, p, K, int(quirk)))
            outs.append((Zi, Zj, Z3))
            st = _stats(cuda_lib, ctx)
            if rep == 0:
                first = st
        assert first['tensor_slabs'] == 3 and first['simt_slabs'] == 0 and first['allocs'] > 0
        assert st['allocs'] == first['allocs'] and st['calls'] == 2 and st['tensor_slabs'] == 6   # nothing allocated again
        rZi, rZj, rZ3 = zloop.zigap_z(lU, lV, D, X, quirk=quirk, third=True)
        Zi, Zj, Z3 = outs[1]
        assert relerr(Zi, rZi) < 1e-3 and relerr(Zj, rZj) < 1e-3, (relerr(Zi, rZi), relerr(Zj, rZj))
        assert np.max(np.abs(Z3 - rZ3)) < 1e-3 * np.max(np.abs(rZ3))
        for a, b in zip(outs[0][:2], outs[1][:2]):
            assert relerr(a, b) < 1e-5
        assert np.max(np.abs(outs[0][2] - outs[1][2])) < 1e-5 * np.max(np.abs(outs[1][2]))     # signed terms cancel (zigap.py:95)
        gZi = np.full((n, K), np.nan, np.float32); gZj = np.full((p, K), np.nan, np.float32)
        _lib.check(cuda_lib.ori_gap_compute_Z_q_expectations_ctx(ctx, _ptr(gZi), _ptr(gZj), _ptr(lU), _ptr(lV), _ptr(X), n, p, K))
        rZi, rZj = zloop.gap_z(lU, lV, X)
        assert relerr(gZi, rZi) < 1e-3 and relerr(gZj, rZj) < 1e-3
        assert _stats(cuda_lib, ctx)['allocs'] == first['allocs']                  # GaP needs a subset of the buffers
    finally:
        _lib.check(cuda_lib.ori_ctx_destroy(ctx))


def test_default_context_allocates_once(cuda_lib):
    """The *_host entry points (what INTEGRATION.md binds) keep one process-wide context: repeated calls of a shape no
    larger than any before allocate no device memory and create no streams."""
    rng = np.random.default_rng(1)
    n, p, K = 300, 200, 5
    lU = rng.normal(-0.5, 1.0, (n, K)).astype(np.float32); lV = rng.normal(-0.5, 1.0, (p, K)).astype(np.float32)
    X = rng.poisson(2.0, (n, p)).astype(np.float32)
    z_op(cuda_lib, lU, lV, X)
    a0 = _stats(cuda_lib)
    for _ in range(3):
        z_op(cuda_lib, lU, lV, X)
    a1 = _stats(cuda_lib)
    assert a1['allocs'] == a0['allocs'] and a1['calls'] == a0['calls'] + 3


def _underflow_case(n, p, K, seed):
    """A third of the cells and of the genes live 70 below the rest: the reference's float32 exp(lU + lV) is 0 for every
    component where both meet (-140), a normal number everywhere else (>= e^-80); no entry sits in the denormal band, where
    the reference's own ratios are imprecise."""
    rng = np.random.default_rng(seed)
    lU = rng.uniform(-3., 2., (n, K)); lV = rng.uniform(-3., 2., (p, K))
    low_i = rng.random(n) < 0.33; low_j = rng.random(p) < 0.33
    lU[low_i] -= 70.; lV[low_j] -= 70.
    lU[rng.random((n, K)) < 0.05] = -1e15                       # exact zeros of NMF factors (psi of a clamped 1e-15)
    X = (rng.poisson(3.0, (n, p)) * (rng.random((n, p)) < 0.6)).astype(np.float32)
    D = np.where(X != 0, 1.0, rng.random((n, p))).astype(np.float32)
    return lU.astype(np.float32), lV.astype(np.float32), X, D, low_i, low_j


@pytest.mark.parametrize('quirk', [True, False])
@pytest.mark.parametrize('shape,tol', [((300, 260, 5), 1e-5), ((150, 90, 40), 1e-5), ((2048, 1024, 12), 2e-3)])
def test_float32_underflow_of_the_reference_is_reproduced(cuda_lib, shape, tol, quirk):
    """zigap.py:86-90 / gap.py:73-76 on both kernel families (the third shape takes the tcgen05 passes): counts of entries
    whose every term underflows in the reference go to no component; everything else keeps its ratios."""
    from oracle import zloop
    n, p, K = shape
    lU, lV, X, D, low_i, low_j = _underflow_case(n, p, K, seed=n + p + K)
    rZi, rZj, rZ3 = zloop.zigap_z(lU, lV, D, X, quirk=quirk, third=True)
    # the case does what it says: the reference drops the counts of (low cell, low gene) pairs
    XD = X * D
    kept = XD[np.ix_(low_i, ~low_j)].sum(1)
    np.testing.assert_allclose(rZi[low_i].sum(1), kept, rtol=1e-4, atol=1e-3)
    assert XD[np.ix_(low_i, low_j)].sum() > 0
    Zi, Zj, Z3 = z_op(cuda_lib, lU, lV, X, D, quirk=quirk, third=True)
    assert relerr(Zi, rZi) < tol, relerr(Zi, rZi)
    assert relerr(Zj, rZj) < tol, relerr(Zj, rZj)
    assert np.max(np.abs(Z3 - rZ3)) < max(tol, 3e-6) * np.max(np.abs(rZ3))
    np.testing.assert_allclose(Zi[low_i].sum(1), kept, rtol=10 * tol, atol=1e-3)
    gZi, gZj = z_op(cuda_lib, lU, lV, X)
    rZi, rZj = zloop.gap_z(lU, lV, X)
    assert relerr(gZi, rZi) < tol and relerr(gZj, rZj) < tol
