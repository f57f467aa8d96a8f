"""GPU: the sparse model's operator seam -- `ori_sparse_zigap_compute_Z_q_expectations_{host,ctx}` in place of
`SparseZIGaP.compute_Z_q_expectations` (sparse_zigap.py:100-116) -- against

  * the reference kernel's recorded outputs (`sparse_k4`, `sparse_ragged`: z_* arrays of oracle/make_golden.py),
  * the sequential float32 C loop (oracle/zloop.c `zl_sparse_z`, pinned by tests/test_oracle_sparse.py),
  * the reference's recorded trajectories, with the INTEGRATION.md section 1 stub inside the oracle's sparse step,
  * and, where `__graft_entry__.build()` installed it under oracle/_ref, the live reference stepped on its own numba kernel.

Tolerances: the CUDA-core kernels 1e-5 relative for DSZ_hat / DZ_hat; DZ_exp_logsum_hat is a sum of signed terms that
cancel (sparse_zigap.py:116), so its absolute error is judged against the array's scale: 3e-6 * max.  Slabs of >= 2^21
entries with K <= 32 run the tcgen05 passes in the fp32-grade mode (ORI_F_PRECISE): 1e-5 / 1e-5 * max (about 3x the
largest error measured on a B200).  Trajectories: the tolerances tests/test_sparse_gpu.py holds the device model to.
"""
import copy
import ctypes
import os
import warnings

import numpy as np
import pytest

from conftest import golden_state, load_golden, relerr

pytestmark = pytest.mark.gpu

TC_TOL = 1e-5          # fp32-grade tcgen05 passes against the sequential float32 loop (3.5e-6 measured)
KEYS = ('a1', 'a2', 'b1', 'b2', 'p_s', 'pi_s', 'pi_d', 'alpha1', 'alpha2', 'beta1', 'beta2')
OUTS = ('DSZ_hat', 'DZ_hat', 'DZ_exp_logsum_hat')


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def sparse_op(lib, lU, lV, St, Sh, D, X, ctx=None, null=()):
    """One call with C-contiguous float32 copies of the inputs; `null` names arguments passed as NULL."""
    from oriana_b200 import _lib
    n, K = lU.shape
    p = lV.shape[0]
    outs = [np.full((n, K), np.nan, np.float32), np.full((p, K), np.nan, np.float32), np.full((p, K), np.nan, np.float32)]
    ins = dict(zip(('lU', 'lV', 'St', 'Sh', 'D', 'X'),
                   (np.ascontiguousarray(a, dtype=np.float32) for a in (lU, lV, St, Sh, D, X))))
    args = [None if k in null else _ptr(a) for k, a in list(zip(OUTS, outs)) + list(ins.items())] + [n, p, K]
    if ctx is None:
        rc = lib.ori_sparse_zigap_compute_Z_q_expectations_host(*args)
    else:
        rc = lib.ori_sparse_zigap_compute_Z_q_expectations_ctx(ctx, *args)
    _lib.check(rc)
    return tuple(outs)


def _errors(got, want):
    """(relerr DSZ, relerr DZ, max|dDZl| / max|DZl|)."""
    scale = max(float(np.max(np.abs(want[2]))), 1e-30)
    return relerr(got[0], want[0]), relerr(got[1], want[1]), float(np.max(np.abs(got[2] - want[2]))) / scale


def _assert_close(got, want, tol, tol3, what):
    e = _errors(got, want)
    print('%s: DSZ %.2e DZ %.2e DZl %.2e (bounds %.0e / %.0e)' % (what, e[0], e[1], e[2], tol, tol3))
    assert e[0] <= tol and e[1] <= tol and e[2] <= tol3, (what, e)


def _stats(lib, ctx=None):
    from oriana_b200 import _lib
    c = [ctypes.c_uint64(0) for _ in range(4)]
    _lib.check(lib.ori_ctx_stats(ctx, *[ctypes.byref(x) for x in c]))
    return dict(zip(('calls', 'allocs', 'tensor_slabs', 'simt_slabs'), (int(x.value) for x in c)))


def _problem(n, p, K, seed):
    """D_hat soft on the zeros, S_hat soft in (0, 1), S_tilde with about 30 % zeros, plus one gene with every component
    masked and (K >= 2) one component masked for every gene."""
    rng = np.random.default_rng(seed)
    lU = rng.normal(-0.5, 1.0, (n, K)).astype(np.float32)
    lV = rng.normal(-0.5, 1.0, (p, K)).astype(np.float32)
    X = (rng.poisson(3.0, (n, p)) * (rng.random((n, p)) < 0.6)).astype(np.float32)
    D = np.where(X != 0, 1.0, rng.random((n, p))).astype(np.float32)
    Sh = rng.uniform(0.02, 0.98, (p, K)).astype(np.float32)
    St = (rng.random((p, K)) >= 0.3).astype(np.float32)
    dead_j = p // 2
    St[dead_j] = 0.
    dead_k = K // 2 if K >= 2 else None
    if dead_k is not None:
        St[:, dead_k] = 0.
    return (lU, lV, St, Sh, D, X), dead_j, dead_k


@pytest.mark.parametrize('name', ['sparse_k4', 'sparse_ragged'])
def test_against_reference_numba_kernel(cuda_lib, name):
    g = load_golden(name)
    D = g['s0_p_d'].astype(np.float32)
    got = sparse_op(cuda_lib, g['z_log_U_hat'], g['z_log_Vp_hat'], g['z_S_tilde'], g['z_S_hat'], D, g['X'])
    _assert_close(got, (g['z_DSZ'], g['z_DZ'], g['z_DZl']), 1e-5, 3e-6, name)


@pytest.mark.parametrize('shape', [(1, 3, 1), (5, 7, 3), (129, 33, 8), (260, 517, 9), (300, 140, 17), (70, 90, 40),
                                   (129, 77, 64)])
def test_against_c_loop_with_masks(cuda_lib, shape):
    """Ragged shapes and every padded-K bucket on the CUDA-core kernels; masked genes and components receive nothing."""
    from oracle import zloop
    n, p, K = shape
    args, dead_j, dead_k = _problem(n, p, K, seed=n * 1000 + p + K)
    got = sparse_op(cuda_lib, *args)
    _assert_close(got, zloop.sparse_z(*args), 1e-5, 3e-6, 'c loop %s' % (shape,))
    DSZ, DZ, DZl = got
    assert not DZ[dead_j].any() and not DZl[dead_j].any()          # its counts go nowhere
    if dead_k is not None:
        assert not DSZ[:, dead_k].any() and not DZ[:, dead_k].any() and not DZl[:, dead_k].any()
    # every count of a gene with an unmasked component lands on some component (no term underflows here)
    XD = (args[5] * args[4]).sum(0)
    live = args[2].any(1)
    np.testing.assert_allclose(DZ.sum(1)[live], XD[live], rtol=1e-5, atol=1e-4)


def _zigap_call(lib, ctx, lU, lV, D, X):
    from oriana_b200 import _lib
    n, K = lU.shape
    p = lV.shape[0]
    Zi = np.empty((n, K), np.float32); Zj = np.empty((p, K), np.float32); Z3 = np.empty((p, K), np.float32)
    _lib.check(lib.ori_zigap_compute_Z_q_expectations_ctx(ctx, _ptr(Zi), _ptr(Zj), _ptr(Z3), _ptr(lU), _ptr(lV), _ptr(D),
                                                          _ptr(X), n, p, K, 1))


@pytest.mark.parametrize('K', [10, 32])
def test_tensor_sized_slabs_take_the_fp32_grade_tcgen05_passes(cuda_lib, K):
    """Three ragged slabs of >= 2^21 entries through an explicit context run the tcgen05 passes; a second call of the same
    shape allocates nothing and agrees with the first up to the order of the float atomics; ZIGaP calls on the same
    context, before and after, allocate nothing for the sparse calls' sake."""
    from oracle import zloop
    from oriana_b200 import _lib
    n, p = 2900, 1500
    args, dead_j, dead_k = _problem(n, p, K, seed=K)
    lU, lV, St, Sh, D, X = args
    ctx = ctypes.c_void_p()
    _lib.check(cuda_lib.ori_ctx_create(ctypes.byref(ctx), 1408))          # 1408 x 1500 = 2.1e6 entries per slab
    try:
        _zigap_call(cuda_lib, ctx, lU, lV, D, X)
        s0 = _stats(cuda_lib, ctx)
        outs, st = [], []
        for rep in range(2):
            outs.append(sparse_op(cuda_lib, *args, ctx=ctx))
            st.append(_stats(cuda_lib, ctx))
        assert st[0]['tensor_slabs'] - s0['tensor_slabs'] == 3 and st[0]['simt_slabs'] == s0['simt_slabs'] == 0
        assert st[1]['tensor_slabs'] - st[0]['tensor_slabs'] == 3 and st[1]['simt_slabs'] == 0
        assert st[1]['allocs'] == st[0]['allocs'] and st[1]['calls'] == s0['calls'] + 2
        _zigap_call(cuda_lib, ctx, lU, lV, D, X)
        assert _stats(cuda_lib, ctx)['allocs'] == st[1]['allocs']
        _assert_close(outs[1], zloop.sparse_z(*args), TC_TOL, TC_TOL, 'tensor K=%d' % K)
        _assert_close(outs[0], outs[1], 1e-5, 1e-5, 'tensor K=%d repeat' % K)
        assert not outs[1][1][dead_j].any() and not outs[1][1][:, dead_k].any()
    finally:
        _lib.check(cuda_lib.ori_ctx_destroy(ctx))


def test_tensor_sized_slabs_above_k32_run_the_cuda_core_kernels(cuda_lib):
    """The sparse model's plan: 32 < K <= 64 runs the CUDA-core kernels whatever the slab size."""
    from oracle import zloop
    from oriana_b200 import _lib
    args, _, _ = _problem(2900, 1500, 40, seed=40)
    ctx = ctypes.c_void_p()
    _lib.check(cuda_lib.ori_ctx_create(ctypes.byref(ctx), 1408))
    try:
        got = sparse_op(cuda_lib, *args, ctx=ctx)
        st = _stats(cuda_lib, ctx)
        assert st['tensor_slabs'] == 0 and st['simt_slabs'] == 3
    finally:
        _lib.check(cuda_lib.ori_ctx_destroy(ctx))
    _assert_close(got, zloop.sparse_z(*args), 1e-5, 3e-6, 'cuda-core 2900 x 1500 K=40')


def _underflow_case(n, p, K, seed):
    """test_z_operator_gpu._underflow_case with the sparse model's masks: a third of the cells and of the genes live 70
    below the rest, so the reference's float32 exp(lU + lV) is 0 for every component where both meet (-140) and a normal
    number everywhere else (>= e^-80); 5 % of the cell factors are exact zeros; S_tilde has about 30 % zeros."""
    rng = np.random.default_rng(seed)
    lU = rng.uniform(-3., 2., (n, K)); lV = rng.uniform(-3., 2., (p, K))
    low_i = rng.random(n) < 0.33; low_j = rng.random(p) < 0.33
    lU[low_i] -= 70.; lV[low_j] -= 70.
    lU[rng.random((n, K)) < 0.05] = -1e15
    X = (rng.poisson(3.0, (n, p)) * (rng.random((n, p)) < 0.6)).astype(np.float32)
    D = np.where(X != 0, 1.0, rng.random((n, p))).astype(np.float32)
    Sh = rng.uniform(0.02, 0.98, (p, K)).astype(np.float32)
    St = (rng.random((p, K)) >= 0.3).astype(np.float32)
    return (lU.astype(np.float32), lV.astype(np.float32), St, Sh, D, X), low_i, low_j


@pytest.mark.parametrize('shape,tensor', [((300, 260, 5), False), ((150, 90, 40), False), ((2048, 1024, 12), True)])
def test_float32_underflow_of_the_reference_is_reproduced(cuda_lib, shape, tensor):
    """sparse_zigap.py:109-111 on both kernel families (the third shape is one tensor slab): counts of entries whose every
    unmasked term underflows in the reference go to no component; everything else keeps its ratios."""
    from oracle import zloop
    n, p, K = shape
    args, low_i, low_j = _underflow_case(n, p, K, seed=n + p + K)
    lU, lV, St, Sh, D, X = args
    want = zloop.sparse_z(*args)
    # the counts a low gene keeps: those of the cells where some unmasked term survives the float32 exp
    with np.errstate(under='ignore', over='ignore'):
        terms = np.exp(lU[:, None, :] + lV[None, low_j, :]) * St[None, low_j, :]
    alive = terms.sum(-1) > 0
    assert not alive[low_i].any()
    XD = (X * D)[:, low_j]
    kept = (XD * alive).sum(0)
    assert XD[low_i].sum() > 0                                          # the case does what it says
    np.testing.assert_allclose(want[1][low_j].sum(1), kept, rtol=1e-4, atol=1e-3)
    before = _stats(cuda_lib)
    got = sparse_op(cuda_lib, *args)
    after = _stats(cuda_lib)
    assert (after['tensor_slabs'] - before['tensor_slabs'], after['simt_slabs'] - before['simt_slabs']) == \
        ((1, 0) if tensor else (0, 1))
    tol = TC_TOL if tensor else 1e-5
    _assert_close(got, want, tol, max(tol, 3e-6), 'underflow %s' % (shape,))
    np.testing.assert_allclose(got[1][low_j].sum(1), kept, rtol=10 * tol, atol=1e-3)


def test_empty_and_bad_arguments(cuda_lib):
    from oriana_b200 import _lib
    K, p = 3, 5
    z = lambda *s: np.zeros(s, np.float32)
    DSZ, DZ, DZl = sparse_op(cuda_lib, z(0, K), z(p, K), z(p, K), z(p, K), z(0, p), z(0, p))
    assert DSZ.shape == (0, K) and not DZ.any() and not DZl.any()          # n = 0: zero gene sums
    args = (z(2, K), z(p, K), np.ones((p, K), np.float32), z(p, K), np.ones((2, p), np.float32), np.ones((2, p), np.float32))
    for null in ('D', 'DZ_exp_logsum_hat', 'St', 'Sh'):
        with pytest.raises(_lib.OrianaB200Error):
            sparse_op(cuda_lib, *args, null=(null,))
    with pytest.raises(_lib.OrianaB200Error, match='error -4'):              # ORI_EUNSUPPORTED
        sparse_op(cuda_lib, z(2, 65), z(p, 65), z(p, 65), z(p, 65), z(2, p), z(2, p))
    sparse_op(cuda_lib, *args)                                              # the same arguments pass


def _stub(lib):
    """The ctypes stub of INTEGRATION.md section 1 for SparseZIGaP.compute_Z_q_expectations, on the loaded library; counts
    its calls and the layouts of X it was handed."""
    fp = ctypes.c_void_p
    keep, seen = [], {'calls': 0, 'x_not_c': 0}

    def ptr(a):
        if a.dtype != np.float32 or a.ndim != 2:                   # the numba signature f4[:, :] raises TypeError too
            raise TypeError('2-D float32 array expected (sparse_zigap.py:100)')
        if not a.flags.c_contiguous:
            a = np.ascontiguousarray(a)
            keep.append(a)
        return fp(a.ctypes.data)

    def sparse_zigap_z(DSZ_hat, DZ_hat, DZ_exp_logsum_hat, log_U_hat, log_V_hat, S_tilde, S_hat, D_hat, X):
        n, p = X.shape
        K = log_U_hat.shape[1]
        seen['calls'] += 1
        seen['x_not_c'] += int(not X.flags.c_contiguous)
        rc = lib.ori_sparse_zigap_compute_Z_q_expectations_host(
            ptr(DSZ_hat), ptr(DZ_hat), ptr(DZ_exp_logsum_hat), ptr(log_U_hat), ptr(log_V_hat), ptr(S_tilde), ptr(S_hat),
            ptr(D_hat), ptr(X), n, p, K)
        keep.clear()
        if rc:
            buf = ctypes.create_string_buffer(512)
            lib.ori_last_error(buf, 512)
            raise RuntimeError(buf.value.decode())
    return sparse_zigap_z, seen


def _tol(name, t):
    return (2e-4 if name == 'sparse_nmf' else 2e-5) if t == 1 else (1.5e-2 if name == 'sparse_nmf' else 5e-3)


@pytest.mark.parametrize('name', ['sparse_k4', 'sparse_ragged', 'sparse_gen', 'sparse_nmf'])
def test_reference_step_with_the_sparse_operator(cuda_lib, monkeypatch, name):
    """oracle/sparse_numpy.step with its Z step replaced by the stub, called the way the reference calls its kernel
    (np.empty outputs, X as a column-major float32 copy, sparse_zigap.py:126-135), against the recorded trajectories."""
    from oracle import sparse_numpy as sn
    stub, seen = _stub(cuda_lib)

    def device_z(log_U_hat, log_Vp_hat, S_tilde, S_hat, D_hat, X, dtype=np.float32):
        n, K = log_U_hat.shape
        p = log_Vp_hat.shape[0]
        outs = np.empty((n, K), np.float32), np.empty((p, K), np.float32), np.empty((p, K), np.float32)
        stub(*outs, log_U_hat, log_Vp_hat, S_tilde, S_hat, D_hat, np.asfortranarray(X, dtype=np.float32))
        return outs

    monkeypatch.setattr(sn, 'z_expectations', device_z)
    g = load_golden(name)
    s = golden_state(g, 0)
    for k in ('deviance', 'explained'):
        s.pop(k, None)
    steps = [int(t) for t in g['steps']]
    worst = {}
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        for t in range(1, max(steps) + 1):
            sn.step(s, tau=float(g['tau']))
            if t not in steps:
                continue
            want = golden_state(g, t)
            for k in KEYS:
                e = relerr(s[k], want[k])
                worst[(t == 1, k)] = max(worst.get((t == 1, k), 0.), e)
                assert e < _tol(name, t), (name, t, k, e)
            assert np.max(np.abs(s['p_d'].astype(np.float32) - want['p_d'])) < (1e-5 if t == 1 else 2e-3), (name, t)
            dev_ref, expl_ref = float(want['deviance']), float(want['explained'])
            if abs(dev_ref) < 1e15:        # beyond: a -inf entry was cast to INT64_MIN (quirk Q10), meaningless
                assert abs(sn.reconstruction_deviance(s) - dev_ref) <= 1e-4 * abs(dev_ref), (name, t)
                assert abs(sn.explained_deviance(s) - expl_ref) <= 1e-4 * abs(expl_ref), (name, t)
    assert seen['calls'] == max(steps) and seen['x_not_c'] == seen['calls']
    print('%s: largest relerr after step 1 %.2e (bound %.0e), later %.2e (bound %.0e)' % (
        name, max(v for (f, _), v in worst.items() if f), _tol(name, 1),
        max((v for (f, _), v in worst.items() if not f), default=0.), _tol(name, 2)))


def test_live_reference_sparse_zigap_with_the_stub(cuda_lib, monkeypatch):
    """One reference SparseZIGaP, deep-copied: one copy steps on the reference's numba kernel, the other with the stub
    patched onto the class (the reference's own X, column-major, sparse_zigap.py:135), 5 steps each."""
    from oracle import cavi_numpy as cn, refshim
    if not os.path.isdir(os.path.join(refshim.INSTALLED, 'oriana', 'models')):
        pytest.skip('the reference is not installed under oracle/_ref')
    pytest.importorskip('numba')
    stub, seen = _stub(cuda_lib)
    X = cn.synth_counts(180, 240, 5, seed=21)
    try:
        refshim.import_reference()
        from oriana.models import SparseZIGaP
        from oriana.singlecell import CountMatrix
        keys = KEYS
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            np.random.seed(3)
            m = SparseZIGaP(CountMatrix(X), k=5, use_factors=False, tau=0.5)
            ref, dev = copy.deepcopy(m), copy.deepcopy(m)
            want = []
            for _ in range(5):
                ref.step()
                want.append({k: np.array(getattr(ref, k)[:], np.float64) for k in keys} | {'D_hat': ref.D_hat.copy()})
            monkeypatch.setattr(SparseZIGaP, 'compute_Z_q_expectations', staticmethod(stub))
            for t in range(1, 6):
                dev.step()
                for k in keys:
                    e = relerr(np.asarray(getattr(dev, k)[:], np.float64), want[t - 1][k])
                    assert e < (2e-5 if t == 1 else 5e-3), (t, k, e)
                assert np.max(np.abs(dev.D_hat - want[t - 1]['D_hat'])) < (1e-5 if t == 1 else 2e-3), t
            monkeypatch.undo()
            d_ref, d_dev = ref.reconstruction_deviance(), dev.reconstruction_deviance()
            if abs(d_ref) < 1e15:
                assert abs(d_dev - d_ref) <= 1e-4 * abs(d_ref)
    finally:
        monkeypatch.undo()
        refshim.release_reference()
    assert seen['calls'] == 5 and seen['x_not_c'] == 5
