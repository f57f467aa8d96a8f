"""GPU: scipy.sparse count matrices through every layer -- the CSR expansion kernel, CountMatrix.to_device, the three
models, and CsrCounts in the host-streamed step.

A CSR ingest writes the same bits into HBM as the dense ingest, so a model built from a CSR and one built from the dense
array, both from the same state with deterministic=True, agree in every bit of every parameter.  The ELBO trace carries
sum lgamma(X + 1), a constant formed once per model with float64 atomics, hence the 1e-13 there (as in
test_u16_counts_gpu.py)."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import golden_state, load_golden, relerr

pytestmark = pytest.mark.gpu
PARAMS = ('a1', 'a2', 'b1', 'b2', 'alpha1', 'alpha2', 'beta1', 'beta2')
U8, U16, F32 = 1, 2, 4


def _stream():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _sparse_counts(n, p, density, vtype, seed):
    rng = np.random.default_rng(seed)
    top = {U8: 255, U16: 65535, F32: 1e6}[vtype]
    X = (rng.integers(1, 40, size=(n, p)) * (rng.random((n, p)) < density)).astype(np.float64)
    if density > 0:
        X[n // 2] = 0                                            # an empty row
        X[0, p - 1] = top
        if vtype == F32:
            X[n - 1, 0] = 2.5
    return X


@pytest.mark.parametrize('dst_bytes', [4, 2])
@pytest.mark.parametrize('vtype', [U8, U16, F32])
@pytest.mark.parametrize('idx_bytes', [2, 4])
def test_expand_csr_kernel_is_exact(cuda_lib, idx_bytes, vtype, dst_bytes):
    """Every element of a sentinel-filled destination is written: counts, zeros, pad columns; slabs from row 0 and from the
    middle of the stream (base != 0)."""
    import torch
    vdt = {U8: np.uint8, U16: np.uint16, F32: np.float32}[vtype]
    shapes = [(7, 13), (33, 130), (3, 1), (4, 40000), (300, 977)] + ([(5, 70000)] if idx_bytes == 4 else [])
    for si, (n, p) in enumerate(shapes):
        for density in (0., 0.05, 1.):
            X = _sparse_counts(n, p, density, vtype, seed=si)
            csr = sp.csr_matrix(X)
            ind = torch.from_numpy(csr.indices.astype(np.uint16 if idx_bytes == 2 else np.int32).view(
                np.int16 if idx_bytes == 2 else np.int32)).cuda()
            val = torch.from_numpy(csr.data.astype(vdt).view(np.int16) if vdt == np.uint16 else csr.data.astype(vdt)).cuda()
            ptr = torch.from_numpy(csr.indptr.astype(np.int64)).cuda()
            q = 16 // dst_bytes
            ldd = (p + q - 1) // q * q
            if dst_bytes == 4:
                dst = torch.full((n, ldd), -7.5, dtype=torch.float32, device='cuda')
                want = np.zeros((n, ldd), dtype=np.float32)
                want[:, :p] = X.astype(np.float32)
            else:
                dst = torch.full((n, ldd), -21555, dtype=torch.int16, device='cuda')
                want = np.zeros((n, ldd), dtype=np.uint16)
                want[:, :p] = X.astype(np.uint16)
            for r0 in (0, n // 3):
                lo = int(csr.indptr[r0])
                rc = cuda_lib.ori_expand_csr_counts(ptr[r0:].data_ptr(), lo, ind[lo:].data_ptr() if ind.numel() else None,
                                                    idx_bytes, val[lo:].data_ptr() if val.numel() else None, vtype,
                                                    dst[r0:].data_ptr(), dst_bytes, ldd, n - r0, p, _stream())
                if vtype == F32 and dst_bytes == 2:
                    assert rc == -1                                # float counts into uint16 storage: ORI_EINVAL
                    break
                assert rc == 0
                got = dst.cpu().numpy()
                if dst_bytes == 2:
                    got = got.view(np.uint16)
                assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), (n, p, density, r0)
    # argument checks: ldd not a multiple of the 16-byte pitch, a misaligned destination, an unknown index width
    d = torch.zeros((2, 16), dtype=torch.float32, device='cuda')
    p64 = torch.zeros((3,), dtype=torch.int64, device='cuda')
    assert cuda_lib.ori_expand_csr_counts(p64.data_ptr(), 0, None, 2, None, U8, d.data_ptr(), 4, 6, 2, 5, _stream()) == -1
    assert cuda_lib.ori_expand_csr_counts(p64.data_ptr(), 0, None, 2, None, U8, d.data_ptr() + 4, 4, 8, 1, 5, _stream()) == -1
    assert cuda_lib.ori_expand_csr_counts(p64.data_ptr(), 0, None, 3, None, U8, d.data_ptr(), 4, 8, 2, 5, _stream()) == -1
    assert cuda_lib.ori_expand_csr_counts(p64.data_ptr(), 0, None, 2, None, U8, d.data_ptr(), 4, 8, 2, 5, _stream()) == 0
    assert not d.any()


def _padded(t):
    """The whole [n, ldx] buffer behind a [n, p] view of it."""
    import torch
    return torch.as_strided(t, (t.shape[0], t.stride(0)), (t.stride(0), 1))


@pytest.mark.parametrize('kind', ['u8', 'u16', 'int64_big', 'float', 'wide'])
def test_count_matrix_to_device_csr_equals_dense(cuda_lib, kind):
    import torch
    from oriana.singlecell import CountMatrix
    rng = np.random.default_rng(4)
    n, p = (20, 70001) if kind == 'wide' else (301, 77)
    X = rng.poisson(2., size=(n, p)) * (rng.random((n, p)) < 0.1)
    X[n // 2] = 0
    X = {'u8': X.astype(np.int64), 'u16': X.astype(np.uint16), 'int64_big': X.astype(np.int64),
         'float': X.astype(np.float64), 'wide': X.astype(np.int32)}[kind]
    if kind == 'u16':
        X[3, 4] = 65535
    if kind == 'int64_big':
        X[3, 4] = 70000
    if kind == 'float':
        X[3, 4] = 2.75
    dense, csr = CountMatrix(X), CountMatrix(sp.csc_matrix(X))
    assert dense.narrow_dtype() == csr.narrow_dtype()
    dtypes = [torch.float32] + ([torch.uint16] if kind == 'u16' else [])
    for dt in dtypes:
        want = _padded(dense.to_device('cuda', dtype=dt))
        view = dense.to_device('cuda', dtype=dt)
        for got in (csr.to_device('cuda', dtype=dt), csr.to_device('cuda', dtype=dt, slab_rows=7),
                    csr._csr_to_device(torch.device('cuda'), 4 if dt == torch.float32 else 2, None, slab_nnz=50)):
            assert got.dtype == view.dtype and got.shape == view.shape and got.stride() == view.stride()
            g, w = _padded(got), want
            if dt == torch.uint16:
                g, w = g.view(torch.int16), w.view(torch.int16)
            assert torch.equal(g, w)
    if kind != 'u16':
        with pytest.raises(TypeError):
            csr.to_device('cuda', dtype=torch.uint16)


@pytest.fixture
def uint16_storage(monkeypatch):
    """Keep every uint16 input as uint16 in HBM, at any size."""
    import torch
    from oriana_b200 import problem
    monkeypatch.setattr(problem, 'counts_storage', lambda u16, *args: torch.uint16 if u16 else torch.float32)


def _model_pair(model, X, K, **kw):
    """(dense model, CSR model, bare-CSR model) of the same counts from the same state, stepped 3 times."""
    from oracle import cavi_numpy as cn
    from oriana.models import GaP, SparseZIGaP, ZIGaP
    from oriana.singlecell import CountMatrix
    cls = dict(zigap=ZIGaP, gap=GaP, sparse=SparseZIGaP)[model]
    out = []
    for src in (CountMatrix(X), CountMatrix(sp.csr_matrix(X)), sp.coo_matrix(X)):
        if model == 'sparse':                                    # the constructor's own draws, from the same seed
            np.random.seed(5)
            m = cls(src, k=K, use_factors=False, deterministic=True, **kw)
        else:
            s = cn.init_state(X.astype(np.float64), K, np.random.default_rng(1), model)
            m = cls(src, k=K, use_factors=False, state=s, deterministic=True, **kw)
        for _ in range(3):
            m.step()
        out.append(m)
    return out


def _assert_identical(a, b):
    names = PARAMS + (('pi_d',) if hasattr(a, 'pi_d') else ())
    for k in names:
        x, y = getattr(a, k).asarray(), getattr(b, k).asarray()
        assert np.array_equal(x, y), (k, float(np.max(np.abs(x - y))))
    assert np.array_equal(a.U_hat, b.U_hat) and np.array_equal(a.V_hat, b.V_hat)
    if a._flags & 4:                                             # ORI_F_ELBO
        np.testing.assert_allclose(b.elbo_trace, a.elbo_trace, rtol=1e-13)
    if hasattr(a, 'reconstruction_deviance'):
        assert np.array_equal(a.p_s.asarray(), b.p_s.asarray())
        assert a.reconstruction_deviance() == b.reconstruction_deviance()
        assert a.explained_deviance() == b.explained_deviance()


MODEL_CASES = {
    'gap_cuda_core': ('gap', (300, 211, 6)),
    'zigap_cuda_core': ('zigap', (300, 211, 6)),
    'sparse_cuda_core': ('sparse', (300, 211, 6)),
    'gap_tensor': ('gap', (2100, 1003, 12)),                     # >= 2^21 entries: the tcgen05 passes
    'zigap_tensor': ('zigap', (2100, 1003, 12)),
    'sparse_tensor': ('sparse', (2100, 1003, 12)),
}


@pytest.mark.parametrize('storage', ['float32', 'uint16'])
@pytest.mark.parametrize('case', sorted(MODEL_CASES))
def test_model_from_csr_is_bit_identical_to_dense(cuda_lib, request, case, storage):
    import torch
    from oracle import cavi_numpy as cn
    model, (n, p, K) = MODEL_CASES[case]
    X = cn.synth_counts(n, p, K, seed=n % 97)
    X[n // 3] = 0
    X[:, p // 2] = 0
    X[1, 2] = 300
    if storage == 'uint16':
        request.getfixturevalue('uint16_storage')
        X = X.astype(np.uint16)
    models = _model_pair(model, X, K)
    for m in models:
        assert m.counts_dtype == (torch.uint16 if storage == 'uint16' else torch.float32)
        assert m.uses_tensor_path == (n * p >= 1 << 21)
    for m in models[1:]:
        assert m.cmatrix.is_sparse
        _assert_identical(models[0], m)


def test_model_from_csr_host_nmf_gap_loglik_and_p_d(cuda_lib):
    """The host NMF warm start factorises the same dense array; GaP's integer_samples follows the CSR's dtype; a fresh
    model's p_d indicator is checked against the CSR's zero pattern."""
    from oracle import cavi_numpy as cn
    from oriana.models import GaP, ZIGaP
    from oriana.singlecell import CountMatrix
    n, p, K = 200, 150, 4
    X = cn.synth_counts(n, p, K, seed=3).astype(np.int64)
    models = []
    for src in (X, sp.csr_matrix(X)):
        np.random.seed(11)
        m = ZIGaP(CountMatrix(src), k=K, use_factors=True, nmf='host', deterministic=True)
        m.step()
        models.append(m)
    assert np.array_equal(models[0]._nmf_U, models[1]._nmf_U) and np.array_equal(models[0]._nmf_V, models[1]._nmf_V)
    _assert_identical(*models)
    for dt, integer in ((np.int64, True), (np.float32, False)):
        s = cn.init_state(X.astype(np.float64), K, np.random.default_rng(1), 'gap')
        gd = GaP(CountMatrix(X.astype(dt)), k=K, use_factors=False, state=s)
        gs = GaP(CountMatrix(sp.csr_matrix(X.astype(dt))), k=K, use_factors=False, state=s)
        assert gs.X.integer_samples == gd.X.integer_samples == integer
        ls, ld = gs.loglikelihood(), gd.loglikelihood()
        assert abs(ls - ld) <= 1e-12 * abs(ld), (ls, ld)
    s = cn.init_state(X.astype(np.float64), K, np.random.default_rng(1), 'zigap')
    s['p_d'] = (X > 0).astype(np.float64)
    S = sp.csr_matrix(X)
    ZIGaP(S, k=K, use_factors=False, state=s)
    bad = dict(s)
    bad['p_d'] = s['p_d'].copy()
    bad['p_d'][np.nonzero(X == 0)[0][0], np.nonzero(X == 0)[1][0]] = 1.
    with pytest.raises(ValueError):
        ZIGaP(S, k=K, use_factors=False, state=bad)


def _h2d_formula(h, form, rows_per_slab, K):
    """Bytes one step sends host -> device: the gene side once, then per slab the counts in their host form and a1, a2."""
    from oriana_b200 import _lib
    p = h.p
    total = 2 * p * K * 4 + 4 * K * 8 + p * 8 + _lib.ORI_SC_NSLOTS * 8
    for r0 in range(0, h.n, rows_per_slab):
        rows = min(rows_per_slab, h.n - r0)
        lo, hi = form.byte_range(r0, r0 + rows)
        if hasattr(form, 'bitmap'):
            e0, e1 = form.escapes(r0, r0 + rows)
            total += rows * form.bitmap.shape[1] * 4 + (hi - lo) + (rows + 1) * 8 + 12 * (e1 - e0)
        else:
            total += (rows + 1) * 8 + (hi - lo) * (form.idx_bytes + form.values.element_size())
        total += 2 * rows * K * 4
    return total


@pytest.mark.parametrize('big', [False, True])
def test_host_streamed_step_with_csr_counts(cuda_lib, big):
    """CsrCounts in HostStreamedCAVI: every slab X is bit-identical to the SparseCounts slab, 3 steps agree with the
    SparseCounts run, and h2d_bytes is each form's byte count.  big=True: counts >= 255 and >= 2^16 (float32 values)."""
    import torch
    from oriana.singlecell import CountMatrix
    from oriana_b200.host_step import CsrCounts, HostStreamedCAVI
    g = load_golden('zigap_ragged')
    s = dict(golden_state(g, 0))
    X = s['X'].copy()
    X[64] = 0
    if big:
        X[3, 7] = 255; X[100, 330] = 70000
    s['X'] = X
    K = s['a1'].shape[1]
    cm = CountMatrix(sp.csr_matrix(X))
    spc, csr = cm.to_sparse_counts(), cm.to_csr_counts()
    assert isinstance(csr, CsrCounts) and csr.values.dtype == (torch.float32 if big else torch.uint8)
    assert torch.equal(csr.dense(), torch.as_tensor(X.astype(np.float32)))
    runs = []
    for form in (spc, csr):
        h = HostStreamedCAVI(form, K, s, dropout=True, slab_rows=64)
        slabs, loop = [], h._slab_loop

        def recording(body, loop=loop, slabs=slabs):
            def rec(sl, P, r0, rows, st):
                slabs.append(sl['X'][:rows].clone())
                body(sl, P, r0, rows, st)
            loop(rec)
        h._slab_loop = recording
        elbo = []
        for _ in range(3):
            b0 = h.h2d_bytes
            elbo.append(h.step())
            assert h.h2d_bytes - b0 == _h2d_formula(h, form, 64, K)
        torch.cuda.synchronize()
        runs.append((h, slabs, elbo))
    (hs, xs, es), (hc, xc, ec) = runs
    assert len(xs) == len(xc) == 3 * ((hs.n + 63) // 64)
    for a, b in zip(xs, xc):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    for k in PARAMS:
        assert relerr(hc.state_dict()[k], hs.state_dict()[k]) < 5e-6, k
    assert abs(ec[-1] - es[-1]) < 1e-6 * abs(es[-1])
