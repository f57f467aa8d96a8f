"""GPU: counts handed in as uint16 stay uint16 in HBM (ORI_F_X_U16) on every model, pass and kernel family.

Every kernel widens a uint16 count to float32 exactly, and everything after that is the float32 model's code, so a model of
uint16 counts and a model of the same counts as float32, started from the same state with deterministic=True, agree in
every bit of every parameter.  The ELBO trace carries sum lgamma(X + 1), a constant formed once per model with float64
atomics, hence the 1e-13 there (as in test_tensor_path_gpu.py's determinism test).

uint16 storage is chosen only where the float32 matrix would not fit the device (`oriana_b200.problem.counts_storage`):
these tests select it for every uint16 input (`uint16_storage`), except the one that checks the default choice."""
import gc

import numpy as np
import pytest

from conftest import golden_state, load_golden, relerr

pytestmark = pytest.mark.gpu
PARAMS = ('a1', 'a2', 'b1', 'b2', 'alpha1', 'alpha2', 'beta1', 'beta2')


@pytest.fixture(autouse=True)
def uint16_storage(monkeypatch):
    """Keep every uint16 input as uint16 in HBM, at any size."""
    import torch
    from oriana_b200 import problem
    monkeypatch.setattr(problem, 'counts_storage', lambda u16, *args: torch.uint16 if u16 else torch.float32)


def _counts(n, p, K, seed, zero_cell=None, zero_gene=None):
    from oracle import cavi_numpy as cn
    X = cn.synth_counts(n, p, K, seed=seed)
    X[seed % n, seed % p] = 65535                      # counts past the uint8 range, up to the largest uint16
    X[(seed + 3) % n, :min(p, 9)] = 300
    if zero_cell is not None:
        X[zero_cell, :] = 0
    if zero_gene is not None:
        X[:, zero_gene] = 0
    return X


def _pair(model, X, K, steps=5, **kw):
    """(float32 model, uint16 model) of the same counts from the same state, stepped `steps` times."""
    import torch
    from oracle import cavi_numpy as cn
    from oriana.models import GaP, SparseZIGaP, ZIGaP
    from oriana.singlecell import CountMatrix
    cls = dict(zigap=ZIGaP, gap=GaP, sparse=SparseZIGaP)[model]
    models = []
    for dt in (np.float32, np.uint16):
        if model == 'sparse':                           # the constructor's own draws, from the same seed
            np.random.seed(5)
            m = cls(CountMatrix(X.astype(dt)), k=K, use_factors=False, **kw)
        else:
            s = cn.init_state(X, K, np.random.default_rng(1), model)
            m = cls(CountMatrix(X.astype(dt)), k=K, use_factors=False, state=s, **kw)
        for _ in range(steps):
            m.step()
        models.append(m)
    m32, m16 = models
    assert m32.counts_dtype == torch.float32 and m16.counts_dtype == torch.uint16
    assert m16._X.dtype == torch.uint16 and m16._X.element_size() == 2
    assert m32.uses_tensor_path == m16.uses_tensor_path
    return m32, m16


def _assert_identical(m32, m16):
    names = PARAMS + (('pi_d',) if hasattr(m32, 'pi_d') else ())
    for k in names:
        a, b = getattr(m32, k).asarray(), getattr(m16, k).asarray()
        assert np.array_equal(a, b), (k, float(np.max(np.abs(a - b))))
    assert np.array_equal(m32.U_hat, m16.U_hat) and np.array_equal(m32.V_hat, m16.V_hat)
    if m32._flags & 4:                                    # ORI_F_ELBO
        np.testing.assert_allclose(m16.elbo_trace, m32.elbo_trace, rtol=1e-13)
    if hasattr(m32, 'reconstruction_deviance'):
        assert m32.reconstruction_deviance() == m16.reconstruction_deviance()
        assert m32.explained_deviance() == m16.explained_deviance()


CASES = {
    'zigap_tensor_kp32': ('zigap', (2100, 1003, 12), dict()),                   # >= 2^21 entries: the default plan
    'zigap_tensor_k40': ('zigap', (700, 517, 40), dict(tensor=True)),
    'zigap_tensor_k64': ('zigap', (600, 389, 64), dict(tensor=True)),
    'zigap_tensor_precise': ('zigap', (640, 333, 12), dict(tensor=True, precise=True)),
    'gap_tensor': ('gap', (900, 261, 10), dict(tensor=True)),
    'sparse_tensor': ('sparse', (800, 301, 8), dict(tensor=True)),
    'sparse_cuda_core_k40': ('sparse', (300, 203, 40), dict()),
    'zigap_force_simt': ('zigap', (500, 129, 7), dict(force_simt=True)),
    'gap_force_simt': ('gap', (410, 150, 9), dict(force_simt=True)),
    'zigap_quirk_tensor': ('zigap', (600, 250, 10), dict(tensor=True, compat_quirk=True)),
    'zigap_quirk_simt': ('zigap', (300, 120, 6), dict(compat_quirk=True)),
    'zigap_graphs_tensor': ('zigap', (640, 300, 12), dict(tensor=True, graphs=True)),
}


@pytest.mark.parametrize('case', sorted(CASES))
def test_uint16_model_is_bit_identical_to_float32(cuda_lib, case):
    model, (n, p, K), kw = CASES[case]
    X = _counts(n, p, K, seed=n % 89, zero_cell=17, zero_gene=5)
    m32, m16 = _pair(model, X, K, deterministic=True, **kw)
    if kw.get('tensor') or n * p >= 1 << 21:
        assert m16.uses_tensor_path
    _assert_identical(m32, m16)


@pytest.mark.parametrize('tensor', [True, False])
@pytest.mark.parametrize('p', [57, 58, 59, 60, 61, 62, 63])
def test_uint16_ragged_shapes(cuda_lib, p, tensor):
    """p = 1 ... 7 (mod 8) below one 64-gene tile, n not a multiple of 256: the padded uint16 pitch and the partial boxes."""
    X = _counts(300, p, 6, seed=p, zero_cell=2, zero_gene=p - 1)
    m32, m16 = _pair('zigap', X, 6, deterministic=True, **(dict(tensor=True) if tensor else dict(force_simt=True)))
    assert m16.uses_tensor_path == tensor
    assert m16._ldx % 8 == 0 and m16._ldx >= p
    _assert_identical(m32, m16)


@pytest.mark.parametrize('model', ['gap', 'zigap'])
@pytest.mark.parametrize('tensor,tol', [(False, 2e-5), (True, 3e-3)])
def test_uint16_underflow_emulation(cuda_lib, model, tensor, tol):
    """emulate_underflow=True (not combinable with deterministic=True): the uint16 model follows the float32 model at the
    tolerances of test_underflow_gpu.py, on both kernel families."""
    X = _counts(2048 if tensor else 260, 1024 if tensor else 330, 6, seed=11)
    m32, m16 = _pair(model, X, 6, emulate_underflow=True, **(dict(tensor=True) if tensor else dict(force_simt=True)))
    for k in PARAMS:
        assert relerr(getattr(m16, k).asarray(), getattr(m32, k).asarray()) < tol, k


@pytest.mark.parametrize('name,tensor', [('zigap_ragged', False), ('zigap_k32', True)])
def test_uint16_golden_trajectory(cuda_lib, name, tensor):
    """The reference's recorded trajectory from uint16 counts, at the tolerances of test_cavi_gpu.py (CUDA-core kernels)
    and test_tensor_path_gpu.py (tcgen05 passes)."""
    import torch
    from oriana.models import ZIGaP
    from oriana.singlecell import CountMatrix
    g = load_golden(name)
    s = golden_state(g, 0)
    steps = [int(t) for t in g['steps']]
    m = ZIGaP(CountMatrix(s['X'].astype(np.uint16)), k=s['a1'].shape[1], use_factors=False, state=s, compat_quirk=True,
              tensor=tensor or None, trace_cap=max(steps) + 8)
    assert m.counts_dtype == torch.uint16 and m.uses_tensor_path == tensor
    for t in range(1, max(steps) + 1):
        m.step()
        if t in steps:
            r = golden_state(g, t)
            for k in PARAMS + ('pi_d',):
                ftol = (3e-3 if k in ('a1', 'a2', 'b1', 'b2') else 5e-4) if tensor else \
                    (2e-5 if t <= 1 else (6e-5 if t <= 10 else 2e-4))
                e = relerr(getattr(m, k).asarray(), r[k])
                assert e < ftol, (name, t, k, e)


def _u16_block(X, pitch):
    """A resident torch.uint16 [n, p] block with row pitch `pitch` (elements)."""
    import torch
    n, p = X.shape
    buf = torch.zeros((n, pitch), dtype=torch.int16, device='cuda')
    buf[:, :p].copy_(torch.from_numpy(X.astype(np.uint16)).view(torch.int16))
    return buf.view(torch.uint16)[:, :p]


def test_resident_uint16_block_is_adopted_or_copied(cuda_lib):
    import torch
    from oracle import cavi_numpy as cn
    from oriana.models import ZIGaP
    from oriana.singlecell import CountMatrix
    n, p, K = 400, 261, 5
    X = _counts(n, p, K, seed=4)
    s = cn.init_state(X, K, np.random.default_rng(1), 'zigap')
    good = _u16_block(X, 272)                                      # pitch a multiple of 8: adopted as it is
    m = ZIGaP(CountMatrix(good), k=K, use_factors=False, state=s, deterministic=True)
    assert m.counts_dtype == torch.uint16 and m._X.data_ptr() == good.data_ptr() and m._ldx == 272
    bad = _u16_block(X, 261)                                       # odd pitch: copied into the padded one
    mb = ZIGaP(CountMatrix(bad), k=K, use_factors=False, state=s, deterministic=True)
    assert mb.counts_dtype == torch.uint16 and mb._X.data_ptr() != bad.data_ptr() and mb._ldx == 264
    ref = ZIGaP(CountMatrix(X.astype(np.float32)), k=K, use_factors=False, state=s, deterministic=True)
    for mm in (m, mb, ref):
        for _ in range(3):
            mm.step()
    for k in PARAMS:
        assert np.array_equal(m.__getattribute__(k).asarray(), ref.__getattribute__(k).asarray()), k
        assert np.array_equal(mb.__getattribute__(k).asarray(), ref.__getattribute__(k).asarray()), k
    assert m.X[:].dtype == np.uint16 and np.array_equal(m.X[:], X)
    assert CountMatrix(X.astype(np.uint16)).as_array().dtype == np.uint16


def test_uint16_allocation_is_half_of_float32(cuda_lib):
    import torch
    from oriana_b200.problem import row_pitch
    from oriana.singlecell import CountMatrix
    n, p = 1024, 1001                                              # n * ldx * 2 is a multiple of the allocator's 512 bytes
    X = _counts(n, p, 4, seed=2).astype(np.uint16)
    gc.collect()                      # earlier tests' models (reference cycles) must not be freed inside the measurement
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    Xd = CountMatrix(X).to_device('cuda', dtype=torch.uint16)
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() - before == n * row_pitch(p, 2) * 2
    assert Xd.dtype == torch.uint16 and Xd.stride(0) == 1008
    assert np.array_equal(Xd.cpu().numpy(), X)


def test_uint16_metrics_and_device_nmf_match_float32(cuda_lib, monkeypatch):
    """frobenius_norm(), GaP's loglikelihood() and the device NMF warm start read uint16 X through float32 slabs: here
    twelve slabs of 127 cells and a ragged last one of 103, against the float32 model read in one piece."""
    from oracle import cavi_numpy as cn
    from oriana.models import GaP, ZIGaP
    from oriana.singlecell import CountMatrix
    n, p, K = 1500, 700, 6
    slab = 127 * p
    X = _counts(n, p, K, seed=9)
    for cls, model in ((GaP, 'gap'), (ZIGaP, 'zigap')):
        s = cn.init_state(X, K, np.random.default_rng(1), model)
        # int32 counts are stored as float32 and, like uint16, make the Poisson terms integer-truncated (poisson.py:68)
        m32 = cls(CountMatrix(X.astype(np.int32)), k=K, use_factors=False, state=s, deterministic=True)
        m16 = cls(CountMatrix(X.astype(np.uint16)), k=K, use_factors=False, state=s, deterministic=True)
        m16._X_SLAB_ENTRIES = slab
        assert len(list(m16._x_slabs(127))) == 12
        for mm in (m32, m16):
            mm.step()
        f32, f16 = m32.frobenius_norm(), m16.frobenius_norm()
        assert abs(f16 - f32) <= 1e-6 * abs(f32), (f16, f32)
        if model == 'gap':
            l32, l16 = m32.loglikelihood(), m16.loglikelihood()
            assert abs(l16 - l32) <= 1e-12 * abs(l32), (l16, l32)      # the same terms, summed in another order
    nmf = []
    for dt in (np.float32, np.uint16):
        if dt == np.uint16:
            monkeypatch.setattr(ZIGaP, '_X_SLAB_ENTRIES', slab)
        np.random.seed(3)
        m = ZIGaP(CountMatrix(X.astype(dt)), k=K, use_factors=True, nmf='device')
        nmf.append((m._nmf_U.cpu().numpy(), m._nmf_V.cpu().numpy()))
    # the slabs' partial X^T U products are added in another order than one GEMM forms them, and 100 multiplicative
    # updates amplify that rounding (measured 1.9e-4 at 127-cell slabs): errors relative to the factor's scale (floor 1e-3 of
    # its largest entry); a misplaced slab would be off by O(1)
    for got, want in zip(nmf[1], nmf[0]):
        assert relerr(got, want, floor=1e-3) < 1e-3


def test_uint16_inputs_that_fit_as_float32_keep_float32_storage(cuda_lib, monkeypatch):
    """The default choice: uint16 counts whose float32 matrix fits the device are stored as float32 -- numpy, host tensor
    and resident CUDA block alike -- and give exactly the float32 model's results."""
    import torch
    from oracle import cavi_numpy as cn
    from oriana.models import ZIGaP
    from oriana.singlecell import CountMatrix
    monkeypatch.undo()
    n, p, K = 700, 261, 6
    X = _counts(n, p, K, seed=6)
    s = cn.init_state(X, K, np.random.default_rng(1), 'zigap')
    X16 = X.astype(np.uint16)
    host = torch.from_numpy(X16)
    models = [ZIGaP(CountMatrix(src), k=K, use_factors=False, state=s, deterministic=True, tensor=True)
              for src in (X.astype(np.float32), X16, host, _u16_block(X, 272))]
    for m in models:
        assert m.counts_dtype == torch.float32 and m._X.dtype == torch.float32
        for _ in range(3):
            m.step()
    for m in models[1:]:
        for k in PARAMS:
            assert np.array_equal(getattr(m, k).asarray(), getattr(models[0], k).asarray()), k


# --------------------------------------------------------------------------- every uint16 value
def _all_values(n, p, seed):
    """[n, p] int64 counts that hold each of the 65536 uint16 values at least once, at random places."""
    rng = np.random.default_rng(seed)
    X = rng.poisson(2.0, (n, p)) * (rng.random((n, p)) < 0.5)
    X.flat[rng.permutation(n * p)[:65536]] = np.arange(65536)
    return X


@pytest.mark.parametrize('p', [127, 128, 129, 257])
def test_uint16_count_statistics_are_exact(cuda_lib, p):
    """The constant statistics of uint16 X against exact sums, over the 128-gene blocks (p = 127 ... 257) and the row
    chunks of `launch_count_stats` / `launch_col_sums` (every row on either side of a chunk seam holds no zero, so a chunk
    that loses its first or last row changes every column's sum):
    - ori_column_sums_u16_f64 is exact: every partial sum is an integer below 2^53, whatever the order of the atomics;
    - ori_row_sums_u16_f32 is exact where the row sums to less than 2^24; above, off by the float32 roundings of its
      five warp-shuffle additions at most (each lane's partial sum is below 2^24);
    - a ZIGaP model on uint16 storage, initial start: pi_d = (X > 0).sum(0) / n and the non-zero count exactly, and
      sum lgamma(X + 1) (lgammaf per entry, CUDA: 6 ulp for positive arguments) within 4e-7 of the float64 sum.
      Measured: 2.9e-9 relative at every p (one B200, 1000 W power limit)."""
    import math
    import torch
    from oriana.models import ZIGaP
    from oriana.singlecell import CountMatrix
    from oriana_b200 import _lib
    from oriana_b200.problem import row_pitch
    from test_kernel_edges_gpu import count_chunk_rows
    n = 3000
    X = _all_values(n - 1, p, seed=p)
    X = np.vstack([np.full((1, p), 65535 if p > 256 else 1), X])        # p = 257: a row sum of 1.68e7 > 2^24
    rpc = count_chunk_rows(n, p)
    assert 16 <= rpc < n // 64
    seams = [r for b in range(rpc, n, rpc) for r in (b - 1, b)]
    X[seams] = np.maximum(X[seams], 1)
    assert np.unique(X).size == 65536
    Xd = _u16_block(X, row_pitch(p, 2))
    cols = torch.zeros((p,), dtype=torch.float64, device='cuda')
    rows = torch.full((n,), float('nan'), dtype=torch.float32, device='cuda')
    _lib.check(cuda_lib.ori_column_sums_u16_f64(Xd.data_ptr(), Xd.stride(0), n, p, cols.data_ptr(), _lib.stream_ptr()))
    _lib.check(cuda_lib.ori_row_sums_u16_f32(Xd.data_ptr(), Xd.stride(0), n, p, rows.data_ptr(), _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert np.array_equal(cols.cpu().numpy(), X.sum(0).astype(np.float64))
    got, want = rows.cpu().numpy().astype(np.float64), X.sum(1)
    small = want < 1 << 24
    assert np.array_equal(got[small], want[small].astype(np.float64))
    assert (p > 256) == (not small.all())
    assert np.all(np.abs(got[~small] - want[~small]) <= 5 * 2.0 ** -24 * want[~small])

    np.random.seed(1)
    m = ZIGaP(CountMatrix(X.astype(np.uint16)), k=4, use_factors=False)
    assert m.counts_dtype == torch.uint16 and m._X.element_size() == 2 and m._ldx % 8 == 0
    assert np.array_equal(m.pi_d.asarray(), (X > 0).sum(0) / n)
    scal = m._scal.cpu().numpy()
    assert scal[_lib.ORI_SC_NNZ] == np.count_nonzero(X)
    lg = np.array([math.lgamma(v + 1.) for v in range(65536)])
    want_lg = float(np.bincount(X.ravel(), minlength=65536) @ lg)
    err = abs(scal[_lib.ORI_SC_LGAMX] - want_lg) / want_lg
    print('p = %d: sum lgamma(X + 1) relative error %.2e' % (p, err))
    assert err < 4e-7, err


ALL_VALUE_PLANS = {      # model, K, model arguments, plan of test_kernel_edges_gpu.py (its tolerances)
    'zigap_tf32_kp32': ('zigap', 12, dict(tensor=True), 'tf32'),
    'zigap_tf32_kp64': ('zigap', 40, dict(tensor=True), 'tf32'),
    'zigap_precise': ('zigap', 12, dict(tensor=True, precise=True), 'precise'),
    'zigap_cuda_core': ('zigap', 12, dict(force_simt=True), 'simt'),
    'gap_tf32_kp32': ('gap', 12, dict(tensor=True), 'tf32'),
}


@pytest.mark.parametrize('case', sorted(ALL_VALUE_PLANS))
def test_every_uint16_value_through_the_passes(cuda_lib, case):
    """A ragged 300 x 257 problem whose counts take each of the 65536 uint16 values: in deterministic mode the uint16
    model is bit-identical to the float32 model (the widening is exact for every bit pattern, not only the few `_counts`
    places), and one plain step from the initial state matches the float64 oracle at the plan's tolerances."""
    from oracle import cavi_numpy as cn
    from test_kernel_edges_gpu import _check_step, _model, _refresh
    model, K, kw, plan = ALL_VALUE_PLANS[case]
    X = _all_values(300, 257, seed=K)
    m32, m16 = _pair(model, X, K, deterministic=True, **kw)
    assert m16.uses_tensor_path == (plan != 'simt')
    _assert_identical(m32, m16)
    s = _refresh(cn.init_state(X, K, np.random.default_rng(2), model), 'init', model)
    kw = {k: v for k, v in kw.items() if k != 'force_simt'}
    m = _model(s, model, plan, 'u16', **kw)
    assert m.uses_tensor_path == (plan != 'simt')
    _check_step(m, s, [], model, plan)
