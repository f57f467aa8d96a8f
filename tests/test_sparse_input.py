"""CPU: scipy.sparse count matrices in CountMatrix and the sparse host forms of the host-streamed step.

Every method gives for a CSR, CSC or COO input what it gives for the dense array of the same counts -- with stored zeros,
duplicate entries (summed as scipy sums them), empty rows and columns -- and nothing densifies the matrix unless asked
to (`as_array()`)."""
import tracemalloc

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oriana_b200.exceptions import DatatypeException
from oriana_b200.host_step import CsrCounts, SparseCounts
from oriana_b200.singlecell.cmatrix import CountMatrix

FORMATS = ('csr', 'csc', 'coo', 'csr_array')


def _counts(n, p, dtype, seed=0, density=0.3):
    rng = np.random.default_rng(seed)
    X = rng.poisson(4., size=(n, p)) * (rng.random((n, p)) < density)
    X[n // 2] = 0                                              # an empty cell
    X[:, p // 3] = 0                                           # an empty gene
    X[0, p - 1] = 255
    if dtype == np.float32:
        X = X.astype(np.float32)
        X[1, 1] = 2.5                                          # non-integral: stored as float32
    elif dtype == np.int64:
        X[n - 1, 0] = 70000                                    # beyond uint16
    else:
        X[n - 1, 0] = 65535
    return X.astype(dtype)


def _messy(X, fmt):
    """The counts of X as `fmt`: some entries split into two duplicates, stored zeros, rows in unsorted order."""
    r, c = np.nonzero(X)
    v = X[r, c]
    half = np.floor(v / 2).astype(X.dtype)
    split = (np.arange(r.size) % 3 == 0) & (half > 0)
    zr, zc = np.nonzero(X == 0)
    zr, zc = zr[::7], zc[::7]                                  # stored zeros
    rows = np.concatenate((r, r[split], zr))
    cols = np.concatenate((c, c[split], zc))
    vals = np.concatenate((np.where(split, v - half, v), half[split], np.zeros(zr.size, X.dtype))).astype(X.dtype)
    perm = np.random.default_rng(1).permutation(rows.size)
    coo = sp.coo_matrix((vals[perm], (rows[perm], cols[perm])), shape=X.shape)
    if fmt == 'coo':
        return coo
    if fmt == 'csc':
        return coo.tocsc()
    # a CSR with unsorted indices and duplicates (not canonical), built from its raw arrays
    order = np.argsort(rows[perm], kind='stable')
    indptr = np.zeros(X.shape[0] + 1, dtype=np.int32)
    np.cumsum(np.bincount(rows[perm], minlength=X.shape[0]), out=indptr[1:])
    csr = sp.csr_matrix((vals[perm][order], cols[perm][order], indptr), shape=X.shape)
    return sp.csr_array(csr) if fmt == 'csr_array' else csr


def _snapshot(S):
    return [a.copy() for a in ((S.data, S.row, S.col) if S.format == 'coo' else (S.data, S.indices, S.indptr))]


def _fields_equal(a, b, names):
    for f in names:
        x, y = getattr(a, f), getattr(b, f)
        assert x.dtype == y.dtype and x.shape == y.shape, f
        assert np.array_equal(x.numpy().view(np.uint8), y.numpy().view(np.uint8)), f


@pytest.mark.parametrize('fmt', FORMATS)
@pytest.mark.parametrize('dtype', [np.uint16, np.int64, np.float32])
@pytest.mark.parametrize('labels', [False, True])
def test_sparse_count_matrix_matches_dense(fmt, dtype, labels):
    n, p = 41, 37
    X = _counts(n, p, dtype)
    S = _messy(X, fmt)
    assert np.array_equal(S.toarray(), X)
    before = _snapshot(S)
    kw = dict(row_names=np.array(['c%d' % i for i in range(n)]), col_names=np.array(['g%d' % j for j in range(p)])) \
        if labels else {}
    cs, cd = CountMatrix(S, **kw), CountMatrix(X.copy(), **kw)
    assert cs.is_sparse and not cd.is_sparse and cs.shape == cd.shape == (n, p)
    a = cs.as_array()
    assert isinstance(a, np.ndarray) and a.dtype == X.dtype and np.array_equal(a, X)
    for mode in ('csr', 'csc'):
        ms, md = cs.as_sparse_matrix(mode), cd.as_sparse_matrix(mode)
        assert ms.format == md.format == mode and ms.nnz == md.nnz and np.array_equal(ms.toarray(), md.toarray())
    assert np.array_equal(cs.row_names, cd.row_names) and np.array_equal(cs.col_names, cd.col_names)
    ts, td = cs.T, cd.T
    assert ts.is_sparse and ts.shape == (p, n) and np.array_equal(ts.as_array(), td.as_array())
    assert np.array_equal(ts.row_names, td.row_names) and np.array_equal(ts.col_names, td.col_names)
    gene = cd.col_names[5]
    assert cs[gene].dtype == cd[gene].dtype and np.array_equal(cs[gene], cd[gene])
    assert cs.is_uint16() == cd.is_uint16() == (dtype == np.uint16)
    assert cs.narrow_dtype() == cd.narrow_dtype()
    for world in (1, 3):
        for r in range(world):
            bs, bd = cs.row_block(r, world), cd.row_block(r, world)
            assert bs.is_sparse and np.array_equal(bs.as_array(), bd.as_array())
            assert np.array_equal(bs.row_names, bd.row_names)
    pick = cd.row_names[[7, 2, 2, 30]]
    fs, fd = cs.filter_rows(pick, inplace=False), cd.filter_rows(pick, inplace=False)
    assert fs.is_sparse and np.array_equal(fs.as_array(), fd.as_array()) and np.array_equal(fs.row_names, fd.row_names)
    # the host forms of the host-streamed step (the dense encoders need torch arithmetic, which uint16 lacks: int64 there)
    cw = CountMatrix(X.astype(np.int64)) if dtype == np.uint16 else cd
    _fields_equal(cs.to_sparse_counts(pin=False), cw.to_sparse_counts(pin=False), ('bitmap', 'nz', 'rowoff', 'row', 'col', 'val'))
    _fields_equal(cs.to_compact(pin=False), cw.to_compact(pin=False), ('u8', 'row', 'col', 'val'))
    csr_s = cs.to_csr_counts(pin=False)
    assert torch.equal(csr_s.dense(), torch.from_numpy(X.astype(np.float32)))
    _fields_equal(csr_s, cw.to_csr_counts(pin=False), ('indptr', 'indices', 'values'))
    # column assignment, then in-place row filtering
    v = (np.arange(n) % 4).astype(dtype)
    cs[gene] = v
    cd[gene] = v
    assert cs.is_sparse and np.array_equal(cs.as_array(), cd.as_array()) and cs.as_array().dtype == X.dtype
    assert cs.filter_rows(pick) is cs and np.array_equal(cs.as_array(), cd.filter_rows(pick).as_array())
    # the caller's matrix is never modified
    for x, y in zip(before, _snapshot(S)):
        assert np.array_equal(x, y)


def test_canonical_csr_is_shared_and_lists_are_refused():
    X = _counts(20, 30, np.int64)
    S = sp.csr_matrix(X)
    assert S.has_canonical_format
    c = CountMatrix(S)
    assert np.shares_memory(c.as_tensor().data, S.data) and np.shares_memory(c.as_tensor().indices, S.indices)
    messy = _messy(X, 'csr')
    c2 = CountMatrix(messy)
    assert not np.shares_memory(c2.as_tensor().data, messy.data) and c2.as_tensor().has_canonical_format
    # duplicates summed, stored zeros kept (scipy's canonical form); as_sparse_matrix() drops them
    assert c2.as_tensor().nnz == S.nnz + (int(np.count_nonzero(X == 0)) + 6) // 7
    assert c2.as_sparse_matrix('csr').nnz == S.nnz
    with pytest.raises(DatatypeException):
        CountMatrix([[1, 2], [3, 4]])
    with pytest.raises(DatatypeException):
        CountMatrix(sp.coo_array(np.arange(5)))                 # 1-D
    with pytest.raises(DatatypeException):
        CountMatrix(S, row_names=['a'])


def test_large_sparse_matrix_is_never_densified():
    """200 000 x 50 000 cells x genes (a 40 GB float32 dense form) with 10^5 non-zeros: every method that has no reason
    to densify runs in a few MB."""
    n, p, nnz = 200_000, 50_000, 100_000
    rng = np.random.default_rng(2)
    rows, cols = rng.integers(0, n, nnz), rng.integers(0, p, nnz)
    S = sp.coo_matrix((rng.integers(1, 300, nnz).astype(np.float32), (rows, cols)), shape=(n, p))
    tracemalloc.start()
    try:
        c = CountMatrix(S)
        t = c.T
        blk = c.row_block(1, 4)
        sub = c.filter_rows(np.arange(0, n, 1000), inplace=False)
        nd = c.narrow_dtype()
        csc, csr = c.as_sparse_matrix(), c.as_sparse_matrix('csr')
        hc = c.to_csr_counts(pin=False)
        peak = tracemalloc.get_traced_memory()[1]
    finally:
        tracemalloc.stop()
    assert peak < 200 << 20, peak
    assert t.shape == (p, n) and blk.shape == (50_000, p) and sub.shape == (200, p) and nd == torch.uint16
    assert csc.format == 'csc' and csr.nnz == c.as_tensor().nnz
    assert hc.indices.dtype == torch.uint16 and hc.values.dtype == torch.uint16 and hc.indices.numel() == csr.nnz


@pytest.mark.parametrize('n,p', [(7, 33), (50, 100), (33, 64), (5, 1), (64, 2049)])
def test_sparse_counts_from_csr_equal_from_tensor(n, p):
    """Bitmap from the indices, saturating bytes, escape list: field for field what the dense encoder makes, across
    chunk boundaries of the CSR encoder."""
    rng = np.random.default_rng(n * p)
    X = (rng.poisson(20, (n, p)) * (rng.random((n, p)) < 0.5)).astype(np.float32)
    X[rng.integers(0, n), rng.integers(0, p)] = 300.
    X[0, p - 1] = 255.; X[n - 1, 0] = 1000.; X[n // 2] = 0.
    ref = SparseCounts.from_tensor(torch.from_numpy(X), pin=False)
    for chunk in (1, 17, 1 << 24):
        got = SparseCounts.from_csr(_messy(X, 'csr'), pin=False, chunk_nnz=chunk)
        _fields_equal(got, ref, ('bitmap', 'nz', 'rowoff', 'row', 'col', 'val'))


@pytest.mark.parametrize('top,vdt', [(200, torch.uint8), (60000, torch.uint16), (70000, torch.float32), (2.5, torch.float32)])
@pytest.mark.parametrize('p', [13, 65536, 70000])
def test_csr_counts_round_trip(top, vdt, p):
    n = 6
    rng = np.random.default_rng(p)
    X = np.zeros((n, p), dtype=np.float32)
    for r in (0, 2, 5):                                        # rows 1, 3, 4 are empty
        cols = rng.choice(p, size=min(p, 9), replace=False)
        X[r, cols] = rng.integers(1, 50, cols.size)
    X[5, p - 1] = top
    for cc in (CsrCounts.from_tensor(torch.from_numpy(X), chunk_rows=4, pin=False), CsrCounts.from_csr(sp.csr_matrix(X), pin=False),
               CountMatrix(sp.csc_matrix(X)).to_csr_counts(pin=False)):
        assert torch.equal(cc.dense(), torch.from_numpy(X))
        assert cc.values.dtype == vdt and cc.indices.dtype == (torch.uint16 if p <= 65536 else torch.int32)
        nnz = int(np.count_nonzero(X))
        assert cc.indices.numel() == nnz and cc.byte_range(1, 2) == (cc.byte_range(0, 1)[1],) * 2
        assert cc.nbytes == 8 * (n + 1) + nnz * (cc.idx_bytes + cc.values.element_size())
    zero = CsrCounts.from_csr(sp.csr_matrix((3, 5), dtype=np.float32), pin=False)
    assert zero.indices.numel() == 0 and not zero.dense().any()
