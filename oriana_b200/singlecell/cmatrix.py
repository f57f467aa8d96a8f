"""Count-matrix container (oriana/singlecell/cmatrix.py:12-121): the hand-off to the models, and the ingest step in
front of the CAVI path (SURVEY.md 8f row 3).

Accepts what the reference accepts (numpy array, pandas DataFrame) plus a torch tensor that may already be resident
in HBM (this rank's row block of a sharded matrix) and a scipy.sparse matrix or array (CSR, CSC, COO, anything with
`.tocsr()`), the form single-cell data arrive in.  Anything else raises DatatypeException (cmatrix.py:25-29).
A sparse matrix is kept as canonical CSR (sorted indices, duplicates summed; copied only when it is not canonical CSR)
and is never densified implicitly: `as_array()` is the explicit request, every other method works on the CSR.
The reference keeps a DataFrame; here the counts stay in the array they arrived in (no copy) and the row / column
labels are kept beside them, so that the label-based calls (`cm['gene']`, `filter_rows`, `row_names`, `col_names`)
behave like the reference's without a pandas round trip of the matrix.

Ingest helpers with no counterpart in the reference: `row_block` (the contiguous cell range a rank owns, SURVEY.md
8e), `to_device` (the matrix in HBM with the 16-byte row pitch the kernels want, uploaded in slabs: float32, widened on
the device from the narrowest integer type that holds the counts, or uint16 as it is for counts handed in as uint16),
`to_compact` (saturating uint8 + escape list for host-streamed runs), `to_sparse_counts` and `to_csr_counts` (the
sparse host forms of the host-streamed step).
"""
import sys

import numpy as np
import torch

from ..exceptions import DatatypeException


def _is_sparse(a):
    """A scipy.sparse matrix or array (no import: an object of that kind means scipy.sparse is loaded already)."""
    sp = sys.modules.get('scipy.sparse')
    return sp is not None and sp.issparse(a)


def canonical_csr(a):
    """`a` (scipy.sparse, any format) as a canonical scipy CSR matrix: sorted indices, duplicates summed as scipy sums
    them.  Canonical CSR input is shared, not copied; the caller's object is never modified."""
    import scipy.sparse
    csr = scipy.sparse.csr_matrix(a if a.format == 'csr' else a.tocsr())     # csr_matrix of a CSR shares its arrays
    if not csr.has_canonical_format:
        if a.format == 'csr':
            csr = csr.copy()
        csr.sum_duplicates()                                                  # sorts the indices too
    return csr


def narrow_count_dtype(a):
    """Narrowest unsigned integer type (torch.uint8 / torch.uint16) that holds every value of the numpy array `a`, or
    None: the values are not non-negative integers below 2^16."""
    if a.size == 0:
        return torch.uint8
    lo, hi = float(a.min()), float(a.max())
    integral = np.issubdtype(a.dtype, np.integer) or bool((a == np.round(a)).all())
    if not integral or lo < 0 or hi >= 65536:
        return None
    return torch.uint8 if hi < 256 else torch.uint16


class CountMatrix:

    def __init__(self, data, row_names=None, col_names=None):
        self._rows = None if row_names is None else np.asarray(row_names)
        self._cols = None if col_names is None else np.asarray(col_names)
        if isinstance(data, torch.Tensor):
            if data.dim() != 2:
                raise DatatypeException('Count matrix must be 2-D, got %d-D' % data.dim())
            self._data = data
        elif isinstance(data, np.ndarray):
            if data.ndim != 2:
                raise DatatypeException('Count matrix must be 2-D, got %d-D' % data.ndim)
            self._data = data
        elif hasattr(data, 'values') and hasattr(data, 'columns'):   # pandas DataFrame
            self._rows, self._cols = np.asarray(data.index), np.asarray(data.columns.values)
            self._data = np.asarray(data.values)
        elif _is_sparse(data) or hasattr(data, 'tocsr'):
            if getattr(data, 'ndim', 2) != 2:
                raise DatatypeException('Count matrix must be 2-D, got %d-D' % data.ndim)
            csr = data if _is_sparse(data) else data.tocsr()
            if not _is_sparse(csr):
                raise DatatypeException('Incompatible type %s' % type(data))
            self._data = canonical_csr(csr)
        else:
            raise DatatypeException('Incompatible type %s' % type(data))
        for names, axis in ((self._rows, 0), (self._cols, 1)):
            if names is not None and len(names) != self._data.shape[axis]:
                raise DatatypeException('%d labels for an axis of length %d' % (len(names), self._data.shape[axis]))

    @property
    def is_sparse(self):
        """True when the counts are held as a scipy CSR matrix."""
        return _is_sparse(self._data)

    # -- the reference's interface ---------------------------------------------------------------------
    def as_array(self):
        """Host numpy array of the counts (cmatrix.py:31-37); a dense copy for sparse counts."""
        if isinstance(self._data, torch.Tensor):
            return self._data.detach().cpu().numpy()
        if self.is_sparse:
            return self._data.toarray()
        return self._data

    def as_sparse_matrix(self, mode='csc'):
        """cmatrix.py:39-54 (the reference returns a csc matrix for either mode; 'csr' gives csr here).  Stored zeros are
        dropped, as when the matrix is built from a dense array."""
        import scipy.sparse
        if self.is_sparse:
            out = self._data.copy() if mode == 'csr' else self._data.tocsc()
            out.eliminate_zeros()
            return out
        arr = self.as_array()
        return scipy.sparse.csr_matrix(arr) if mode == 'csr' else scipy.sparse.csc_matrix(arr)

    @staticmethod
    def from_csv(filepath, delimiter=',', has_col_names=True, has_row_names=True):
        """cmatrix.py:56-79."""
        import pandas as pd
        df = pd.read_csv(filepath, sep=delimiter, header=0 if has_col_names else None,
                         index_col=0 if has_row_names else False, skip_blank_lines=True)
        return CountMatrix(df)

    @property
    def shape(self):
        return tuple(self._data.shape)

    @property
    def T(self):
        data = self._data.T.tocsr() if self.is_sparse else self._data.T
        return CountMatrix(data, row_names=self._cols, col_names=self._rows)

    @property
    def col_names(self):
        """cmatrix.py:88-95 (a RangeIndex when the matrix came without labels, like a fresh DataFrame)."""
        return np.arange(self.shape[1]) if self._cols is None else self._cols

    @property
    def row_names(self):
        """cmatrix.py:97-104."""
        return np.arange(self.shape[0]) if self._rows is None else self._rows

    def _col_index(self, key):
        hit = np.nonzero(self.col_names == key)[0]
        if not hit.size:
            raise KeyError(key)
        return int(hit[0])

    def __getitem__(self, key):
        """Column `key` by label (DataFrame semantics, cmatrix.py:109-110)."""
        j = self._col_index(key)
        if self.is_sparse:
            return self._data[:, j:j + 1].toarray()[:, 0]
        return self._data[:, j]

    def __setitem__(self, key, value):
        """cmatrix.py:106-107.  Sparse counts: a new CSR with column `key` replaced (the caller's matrix is not touched)."""
        j = self._col_index(key)
        if self.is_sparse:
            self._data = self._set_sparse_column(j, value)
            return
        self._data[:, j] = torch.as_tensor(value) if isinstance(self._data, torch.Tensor) else value

    def _set_sparse_column(self, j, value):
        import scipy.sparse
        X = self._data
        col = np.empty((X.shape[0],), dtype=X.dtype)
        col[:] = value                                             # numpy's cast and broadcast, as for a dense column
        coo = X.tocoo()
        keep = coo.col != j
        rows = np.flatnonzero(col)
        data = np.concatenate((coo.data[keep], col[rows]))
        ij = (np.concatenate((coo.row[keep], rows)), np.concatenate((coo.col[keep], np.full(rows.size, j, dtype=coo.col.dtype))))
        return canonical_csr(scipy.sparse.coo_matrix((data, ij), shape=X.shape))

    def filter_rows(self, rows, inplace=True):
        """Keep the rows with the given labels, in the given order (cmatrix.py:115-121)."""
        names = self.row_names
        pos = {k: i for i, k in enumerate(names.tolist())}
        try:
            idx = np.asarray([pos[k] for k in np.asarray(rows).tolist()], dtype=np.int64)
        except KeyError as e:
            raise KeyError('unknown row label %s' % e)
        sel = torch.as_tensor(idx, device=self._data.device) if isinstance(self._data, torch.Tensor) else idx   # CSR: row selection
        data, rn = self._data[sel], names[idx]
        if inplace:
            self._data, self._rows = data, rn
            return self
        return CountMatrix(data, row_names=rn, col_names=self._cols)

    def __repr__(self):
        return 'CountMatrix(shape=%s)' % (self.shape,)

    # -- ingest for the device path --------------------------------------------------------------------
    def as_tensor(self):
        """The counts as they are stored (device tensor or numpy array), without a copy."""
        return self._data

    @staticmethod
    def row_range(n, rank, world):
        """Contiguous block of cells owned by `rank` of `world` (blocks differ by at most one row)."""
        base, extra = divmod(int(n), int(world))
        r0 = rank * base + min(rank, extra)
        return r0, r0 + base + (1 if rank < extra else 0)

    def row_block(self, rank, world):
        """This rank's cells as a CountMatrix (a view, no copy; for sparse counts the CSR of the row range)."""
        r0, r1 = self.row_range(self.shape[0], rank, world)
        return CountMatrix(self._data[r0:r1], row_names=None if self._rows is None else self._rows[r0:r1],
                           col_names=self._cols)

    def is_uint16(self):
        """True when the counts are a uint16 array, tensor or sparse matrix: the device models may then keep them as
        uint16 in HBM (`oriana_b200.problem.counts_storage`)."""
        dt = self._data.dtype
        return dt == torch.uint16 if isinstance(self._data, torch.Tensor) else dt == np.uint16

    def narrow_dtype(self):
        """Narrowest unsigned integer type that holds every count (None: the counts are not non-negative integers
        below 2^16, keep float32).  Sparse counts: from the stored values, O(nnz) (the implicit zeros fit any type)."""
        a = self._data
        if not isinstance(a, torch.Tensor):
            return narrow_count_dtype(a.data if self.is_sparse else a)
        if a.numel() == 0:
            return torch.uint8
        lo, hi = float(a.min()), float(a.max())
        integral = (not a.dtype.is_floating_point) or bool((a == a.round()).all())
        if not integral or lo < 0 or hi >= 65536:
            return None
        return torch.uint8 if hi < 256 else torch.uint16

    def to_device(self, device='cuda', slab_rows=None, dtype=torch.float32):
        """[n, p] view of a [n, ldx] device buffer (ldx: the kernels' 16-byte row pitch), filled slab by slab.
        dtype=torch.float32: integer counts cross PCIe in their narrow type and are widened by `ori_widen_counts_f32`.
        dtype=torch.uint16 (counts that are uint16 already): the slabs are copied into the padded pitch as they are.
        Sparse counts: CSR slabs of bounded size (uint16 column indices when p <= 65536, the counts in the narrowest type
        `narrow_dtype()` allows, else float32) are expanded in HBM by `ori_expand_csr_counts`; the result is the dense
        path's, bit for bit, pad columns included."""
        from .. import _lib
        from ..problem import row_pitch
        lib = _lib.load()
        dev = torch.device(device)
        n, p = self.shape
        if dtype == torch.uint16:
            if not self.is_uint16():
                raise TypeError('to_device(dtype=torch.uint16) needs uint16 counts, got %s' % self._data.dtype)
            if self.is_sparse:
                return self._csr_to_device(dev, 2, slab_rows)
            # the copies go through int16 views: same bits, and every copy kernel handles int16
            out = torch.zeros((n, row_pitch(p, 2)), dtype=torch.int16, device=dev)
            step = slab_rows or max(1, (1 << 27) // max(1, p))
            for r in range(0, n, step):
                blk = self._data[r:r + step]
                blk = blk if isinstance(blk, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(blk))
                out[r:r + step, :p].copy_(blk.view(torch.int16))
            return out.view(torch.uint16)[:, :p]
        if dtype != torch.float32:
            raise TypeError('to_device stores counts as float32 or uint16, not %s' % dtype)
        if self.is_sparse:
            return self._csr_to_device(dev, 4, slab_rows)
        ldx = row_pitch(p)
        out = torch.zeros((n, ldx), dtype=torch.float32, device=dev)
        if isinstance(self._data, torch.Tensor) and self._data.is_cuda:
            if self.is_uint16():           # torch has no uint16 arithmetic: the library widens it
                src = self._data if self._data.stride(1) == 1 else self._data.contiguous()
                if n:
                    _lib.check(lib.ori_widen_counts_f32(src.data_ptr(), 2, max(src.stride(0), p), out.data_ptr(), ldx, n, p,
                                                        _lib.stream_ptr()))
            else:
                out[:, :p] = self._data.to(torch.float32)
            return out[:, :p]
        # uint16 torch tensors cross as they are (every count fits; torch cannot scan them for a narrower type)
        nd = torch.uint16 if isinstance(self._data, torch.Tensor) and self.is_uint16() else self.narrow_dtype()
        step = slab_rows or max(1, (1 << 26) // max(1, p))
        for r in range(0, n, step):
            blk = self._data[r:r + step]
            blk = blk if isinstance(blk, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(blk))
            if nd is None:
                out[r:r + step, :p] = blk.to(torch.float32).to(dev)
                continue
            src = blk.to(nd).contiguous().to(dev)
            rows = src.shape[0]
            _lib.check(lib.ori_widen_counts_f32(src.data_ptr(), src.element_size(), p, out[r:r + step].data_ptr(), ldx,
                                                rows, p, _lib.stream_ptr()))
        return out[:, :p]

    def _csr_to_device(self, dev, dst_bytes, slab_rows, slab_nnz=1 << 25):
        """The CSR in HBM as float32 (dst_bytes 4) or uint16 (2) X of the kernels' row pitch: slabs of at most `slab_rows`
        rows and, unless one row holds more, `slab_nnz` non-zeros, each expanded by ori_expand_csr_counts, which writes
        every element of its rows (no memset)."""
        from .. import _lib
        from ..problem import row_pitch
        lib = _lib.load()
        X = self._data
        n, p = X.shape
        ldx = row_pitch(p, dst_bytes)
        out = torch.empty((n, ldx), dtype=torch.float32 if dst_bytes == 4 else torch.int16, device=dev)
        nd = self.narrow_dtype()
        vdt, vtype = {torch.uint8: (np.uint8, _lib.ORI_CSR_U8), torch.uint16: (np.uint16, _lib.ORI_CSR_U16),
                      None: (np.float32, _lib.ORI_CSR_F32)}[nd]
        idt = np.uint16 if p <= 65536 else np.int32

        def up(a):                     # 16-bit fields cross through int16 views (same bits)
            t = torch.from_numpy(np.ascontiguousarray(a))
            return (t.view(torch.int16) if t.dtype == torch.uint16 else t).to(dev)
        ptr = X.indptr.astype(np.int64)
        max_rows = slab_rows or max(1, (1 << 26) // max(1, p))
        r0 = 0
        while r0 < n:
            r1 = max(r0 + 1, int(np.searchsorted(ptr, ptr[r0] + slab_nnz, side='right')) - 1)
            r1 = min(n, r0 + max_rows, r1)
            lo, hi = int(ptr[r0]), int(ptr[r1])
            d_ptr, d_ind, d_val = up(ptr[r0:r1 + 1]), up(X.indices[lo:hi].astype(idt)), up(X.data[lo:hi].astype(vdt))
            _lib.check(lib.ori_expand_csr_counts(d_ptr.data_ptr(), lo, d_ind.data_ptr() or None, np.dtype(idt).itemsize,
                                                 d_val.data_ptr() or None, vtype, out[r0:].data_ptr(), dst_bytes, ldx,
                                                 r1 - r0, p, _lib.stream_ptr()))
            r0 = r1
        return (out if dst_bytes == 4 else out.view(torch.uint16))[:, :p]

    def to_compact(self, pin=True):
        """Saturating uint8 + escape list (`oriana_b200.host_step.CompactCounts`) for host-streamed CAVI."""
        from ..host_step import CompactCounts
        if self.is_sparse:
            return CompactCounts.from_csr(self._data, pin=pin)
        a = self._data if isinstance(self._data, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(self._data))
        return CompactCounts.from_tensor(a, pin=pin)

    def to_sparse_counts(self, pin=True):
        """Bitmap + non-zero bytes + escape list (`oriana_b200.host_step.SparseCounts`): the streaming form of
        `as_sparse_matrix()` (cmatrix.py:100-104) for host-streamed CAVI, p / 8 + nnz bytes per cell."""
        from ..host_step import SparseCounts
        if self.is_sparse:
            return SparseCounts.from_csr(self._data, pin=pin)
        a = self._data if isinstance(self._data, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(self._data))
        return SparseCounts.from_tensor(a, pin=pin)

    def to_csr_counts(self, pin=True):
        """Row offsets + column indices + counts (`oriana_b200.host_step.CsrCounts`) for host-streamed CAVI: (index +
        count) bytes per non-zero, 3 with uint16 indices and uint8 counts -- below 1/16 non-zeros the smallest host form."""
        from ..host_step import CsrCounts
        if self.is_sparse:
            return CsrCounts.from_csr(self._data, pin=pin)
        a = self._data if isinstance(self._data, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(self._data))
        return CsrCounts.from_tensor(a, pin=pin)
