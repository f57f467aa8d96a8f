"""Count-matrix container (oriana/singlecell/cmatrix.py:12-121): the hand-off to the models, and the ingest step in
front of the CAVI path (SURVEY.md 8f row 3).

Accepts what the reference accepts (numpy array, pandas DataFrame) plus a torch tensor that may already be resident
in HBM (this rank's row block of a sharded matrix).  Anything else raises DatatypeException (cmatrix.py:25-29).
The reference keeps a DataFrame; here the counts stay in the array they arrived in (no copy) and the row / column
labels are kept beside them, so that the label-based calls (`cm['gene']`, `filter_rows`, `row_names`, `col_names`)
behave like the reference's without a pandas round trip of the matrix.

Ingest helpers with no counterpart in the reference: `row_block` (the contiguous cell range a rank owns, SURVEY.md
8e), `to_device` (the matrix in HBM with the 16-byte row pitch the kernels want, uploaded in slabs: float32, widened on
the device from the narrowest integer type that holds the counts, or uint16 as it is for counts handed in as uint16),
`to_compact` (saturating uint8 + escape list for host-streamed runs).
"""
import numpy as np
import torch

from ..exceptions import DatatypeException


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
        else:
            raise DatatypeException('Incompatible type %s' % type(data))
        for names, axis in ((self._rows, 0), (self._cols, 1)):
            if names is not None and len(names) != self._data.shape[axis]:
                raise DatatypeException('%d labels for an axis of length %d' % (len(names), self._data.shape[axis]))

    # -- the reference's interface ---------------------------------------------------------------------
    def as_array(self):
        """Host numpy array of the counts (cmatrix.py:31-37)."""
        if isinstance(self._data, torch.Tensor):
            return self._data.detach().cpu().numpy()
        return self._data

    def as_sparse_matrix(self, mode='csc'):
        """cmatrix.py:39-54 (the reference returns a csc matrix for either mode; 'csr' gives csr here)."""
        import scipy.sparse
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
        return CountMatrix(self._data.T, row_names=self._cols, col_names=self._rows)

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
        return self._data[:, self._col_index(key)]

    def __setitem__(self, key, value):
        """cmatrix.py:106-107."""
        self._data[:, self._col_index(key)] = torch.as_tensor(value) if isinstance(self._data, torch.Tensor) else value

    def filter_rows(self, rows, inplace=True):
        """Keep the rows with the given labels, in the given order (cmatrix.py:115-121)."""
        names = self.row_names
        pos = {k: i for i, k in enumerate(names.tolist())}
        try:
            idx = np.asarray([pos[k] for k in np.asarray(rows).tolist()], dtype=np.int64)
        except KeyError as e:
            raise KeyError('unknown row label %s' % e)
        sel = torch.as_tensor(idx, device=self._data.device) if isinstance(self._data, torch.Tensor) else idx
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
        """This rank's cells as a CountMatrix (a view, no copy)."""
        r0, r1 = self.row_range(self.shape[0], rank, world)
        return CountMatrix(self._data[r0:r1], row_names=None if self._rows is None else self._rows[r0:r1],
                           col_names=self._cols)

    def is_uint16(self):
        """True when the counts are a uint16 array or tensor: the device models may then keep them as uint16 in HBM
        (`oriana_b200.problem.counts_storage`)."""
        dt = self._data.dtype
        return dt == torch.uint16 if isinstance(self._data, torch.Tensor) else dt == np.uint16

    def narrow_dtype(self):
        """Narrowest unsigned integer type that holds every count (None: the counts are not non-negative integers
        below 2^16, keep float32)."""
        a = self._data
        if isinstance(a, torch.Tensor):
            if a.numel() == 0:
                return torch.uint8
            lo, hi = float(a.min()), float(a.max())
            integral = (not a.dtype.is_floating_point) or bool((a == a.round()).all())
        else:
            if a.size == 0:
                return torch.uint8
            lo, hi = float(a.min()), float(a.max())
            integral = np.issubdtype(a.dtype, np.integer) or bool((a == np.round(a)).all())
        if not integral or lo < 0 or hi >= 65536:
            return None
        return torch.uint8 if hi < 256 else torch.uint16

    def to_device(self, device='cuda', slab_rows=None, dtype=torch.float32):
        """[n, p] view of a [n, ldx] device buffer (ldx: the kernels' 16-byte row pitch), filled slab by slab.
        dtype=torch.float32: integer counts cross PCIe in their narrow type and are widened by `ori_widen_counts_f32`.
        dtype=torch.uint16 (counts that are uint16 already): the slabs are copied into the padded pitch as they are."""
        from .. import _lib
        from ..problem import row_pitch
        lib = _lib.load()
        dev = torch.device(device)
        n, p = self.shape
        if dtype == torch.uint16:
            if not self.is_uint16():
                raise TypeError('to_device(dtype=torch.uint16) needs uint16 counts, got %s' % self._data.dtype)
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

    def to_compact(self, pin=True):
        """Saturating uint8 + escape list (`oriana_b200.host_step.CompactCounts`) for host-streamed CAVI."""
        from ..host_step import CompactCounts
        a = self._data if isinstance(self._data, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(self._data))
        return CompactCounts.from_tensor(a, pin=pin)

    def to_sparse_counts(self, pin=True):
        """Bitmap + non-zero bytes + escape list (`oriana_b200.host_step.SparseCounts`): the streaming form of
        `as_sparse_matrix()` (cmatrix.py:100-104) for host-streamed CAVI, p / 8 + nnz bytes per cell."""
        from ..host_step import SparseCounts
        a = self._data if isinstance(self._data, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(self._data))
        return SparseCounts.from_tensor(a, pin=pin)
