"""CAVI iterations on HOST-resident data: the reference-facing call with host buffers.

The reference keeps X and every parameter in host numpy arrays and its `step()` (base.py:54-56) reads and
writes them in place.  `HostStreamedCAVI.step()` is the same contract on the B200: every step, the count
matrix and the row-side parameters are streamed from (pinned) host memory in row slabs -- every host -> device
copy on one copy stream, so the slabs follow each other at the PCIe line rate -- the three per-slab kernels
(row pass -> U update -> gene pass) run on the slab's own compute stream while the next slab is in flight, the
updated row parameters stream back, and the gene-side update + M-step run once at the end.  Because the row
side of the iteration never needs another row (SURVEY.md section 8e iii), a slab is needed on the device
only while it is processed: the device footprint is two slabs, independent of n (out-of-core in HBM).

All arithmetic is in the CUDA library (C ABI, include/oriana_b200.h); torch is used for pinned memory,
streams and the copies.  No CPU fallback.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .problem import build_problem, gene_buffers, kernel_plan, logit_pi, row_pitch
from .sharding import RowSharding


def bind_host_thread_to_gpu(device_index):
    """Pin the calling process to the CPU cores NVML names as local to GPU `device_index` (its NUMA node), so that the
    pinned buffers allocated afterwards are first-touched -- i.e. placed -- on that node and the copy threads run next to
    them.  Returns the core list, or None when NVML / the affinity call is unavailable (nothing is changed then)."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(device_index))
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cores = [64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cores = sorted(c for c in cores if c in allowed)
        if not cores:
            return None
        os.sched_setaffinity(0, cores)
        return cores
    except Exception:
        return None


class _EscapeList:
    """The counts >= 255, which a byte cannot hold: X[row, col] = val, sorted by row (int32, int32, float32; pinned).
    Each slab's escapes follow it to the device, where `ori_scatter_counts_f32` writes them into X."""

    def _set_escapes(self, row, col, val):
        assert row.dtype == torch.int32 and col.dtype == torch.int32 and val.dtype == torch.float32
        assert row.numel() == col.numel() == val.numel()
        self.row, self.col, self.val, self._row_np = row, col, val, row.numpy()
        assert (np.diff(self._row_np) >= 0).all(), 'escape list must be sorted by row'

    @staticmethod
    def _gather_escapes(blk, r0, parts):
        """Append the escapes of the row block `blk`, whose first row is row r0, to `parts`."""
        idx = (blk >= 255).nonzero(as_tuple=False)
        if idx.numel():
            parts.append(((idx[:, 0] + r0).to(torch.int32).cpu(), idx[:, 1].to(torch.int32).cpu(),
                          blk[idx[:, 0], idx[:, 1]].to(torch.float32).cpu()))

    @staticmethod
    def _join_escapes(parts, pin):
        if not parts:                                  # no escapes: empty, unpinned
            return [torch.empty((0,), dtype=dt) for dt in (torch.int32, torch.int32, torch.float32)]
        return [t.pin_memory() if pin else t for t in (torch.cat(c) for c in zip(*parts))]

    def escapes(self, r0, r1):
        """[lo, hi) of the escapes of rows [r0, r1)."""
        return int(np.searchsorted(self._row_np, r0)), int(np.searchsorted(self._row_np, r1))

    def _with_escapes(self, X):
        """The float32 host matrix X of the byte form with the escapes written in."""
        X[self.row.long(), self.col.long()] = self.val
        return X


class CompactCounts(_EscapeList):
    """A count matrix held on the host as saturating uint8 plus an escape list for the (rare) counts >= 255:
    one byte per entry crosses PCIe per step instead of four.  Lossless: `dense()` gives the counts back.

        u8    [n, p] uint8, min(X, 255)              (pinned)
        row, col, val  escapes sorted by row: X[row, col] = val  (int32, int32, float32; pinned)
    """

    def __init__(self, u8, row, col, val):
        assert u8.dtype == torch.uint8 and u8.dim() == 2 and not u8.is_cuda
        self.u8, self.shape = u8, tuple(u8.shape)
        self._set_escapes(row, col, val)

    @classmethod
    def from_tensor(cls, X, chunk_rows=1 << 15, pin=True):
        """Encode a [n, p] count tensor (any real dtype, host or device; non-negative integers)."""
        n, p = X.shape
        pin = pin and torch.cuda.is_available()
        u8 = torch.empty((n, p), dtype=torch.uint8, pin_memory=pin)
        parts = []
        for r in range(0, n, chunk_rows):
            blk = X[r:r + chunk_rows]
            u8[r:r + chunk_rows].copy_(torch.clamp(blk, max=255).to(torch.uint8))
            cls._gather_escapes(blk, r, parts)
        return cls(u8, *cls._join_escapes(parts, pin))

    def dense(self):
        return self._with_escapes(self.u8.to(torch.float32))

    @property
    def nbytes(self):
        return self.u8.numel() + 12 * self.row.numel()


class SparseCounts(_EscapeList):
    """A count matrix held on the host the way single-cell data is shaped -- mostly zeros (cmatrix.py:100-104,
    `as_sparse_matrix`): per cell one bit per gene, the non-zero counts in gene order as saturating bytes, and the escape
    list of `CompactCounts` for the counts >= 255.  p / 8 + nnz bytes per cell cross PCIe per step instead of p
    (0.63 bytes per entry at 50 % zeros, 0.23 at 90 %); `ori_expand_bitmap_counts_f32` rebuilds the float32 slab in HBM.
    Lossless: `dense()` gives the counts back.

        bitmap  [n, W] int32, W = ceil(p / 32); bit l of word w = (X[:, 32 w + l] != 0)     (pinned)
        nz      [nnz] uint8, min(X, 255) of the non-zero entries, row-major                   (pinned)
        rowoff  [n + 1] int64, row r's bytes = nz[rowoff[r] : rowoff[r + 1]]                  (pinned)
        row, col, val  escapes sorted by row (int32, int32, float32; pinned)
    """

    def __init__(self, shape, bitmap, nz, rowoff, row, col, val):
        n, p = shape
        assert bitmap.dtype == torch.int32 and tuple(bitmap.shape) == (n, (p + 31) // 32) and not bitmap.is_cuda
        assert nz.dtype == torch.uint8 and rowoff.dtype == torch.int64 and rowoff.numel() == n + 1
        self.shape = (int(n), int(p))
        self.bitmap, self.nz, self.rowoff = bitmap, nz, rowoff
        self._off_np = rowoff.numpy()
        assert int(self._off_np[-1]) == nz.numel() and (np.diff(self._off_np) >= 0).all()
        self._set_escapes(row, col, val)

    @staticmethod
    def _pack_bits(mask):
        """[rows, p] bool -> [rows, ceil(p / 32)] int32, bit l of word w = mask[:, 32 w + l]."""
        rows, p = mask.shape
        W = (p + 31) // 32
        if W * 32 != p:
            mask = torch.nn.functional.pad(mask, (0, W * 32 - p))
        m = mask.view(rows, W, 4, 8).to(torch.int32)
        w8 = (1 << torch.arange(8, device=mask.device, dtype=torch.int32))
        b = (m * w8).sum(dim=3)                                   # four bytes per word, each 0..255
        lo = b[..., 0] | (b[..., 1] << 8) | (b[..., 2] << 16)
        return lo | torch.where(b[..., 3] >= 128, b[..., 3] - 256, b[..., 3]) << 24

    @classmethod
    def from_tensor(cls, X, chunk_rows=1 << 13, pin=True):
        """Encode a [n, p] count tensor (any real dtype, host or device; non-negative integers)."""
        n, p = X.shape
        pin = pin and torch.cuda.is_available()
        W = (p + 31) // 32
        counts = torch.empty((n,), dtype=torch.int64)
        for r in range(0, n, chunk_rows):
            counts[r:r + chunk_rows] = (X[r:r + chunk_rows] != 0).sum(dim=1).cpu()
        rowoff = torch.zeros((n + 1,), dtype=torch.int64)
        rowoff[1:] = torch.cumsum(counts, 0)
        total = int(rowoff[-1])
        bitmap = torch.empty((n, W), dtype=torch.int32, pin_memory=pin)
        nz = torch.empty((total,), dtype=torch.uint8, pin_memory=pin and total > 0)
        parts = []
        for r in range(0, n, chunk_rows):
            blk = X[r:r + chunk_rows]
            mask = blk != 0
            bitmap[r:r + chunk_rows].copy_(cls._pack_bits(mask))
            lo, hi = int(rowoff[r]), int(rowoff[min(n, r + chunk_rows)])
            nz[lo:hi].copy_(torch.clamp(blk[mask], max=255).to(torch.uint8))
            cls._gather_escapes(blk, r, parts)
        if pin:
            rowoff = rowoff.pin_memory()
        return cls((n, p), bitmap, nz, rowoff, *cls._join_escapes(parts, pin))

    def byte_range(self, r0, r1):
        return int(self._off_np[r0]), int(self._off_np[r1])

    def dense(self):
        """The float32 matrix back on the host (numpy bit unpacking; the device path is ori_expand_bitmap_counts_f32)."""
        n, p = self.shape
        bits = np.unpackbits(self.bitmap.numpy().view(np.uint8).reshape(n, -1), axis=1, bitorder='little')[:, :p].astype(bool)
        X = np.zeros((n, p), dtype=np.float32)
        X[bits] = self.nz.numpy().astype(np.float32)
        return self._with_escapes(torch.from_numpy(X))

    @property
    def nbytes(self):
        return 4 * self.bitmap.numel() + self.nz.numel() + 8 * self.rowoff.numel() + 12 * self.row.numel()

    @staticmethod
    def smaller_than_bytes(X, sample_rows=4096):
        """True when the bitmap form needs fewer bytes than one byte per entry (estimated on the leading rows)."""
        blk = X[:sample_rows]
        return float((blk != 0).float().mean()) < 0.85


class HostStreamedCAVI:

    @staticmethod
    def _default_slab(n, ldx):
        """Cells per slab: up to 32768 cells / 4 GB of float32 X, a multiple of the tensor kernels' accumulation chunk (16384 sweep
        entries, csrc/kernels_tc.cu ORI_TC_CHUNK) where the matrix is that long -- the gene-side sums of a slab are then chained
        exactly like those of a device-resident matrix, so both give the same numbers -- else a multiple of 128."""
        rows = min(n, (4 << 30) // (4 * ldx))
        if rows >= 16384:
            return min(rows // 16384 * 16384, 32768)
        return max(128, rows // 128 * 128)

    def __init__(self, X_host, k, state, dropout=True, compat_quirk=False, slab_rows=None, sharded=False,
                 process_group=None, elbo=True, keep_hyper=True, precise=False):
        """X_host: CPU tensor [n, p] (pin it for asynchronous copies), float32 like the array the reference
        feeds its kernel (zigap.py:112) or the same counts kept compactly as uint16 / uint8 (half / a quarter of
        the bytes per step over PCIe; widened to float32 on the device), or a `CompactCounts` (saturating uint8
        plus an escape list for counts >= 255).  state: host arrays a1, a2 [n, k],
        b1, b2 [p, k], alpha1, alpha2, beta1, beta2 [k] (a reference model's state vector)."""
        self._dev = _lib.require_cuda()
        self._lib = _lib.load()
        self._compact = X_host if isinstance(X_host, (CompactCounts, SparseCounts)) else None
        self._sparse = X_host if isinstance(X_host, SparseCounts) else None
        if self._sparse is not None:
            self.X, self._xbytes = None, 1             # bitmap + non-zero bytes per slab; the escapes follow each slab
            self.n, self.p = self._sparse.shape
        else:
            if self._compact is not None:
                X_host = self._compact.u8              # saturating bytes; the escapes follow each slab
            assert X_host.dtype in (torch.float32, torch.uint16, torch.uint8) and X_host.dim() == 2 and not X_host.is_cuda
            self.X = X_host
            self._xbytes = X_host.element_size()
            self.n, self.p = int(X_host.shape[0]), int(X_host.shape[1])
        self.k = int(k)
        n, p, K, dev = self.n, self.p, self.k, self._dev
        ldx = self._ldx = row_pitch(p)
        if slab_rows is None:
            slab_rows = self._default_slab(n, ldx)
        self.slab = S = int(min(max(1, slab_rows), max(1, n)))
        # slabs large enough to fill the machine take the tcgen05/TMA kernels, like the device model
        self._tensor, self._KP, plan_flags = kernel_plan(K, S * p, precise=precise)
        self._shard = RowSharding(process_group, enabled=bool(sharded or process_group is not None))
        self.n_total = self._shard.total_rows(n, dev)
        self.dropout = bool(dropout)
        self._flags = (_lib.ORI_F_DROPOUT if dropout else 0) | (_lib.ORI_F_ELBO if elbo else 0) \
            | (_lib.ORI_F_QUIRK if (compat_quirk and dropout) else 0) | plan_flags \
            | (_lib.ORI_F_FIXED_CHAIN if n > S else 0)
        self.h2d_bytes = 0
        self.d2h_bytes = 0

        pin = torch.cuda.is_available()

        def host(a, dtype, shape):
            t = torch.as_tensor(np.asarray(a), dtype=dtype).reshape(shape).contiguous()
            return t.pin_memory() if pin else t
        # host-resident state (what a caller reads between steps)
        self.a1 = host(state['a1'], torch.float32, (n, K)); self.a2 = host(state['a2'], torch.float32, (n, K))
        self.b1 = host(state['b1'], torch.float32, (p, K)); self.b2 = host(state['b2'], torch.float32, (p, K))
        self.hyper = host(np.stack([state[q] for q in ('alpha1', 'alpha2', 'beta1', 'beta2')]), torch.float64, (4, K))
        self.pi_d = host(np.zeros(p), torch.float64, (p,))
        self.lp = host(np.full(p, -np.inf), torch.float32, (p,))
        self.pfloor = host(np.zeros(p), torch.float32, (p,))
        self.scal = host(np.zeros(_lib.SCAL_SLOTS), torch.float64, (_lib.SCAL_SLOTS,))
        self.elbo_trace = []
        self.iterations = 0

        f32 = dict(dtype=torch.float32, device=dev); f64 = dict(dtype=torch.float64, device=dev)
        # device: gene side + reduction buffers (small), two sets of slab buffers.  lp, pfloor and pi_d exist with or
        # without dropout (every step uploads lp and pfloor)
        KP = self._KP
        g = self._g = gene_buffers(p, K, KP, dev, dropout=True, sparse=False, trace_cap=4)
        g['xcol'] = torch.zeros((p,), **f32)
        self._slabs = []
        for _ in range(2 if n > S else 1):
            s = dict(X=torch.zeros((S, ldx), **f32), red64=torch.zeros_like(g['red64']),
                     acc64=torch.zeros_like(g['red64']), xrow=torch.zeros((S,), **f32),
                     cs64=torch.zeros((p,), **f64), csacc=torch.zeros((p,), **f64),
                     tc_ws=torch.empty((int(self._lib.ori_tc_workspace_floats(S, p, KP)) + 32,), **f32) if self._tensor else None)
            for name in ('a1', 'a2', 'Zi', 'a2s', 'eUw'):
                s[name] = torch.zeros((S, KP), **f32)
            s['U_hat'], s['eU'] = [[torch.zeros((S, KP), **f32) for _ in range(2)] for _ in range(2)]
            if self._sparse is not None:
                off = self._sparse._off_np
                nzcap = max(int(off[min(n, r + S)] - off[r]) for r in range(0, n, S)) + 16
                s['bm'] = torch.zeros((S, (p + 31) // 32), dtype=torch.int32, device=dev)
                s['nz'] = torch.zeros((nzcap,), dtype=torch.uint8, device=dev)
                s['off'] = torch.zeros((S + 1,), dtype=torch.int64, device=dev)
            elif self._xbytes != 4:
                s['Xq'] = torch.zeros((S, p), dtype=X_host.dtype, device=dev)      # compact counts as they arrive
            if self._compact is not None:
                cap = max(1024, int(4 * self._compact.row.numel() * S / max(1, n)) + 1024)
                s['esc'] = [torch.zeros((cap,), dtype=torch.int32, device=dev), torch.zeros((cap,), dtype=torch.int32, device=dev),
                            torch.zeros((cap,), dtype=torch.float32, device=dev)]
            s['stage'] = torch.zeros((2, S, K), **f32)     # unpadded a1|a2 as they travel
            self._slabs.append(s)
        self._streams = [torch.cuda.Stream(device=dev) for _ in self._slabs]
        self._copy_stream = torch.cuda.Stream(device=dev)
        self._Pg = self._problem(None, 0)
        self._keep_hyper = keep_hyper
        self._init_pass()
        # mid-run state (e.g. this class's own state_dict(), or a device model's): D_hat of the first step is the sigmoid
        # generated by pi_prev (zigap.py:131-132), not the indicator of a freshly constructed model (zigap.py:77)
        it0 = int(state.get('iterations', 0) or 0)
        if self.dropout and state.get('pi_prev') is not None:
            self.pi_d.copy_(torch.as_tensor(np.asarray(state['pi_prev'], dtype=np.float64).reshape(p)))
            lp, pfloor = logit_pi(self.pi_d)
            self.lp.copy_(lp); self.pfloor.copy_(pfloor)
        elif self.dropout and it0 > 0:
            raise ValueError('a mid-run state (iterations=%d) must carry "pi_prev", the Bernoulli prior that generated its '
                             'dropout posterior (SURVEY.md section 8c)' % it0)
        self.iterations = it0

    # ------------------------------------------------------------------------------------------------
    def _problem(self, s, rows):
        """The problem of one slab, or (s=None) of the gene side alone: ori_problem_check wants the row pointers even then,
        so they point at a gene-side buffer."""
        if s is None:
            d = self._g['red32']
            row = dict(a1=d, a2=d, Zi=d, a2s=d, eUw=d, U_hat=(d, d), eU=(d, d))
        else:
            row = {q: s[q] for q in ('X', 'a1', 'a2', 'U_hat', 'eU', 'Zi', 'a2s', 'eUw', 'xrow', 'tc_ws')}
        return build_problem(n_rows=rows, n_total=self.n_total, ldx=self._ldx, p=self.p, K=self.k, KP=self._KP,
                             flags=self._flags, trace_cap=4, **self._g, **row)

    def _call(self, name, P, *args, stream=None):
        st = ctypes.c_void_p((stream or torch.cuda.current_stream()).cuda_stream)
        _lib.check(getattr(self._lib, name)(ctypes.byref(P), *args, st))

    def _upload_genes(self):
        g, K = self._g, self.k
        for name in ('b1', 'b2'):
            g[name][:, :K].copy_(getattr(self, name), non_blocking=True)
        g['hyper'].copy_(self.hyper, non_blocking=True)
        g['lp'].copy_(self.lp, non_blocking=True); g['pfloor'].copy_(self.pfloor, non_blocking=True)
        g['scal'].copy_(self.scal, non_blocking=True)
        self.h2d_bytes += 2 * self.p * K * 4 + 4 * K * 8 + self.p * 8 + _lib.SCAL_SLOTS * 8

    def _copy_slab(self, s, r0, rows):
        """Host -> device copies of one slab (current stream = the copy stream): X in the form the host holds it, the escape
        list, the row parameters.  Returns what `_finish_upload` needs."""
        K, p = self.k, self.p
        info = dict(lo=0, cnt=0)
        xbytes_sent = rows * p * self._xbytes
        if self._xbytes == 4:
            s['X'][:rows, :p].copy_(self.X[r0:r0 + rows], non_blocking=True)
        elif self._sparse is not None:
            sp = self._sparse
            lo, hi = sp.byte_range(r0, r0 + rows)
            s['bm'][:rows].copy_(sp.bitmap[r0:r0 + rows], non_blocking=True)
            if hi > lo:
                s['nz'][:hi - lo].copy_(sp.nz[lo:hi], non_blocking=True)
            s['off'][:rows + 1].copy_(sp.rowoff[r0:r0 + rows + 1], non_blocking=True)
            info['lo'] = lo
            xbytes_sent = rows * s['bm'].shape[1] * 4 + (hi - lo) + (rows + 1) * 8
        else:
            s['Xq'][:rows].copy_(self.X[r0:r0 + rows], non_blocking=True)
        if self._compact is not None:
            lo, hi = self._compact.escapes(r0, r0 + rows)
            cnt = info['cnt'] = hi - lo
            if cnt:
                if cnt > s['esc'][0].numel():          # a slab with unusually many large counts: grow its buffers
                    s['esc'] = [torch.zeros((2 * cnt,), dtype=t.dtype, device=t.device) for t in s['esc']]
                for dst, src in zip(s['esc'], (self._compact.row, self._compact.col, self._compact.val)):
                    dst[:cnt].copy_(src[lo:hi], non_blocking=True)
                self.h2d_bytes += 12 * cnt
        s['stage'][0, :rows].copy_(self.a1[r0:r0 + rows], non_blocking=True)
        s['stage'][1, :rows].copy_(self.a2[r0:r0 + rows], non_blocking=True)
        self.h2d_bytes += xbytes_sent + 2 * rows * K * 4
        return info

    def _finish_upload(self, s, r0, rows, info):
        """Device side of the upload (current stream = the slab's compute stream): compact counts -> float32 X, escapes, row
        sums, padded row parameters."""
        K, p = self.k, self.p
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        if self._sparse is not None:
            _lib.check(self._lib.ori_expand_bitmap_counts_f32(s['bm'].data_ptr(), s['bm'].shape[1], s['nz'].data_ptr(),
                                                              s['off'].data_ptr(), info['lo'], s['X'].data_ptr(), self._ldx,
                                                              rows, p, st))
        elif self._xbytes != 4:
            _lib.check(self._lib.ori_widen_counts_f32(s['Xq'].data_ptr(), self._xbytes, p, s['X'].data_ptr(), self._ldx,
                                                      rows, p, st))
        if info['cnt']:
            _lib.check(self._lib.ori_scatter_counts_f32(s['X'].data_ptr(), self._ldx, r0, rows, p, s['esc'][0].data_ptr(),
                                                        s['esc'][1].data_ptr(), s['esc'][2].data_ptr(), info['cnt'], st))
        # row sums of the slab (ELBO scale term, include/oriana_b200.h xrow): X is in HBM anyway
        _lib.check(self._lib.ori_row_sums_f32(s['X'].data_ptr(), self._ldx, rows, p, s['xrow'].data_ptr(), st))
        s['a1'][:rows, :K] = s['stage'][0, :rows]; s['a2'][:rows, :K] = s['stage'][1, :rows]

    def _slab_loop(self, body):
        """Slabs in order.  ALL host -> device copies go through one copy stream, so they run one after the other at the
        full PCIe rate while the previous slab's kernels run on its compute stream (issued from two compute streams, the
        copies of two slabs shared the link and both slabs then computed with the link idle: 10 instead of 7.5 ms per
        slab, scripts/gpu_e2e_timeline.py).  A slab's buffers are refilled once its previous occupant's kernels and
        device -> host copies are done."""
        main = torch.cuda.current_stream()
        ready = torch.cuda.Event(); ready.record(main)
        copy_st = self._copy_stream
        copy_st.wait_event(ready)
        done = [None] * len(self._slabs)
        for i, r0 in enumerate(range(0, self.n, self.slab)):
            b = i % len(self._slabs)
            st, s = self._streams[b], self._slabs[b]
            if i < len(self._slabs):
                st.wait_event(ready)
            rows = min(self.slab, self.n - r0)
            if done[b] is not None:
                copy_st.wait_event(done[b])
            with torch.cuda.stream(copy_st):
                info = self._copy_slab(s, r0, rows)
                arrived = torch.cuda.Event(); arrived.record(copy_st)
            st.wait_event(arrived)
            with torch.cuda.stream(st):
                self._finish_upload(s, r0, rows, info)
                body(s, self._problem(s, rows), r0, rows, st)
                done[b] = torch.cuda.Event(); done[b].record(st)
        main.wait_stream(copy_st)
        for st in self._streams:
            main.wait_stream(st)

    def _init_pass(self):
        """Constant statistics of X + expectations of the initial state + (optionally) the first M-step
        (base.py:43-52), streamed once."""
        g = self._g
        self._upload_genes()
        g['red64'].zero_()
        Pg = self._Pg

        def body(s, P, r0, rows, st):
            P.red64 = s['red64'].data_ptr()
            self._call('ori_count_stats', P, stream=st)            # zero-fills its red64, then counts
            self._call('ori_row_update', P, 0, 2, stream=st)       # + sum_i log U_hat, sum_i U_hat, entropy
            s['acc64'].add_(s['red64'])                            # per-stream partial (no cross-stream RMW)
            _lib.check(self._lib.ori_column_sums_f64(s['X'].data_ptr(), self._ldx, rows, self.p, s['cs64'].data_ptr(),
                                                     ctypes.c_void_p(st.cuda_stream)))
            s['csacc'].add_(s['cs64'])
        for s in self._slabs:
            s['acc64'].zero_(); s['csacc'].zero_()
        self._slab_loop(body)
        cs = torch.zeros((self.p,), dtype=torch.float64, device=self._dev)
        for s in self._slabs:
            g['red64'].add_(s['acc64']); cs.add_(s['csacc'])
        self._shard.allreduce_sum(g['red64'])
        g['xcol'].copy_(self._shard.allreduce_sum(cs).to(torch.float32))
        self._call('ori_init_expectations', Pg, 0)                 # n_rows = 0: gene side only
        self._call('ori_mstep', Pg, _lib.ORI_M_INIT_KEEP if self._keep_hyper else _lib.ORI_M_INIT)
        self._download_genes()
        torch.cuda.current_stream().synchronize()

    def _download_genes(self):
        g, K = self._g, self.k
        self.hyper.copy_(g['hyper'], non_blocking=True)
        self.scal.copy_(g['scal'], non_blocking=True)
        self.d2h_bytes += 4 * K * 8 + _lib.SCAL_SLOTS * 8
        if self.dropout:
            self.pi_d.copy_(g['pi_d'], non_blocking=True)
            self.lp.copy_(g['lp'], non_blocking=True); self.pfloor.copy_(g['pfloor'], non_blocking=True)
            self.d2h_bytes += self.p * 16

    # ------------------------------------------------------------------------------------------------
    def step(self):
        """One CAVI iteration (base.py:54-56), host buffers in, host buffers out.  Returns the ELBO of the
        state the step started from (it falls out of the row pass)."""
        g, K, quirk = self._g, self.k, bool(self._flags & _lib.ORI_F_QUIRK)
        self._upload_genes()
        Pg = self._Pg
        self._call('ori_init_expectations', Pg, 0)                  # V_hat, eV from (b1, b2): gene side only
        g['red32'].zero_(); g['red64'].zero_()

        def body(s, P, r0, rows, st):
            self._call('ori_row_update', P, 0, 3, stream=st)        # U_hat, eU of the incoming (a1, a2)
            s['Zi'].zero_(); s['a2s'].zero_()
            self._call('ori_pass_rows', P, 0, stream=st)
            self._call('ori_row_update', P, 0, 1, stream=st)
            self._call('ori_pass_genes', P, 0, stream=st)
            s['stage'][0, :rows] = s['a1'][:rows, :K]; s['stage'][1, :rows] = s['a2'][:rows, :K]
            self.a1[r0:r0 + rows].copy_(s['stage'][0, :rows], non_blocking=True)
            self.a2[r0:r0 + rows].copy_(s['stage'][1, :rows], non_blocking=True)
            self.d2h_bytes += 2 * rows * K * 4
        self._slab_loop(body)
        if self._shard.enabled:
            self._shard.allreduce_sum(g['red32']); self._shard.allreduce_sum(g['red64'])
        self._call('ori_gene_update', Pg, 1)
        self._call('ori_mstep', Pg, _lib.ORI_M_STEP)
        self.b1.copy_(g['b1'][:, :K], non_blocking=True); self.b2.copy_(g['b2'][:, :K], non_blocking=True)
        self.d2h_bytes += 2 * self.p * K * 4
        self._download_genes()
        torch.cuda.current_stream().synchronize()                   # results are on the host when we return
        self.iterations += 1
        e = float(self.scal[4])
        self.elbo_trace.append(e)
        return e

    def state_dict(self):
        s = dict(a1=self.a1.numpy().astype(np.float64), a2=self.a2.numpy().astype(np.float64),
                 b1=self.b1.numpy().astype(np.float64), b2=self.b2.numpy().astype(np.float64))
        for i, q in enumerate(('alpha1', 'alpha2', 'beta1', 'beta2')):
            s[q] = self.hyper[i].numpy().copy()
        if self.dropout:
            s['pi_prev'] = self.pi_d.numpy().copy()      # generates the current D_hat (zigap.py:131-132)
        s['iterations'] = self.iterations
        return s
