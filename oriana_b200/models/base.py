"""`FactorModel` -- base class of the Gamma-Poisson factor models (oriana/models/base.py:13-130).

Same constructor, hooks and `step()` as the reference; the state lives in HBM and every update runs in the
CUDA library (`include/oriana_b200.h`).  One CAVI iteration (`step()`, base.py:54-56) is

    update_variational_parameters()   E-step  zigap.py:97-141 / gap.py:82-115
        row pass  -> U update -> gene pass -> [allreduce over ranks] -> V update
    update_prior_hyper_parameters()   M-step  zigap.py:143-158 / gap.py:117-129

Differences that are visible to a caller, all forced by scale (SURVEY.md sections 7-8):
  * D_hat / p_d (n x p) is never stored: it is recomputed inside both passes from (U_hat, V_hat, pi).
    `model.D_hat`, `model.p_d` materialise it on request; `model.pi_d` (which the reference refreshes at the
    end of each step from the stored p_d) is produced by the NEXT row pass, or by a flush pass when read.
  * UV = U V^T (n x p float64) is not materialised by `step()`; call `model.UV.forward()` if you want it.
  * the model can own a row block of a larger matrix (`sharded=True`): only the gene-side sums are
    all-reduced (NCCL) per iteration.
  * an ELBO trace is kept (`model.elbo_trace`, `model.elbo()`); the reference has none.
"""
from abc import ABCMeta, abstractmethod
import ctypes

import numpy as np
import torch

from .. import _lib
from .. import problem as _problem
from ..dims import Dimensions
from ..nodes import Einsum
from ..parameters import Parameter
from ..problem import build_problem, gene_buffers, kernel_plan, row_pitch
from ..sharding import RowSharding
from ..singlecell.cmatrix import CountMatrix


class DeviceView(Parameter):
    """A `Parameter` whose storage is a view of the model's device state.  Reads return float64 host
    copies (the reference keeps parameters in float64, parameters.py:11); writes go to HBM and make the
    model re-derive its expectations before the next step."""

    def __init__(self, owner, getter, on_write=True):
        self._owner = owner
        self._getter = getter
        self._on_write = on_write

    @property
    def _t(self):
        return self._getter()

    @property
    def tensor(self):
        return self._getter()

    def asarray(self):
        return self._getter().detach().to(torch.float64).cpu().numpy()

    def __setitem__(self, key, value):
        Parameter.__setitem__(self, key, value)
        if self._on_write:
            self._owner._dirty = True

    @property
    def buffer(self):
        return self.asarray()

    @buffer.setter
    def buffer(self, data):
        self[...] = data


class FactorModel(metaclass=ABCMeta):

    _dropout = False     # ZIGaP sets this
    _sparse = False      # SparseZIGaP sets this
    _X_SLAB_ENTRIES = 1 << 25   # matrix entries per row slab of the metrics and of the uint16 NMF warm start

    def __init__(self, cmatrix, k=2, use_factors=True, *, state=None, compat_quirk=False, sharded=False,
                 process_group=None, elbo=True, trace_cap=4096, force_simt=False, tensor=None, nmf=None, graphs=False,
                 keep_hyper=True, precise=False, emulate_underflow=False, deterministic=False):
        self._dev = _lib.require_cuda()
        self._lib = _lib.load()
        _lib.check(self._lib.ori_device_check(self._dev.index or 0))
        if not isinstance(cmatrix, CountMatrix):
            cmatrix = CountMatrix(cmatrix)
        self.cmatrix = cmatrix

        # dimensions (base.py:21-24)
        self.k = int(k)
        self.n = int(cmatrix.shape[0])
        self.m = self.p = int(cmatrix.shape[1])
        self.dims = Dimensions({'n': self.n, 'm': self.m, 'p': self.p, 'k': self.k})
        self.precise = bool(precise)
        self._tensor, self._KP, plan_flags = kernel_plan(self.k, self.n * self.p, precise=self.precise, tensor=tensor,
                                                         force_simt=force_simt, sparse=self._sparse)
        self._shard = RowSharding(process_group if (sharded or process_group is not None) else None,
                                  enabled=bool(sharded or process_group is not None))
        self.n_total = self._shard.total_rows(self.n, self._dev)
        self._flags = (_lib.ORI_F_DROPOUT if self._dropout else 0) | (_lib.ORI_F_ELBO if elbo else 0) \
            | (_lib.ORI_F_QUIRK if (compat_quirk and self._dropout) else 0) | (_lib.ORI_F_SPARSE if self._sparse else 0) \
            | (_lib.ORI_F_DEVICE_ITER if graphs else 0) | plan_flags
        # graphs=True: step() replays one captured CUDA graph per generation parity (every launch of the iteration and
        # the memsets) instead of ~15 separate launches; single rank only
        if graphs and (sharded or process_group is not None):
            raise ValueError('graphs=True is a single-rank feature: capturing the NCCL all-reduces of a sharded step '
                             'is not supported')
        # emulate_underflow=True: reproduce the reference's float32 exp underflow in the multinomial step (zigap.py:86-90,
        # gap.py:73-76: terms with log_U_hat + log_V_hat <= -103.97 are 0 there; an entry whose terms all are assigns its
        # count to no component).  Off by default, like the quirk: the default keeps the exact ratios.
        self.emulate_underflow = bool(emulate_underflow)
        # deterministic=True: every floating-point sum is formed in a fixed order (ORI_F_DETERMINISTIC): two runs from the same
        # state on the same device agree bit for bit
        self.deterministic = bool(deterministic)
        if self.deterministic:
            if not self._tensor and self.n * self.p > (1 << 26):
                raise ValueError('deterministic=True on the CUDA-core kernels is limited to 2^26 matrix entries')
            if self.emulate_underflow:
                raise ValueError('deterministic=True and emulate_underflow=True cannot be combined')
            self._flags |= _lib.ORI_F_DETERMINISTIC
        self._graphs = {} if graphs else None
        self.graph_replays = 0
        self._graph_kernels = 0
        self.compat_quirk = bool(compat_quirk and self._dropout)
        self._trace_cap = int(trace_cap)
        if nmf not in (None, 'host', 'device'):
            raise ValueError("nmf must be None, 'host' or 'device'")
        self._nmf_mode = nmf
        # with state=: keep the state's alpha / beta (a model copied mid-run or out of a reference model, whose constructor
        # has already run its M-step) or, keep_hyper=False, run the constructor's M-step on the expectations (base.py:52)
        self._keep_hyper_arg = bool(keep_hyper)
        self._gen = 0
        self._iter = 0
        self._dirty = False
        self._pi_stale = False
        self._D_cache = None
        self._started = False
        self._timers = None

        self._allocate(cmatrix)

        # model graph (base.py:27-31); UV is NOT forwarded here (n x p float64)
        self.U = self.build_u_node()
        self.V = self.build_v_node()
        self.UV = Einsum('nk,mk->nm', self.U, self.V, name='UV')
        self.X = self.build_x_node(self.cmatrix, self.UV)
        self.define_variational_distribution()

        self.use_factors = use_factors
        if state is not None:
            self.load_state(state)
        else:
            if use_factors:
                self._nmf_warm_start()
            self.initialize_parameters()

    # ------------------------------------------------------------------------------------------------
    def _allocate(self, cmatrix):
        dev, n, p, K, KP = self._dev, self.n, self.p, self.k, self._KP
        f32 = dict(dtype=torch.float32, device=dev)
        f64 = dict(dtype=torch.float64, device=dev)
        # counts handed in as uint16 stay uint16 in HBM (ORI_F_X_U16, half the bytes) when float32 would not fit the device
        u16 = _problem.counts_storage(cmatrix.is_uint16(), n, p, KP, torch.cuda.mem_get_info(dev)[0]) == torch.uint16
        xdt, esz = (torch.uint16, 2) if u16 else (torch.float32, 4)
        if u16:
            self._flags |= _lib.ORI_F_X_U16
        ldx = row_pitch(p, esz)
        src = cmatrix.as_tensor()
        if isinstance(src, torch.Tensor) and src.is_cuda and src.dtype == xdt \
                and src.shape[1] == p and src.stride(1) == 1 and src.stride(0) % (16 // esz) == 0 \
                and src.stride(0) >= p and src.data_ptr() % 16 == 0:
            self._X = src                      # adopt a resident row block without copying it
            ldx = src.stride(0) if n > 1 else max(ldx, src.stride(0))
            self._Xfull = None
        else:
            # ingest (cmatrix.py -> HBM): float32 storage: slabs cross PCIe in the narrowest integer type that holds the
            # counts and are widened on the device; no n x p float32 copy on the host.  uint16 storage: copied as is
            self._X = cmatrix.to_device(dev, dtype=xdt)
            self._Xfull = self._X
        self._ldx = ldx

        def rowf():
            return torch.zeros((n, KP), **f32)

        def genef():
            return torch.zeros((p, KP), **f32)
        self._a1, self._a2, self._Zi = rowf(), rowf(), rowf()
        self._Uhat, self._eU = [rowf(), rowf()], [rowf(), rowf()]
        self._a2s = rowf() if self._dropout else None
        g = gene_buffers(p, K, KP, dev, dropout=self._dropout, sparse=self._sparse, trace_cap=self._trace_cap)
        self._b1, self._b2, self._Vhat, self._eV, self._red32 = g['b1'], g['b2'], g['V_hat'], g['eV'], g['red32']
        self._lp, self._pfloor, self._pi, self._hyper = g['lp'], g['pfloor'], g['pi_d'], g['hyper']
        self._red64, self._scal, self._trace = g['red64'], g['scal'], g['elbo_trace']
        # row sums of this rank's X and column sums of the whole X: the ELBO takes the per-row / per-gene scales of
        # the exp(E[log .]) operands back through them (include/oriana_b200.h, xrow / xcol)
        self._xrow = xcol = None
        if self._flags & _lib.ORI_F_ELBO:
            self._xrow = torch.zeros((max(n, 1),), **f32)
            cs = torch.zeros((p,), **f64)
            self._x_sums(cs, rows=self._xrow)
            xcol = self._shard.allreduce_sum(cs).to(torch.float32)
        under = self.emulate_underflow
        # every array the problem points at: this dict owns the memory of those the model has no name for
        self._arrays = dict(
            X=self._X, a1=self._a1, a2=self._a2, U_hat=self._Uhat, eU=self._eU, Zi=self._Zi, a2s=self._a2s,
            eUw=rowf() if (self._flags & _lib.ORI_F_QUIRK) else None, xrow=self._xrow, xcol=xcol,
            thrU=torch.zeros((2, max(n, 1)), **f32) if under else None, thrV=torch.zeros((p,), **f32) if under else None,
            tc_ws=torch.empty((int(self._lib.ori_tc_workspace_floats(n, p, KP)) + 32,), **f32) if self._tensor else None,
            det_ws=torch.zeros((int(self._lib.ori_det_workspace_doubles(n, p, KP)) + 8,), **f64) if self.deterministic else None,
            **g, **self._extra_fields(rowf, genef))
        P = self._P = build_problem(n_rows=n, n_total=self.n_total, ldx=ldx, p=p, K=K, KP=KP, flags=self._flags,
                                   trace_cap=self._trace_cap, **self._arrays)
        _lib.check(self._lib.ori_problem_check(ctypes.byref(P)))
        self.uses_tensor_path = bool(self._lib.ori_uses_tensor_path(ctypes.byref(P)))
        if self._tensor and not self.uses_tensor_path and n > 0:
            raise _lib.OrianaB200Error('tensor path requested but not available on this device / driver')

        K_ = K
        self.a1 = DeviceView(self, lambda: self._a1[:, :K_])
        self.a2 = DeviceView(self, lambda: self._a2[:, :K_])
        self.b1 = DeviceView(self, lambda: self._b1[:, :K_])
        self.b2 = DeviceView(self, lambda: self._b2[:, :K_])
        self.alpha1 = DeviceView(self, lambda: self._hyper[0])
        self.alpha2 = DeviceView(self, lambda: self._hyper[1])
        self.beta1 = DeviceView(self, lambda: self._hyper[2])
        self.beta2 = DeviceView(self, lambda: self._hyper[3])

    @property
    def counts_dtype(self):
        """Storage of the count matrix in HBM: torch.uint16 for counts handed in as uint16, torch.float32 otherwise."""
        return torch.uint16 if self._flags & _lib.ORI_F_X_U16 else torch.float32

    def _x_sums(self, cols, rows=None):
        """Column sums (float64) of this rank's X into `cols` and, given `rows`, its row sums (float32), by the entry
        points of X's storage type."""
        u16 = bool(self._flags & _lib.ORI_F_X_U16)
        args = (self._X.data_ptr(), self._ldx, self.n, self.p)
        if rows is not None:
            fn = self._lib.ori_row_sums_u16_f32 if u16 else self._lib.ori_row_sums_f32
            _lib.check(fn(*args, rows.data_ptr(), _lib.stream_ptr()))
        fn = self._lib.ori_column_sums_u16_f64 if u16 else self._lib.ori_column_sums_f64
        _lib.check(fn(*args, cols.data_ptr(), _lib.stream_ptr()))

    def _x_slabs(self, rows):
        """(first row, float32 [r, p] block) over this rank's X.  float32 storage: views of X, `rows` ignored (one block).
        uint16 storage: slabs of at most `rows` cells widened by `ori_widen_counts_f32` into one float32 scratch that
        every slab reuses -- the whole matrix is never widened at once."""
        if not self._flags & _lib.ORI_F_X_U16:
            yield 0, self._X
            return
        rows = max(1, min(int(rows), self.n))
        ldw = row_pitch(self.p)
        scratch = torch.empty((rows, ldw), dtype=torch.float32, device=self._dev)
        for r in range(0, self.n, rows):
            nr = min(rows, self.n - r)
            _lib.check(self._lib.ori_widen_counts_f32(self._X[r:].data_ptr(), 2, self._ldx, scratch.data_ptr(), ldw, nr,
                                                      self.p, _lib.stream_ptr()))
            yield r, scratch[:nr, :self.p]

    def _extra_fields(self, rowf, genef):
        """Hook for model-specific device state (SparseZIGaP): further `ori_problem_t` fields by name."""
        return {}

    def _call(self, name, *args):
        self._P.iter = self._iter
        _lib.check(getattr(self._lib, name)(ctypes.byref(self._P), *args, _lib.stream_ptr()))

    # ------------------------------------------------------------------------------------------------
    def _nmf_warm_start(self):
        """`use_factors=True`: the reference seeds a1, b1 with sklearn NMF factors of X (base.py:38-40).  Matrices the
        host can factorise on one rank go through sklearn exactly like the reference; larger or row-sharded ones
        (where the reference cannot run at all) are factorised in HBM (`_nmf_device`, SURVEY.md 8f row 4)."""
        mode = self._nmf_mode
        if mode is None:
            mode = 'device' if (self._shard.enabled or self.n * self.p > 50_000_000) else 'host'
        if mode == 'host':
            if self._shard.enabled:
                raise ValueError("nmf='host' needs the whole matrix on one rank")
            from sklearn.decomposition import NMF
            model = NMF(n_components=self.k)
            X = self.cmatrix.as_array()
            self._nmf_U = model.fit_transform(X)
            self._nmf_V = model.components_.T
        else:
            self._nmf_U, self._nmf_V = self._nmf_device()

    def _nmf_device(self, iters=100, eps=1e-9):
        """Non-negative factorisation X ~ U V^T (Frobenius) by Lee-Seung multiplicative updates on the resident row
        block: two library GEMMs per sweep (X V and X^T U; torch.matmul, fp32), the p x k and k x k products summed
        over ranks.  Initialisation as sklearn's `init='random'`: sqrt(mean(X) / k) * |N(0, 1)|, seeded from
        `np.random` (rank 0's gene factors are broadcast).  Initialisation only: not part of the CAVI iteration."""
        dev, k = self._dev, self.k
        slab = max(1, self._X_SLAB_ENTRIES // max(1, self.p))     # uint16 X: GEMMs over bounded float32 slabs
        gen = torch.Generator(device=dev)
        gen.manual_seed(int(np.random.randint(0, 2 ** 31 - 1)))
        tot = sum(X.sum(dtype=torch.float64) for _, X in self._x_slabs(slab))
        tot = self._shard.allreduce_sum(torch.as_tensor(tot, dtype=torch.float64, device=dev).reshape(1))[0]
        scale = float(torch.sqrt(tot / (float(self.n_total) * self.p * k)).item()) or 1.0
        U = scale * torch.randn((self.n, k), device=dev, generator=gen).abs_()
        V = scale * torch.randn((self.p, k), device=dev, generator=gen).abs_()
        self._shard.broadcast(V)
        for _ in range(iters):
            VtV = V.T @ V
            XtU = None
            for r, X in self._x_slabs(slab):
                Ur = U[r:r + X.shape[0]]
                Ur *= (X @ V) / (Ur @ VtV + eps)
                XtU = X.T @ Ur if XtU is None else XtU + X.T @ Ur
            XtU = self._shard.allreduce_sum(V.new_zeros(V.shape) if XtU is None else XtU)
            UtU = self._shard.allreduce_sum(U.T @ U)
            V *= XtU / (V @ UtU + eps)
        return U, V

    def initialize_parameters(self):
        """base.py:43-52."""
        self.initialize_variational_parameters()
        self.update_expectations()
        self.update_prior_hyper_parameters()

    def _set_factor(self, dst, values):
        K = self.k
        if isinstance(values, torch.Tensor):
            v = values.to(device=self._dev, dtype=torch.float64)
        else:
            v = torch.as_tensor(np.asarray(values, dtype=np.float64), device=self._dev)
        dst.zero_()
        dst[:, :K] = torch.clamp(torch.nan_to_num(v), min=1e-15).to(torch.float32)   # zigap.py:63,73

    def _draw_factor_inits(self):
        """zigap.py:58-75 / gap.py:49-65: a1, b1 from the NMF factors or Gamma(1) draws; a2 = b2 = 1.

        RNG stream: the reference's constructor ALWAYS runs sklearn's NMF (base.py:37-40), whose default initialisation
        draws from the global `np.random` state, before it reaches these Gamma(1) draws; with `use_factors=False` this
        class skips the factorisation (it is discarded by the reference in that case), so after `np.random.seed(s)` the
        draws below are NOT the reference's.  Parity runs therefore copy the state vector out of a constructed reference
        model (`state=`, SURVEY.md section 8c) instead of re-deriving it from a seed."""
        if self.use_factors:
            a1, b1 = self._nmf_U, self._nmf_V
        else:
            a1 = np.random.gamma(1., size=(self.n, self.k))
            b1 = np.random.gamma(1., size=(self.m, self.k))
        self._set_factor(self._a1, a1)
        self._set_factor(self._b1, b1)
        self._set_factor(self._a2, np.ones((self.n, self.k)))
        self._set_factor(self._b2, np.ones((self.m, self.k)))
        # the gene side is replicated: every rank must start from the same draws (rank 0's), whatever the
        # state of the per-process numpy generators
        self._shard.broadcast(self._b1)
        self._shard.broadcast(self._b2)
        self._shard.broadcast(self._hyper)

    # ------------------------------------------------------------------------------------------------
    def update_expectations(self):
        """zigap.py:160-165: U_hat, V_hat, log-expectations from (a1, a2, b1, b2), on the device."""
        self._call('ori_count_stats') if not self._started else self._red64.zero_()
        self._call('ori_init_expectations', self._gen)
        self._shard.allreduce_sum(self._red64)
        self._D_cache = None

    def step(self):
        """One CAVI iteration (base.py:54-56)."""
        if self._graphs is not None and self._timers is None and not self._dirty:
            return self._step_graph()
        self.update_variational_parameters()   # E-step
        self.update_prior_hyper_parameters()   # M-step

    def _step_graph(self):
        """step() as the replay of a CUDA graph.  Two graphs are captured lazily, one per parity of the row-factor
        generation (the kernels receive the ping-pong index as an argument); the iteration count lives on the device
        (ORI_F_DEVICE_ITER).  The first step of each parity runs eagerly once (lazy one-time initialisation inside the
        library must not happen under capture)."""
        self._check_trace_room()
        key = self._gen
        g = self._graphs.get(key)
        if g is None:
            self._graphs[key] = 'warm'                    # this parity has now run eagerly once
            self.update_variational_parameters()
            self.update_prior_hyper_parameters()
            return
        if g == 'warm':
            self._scal[_lib.ORI_SC_ITER] = float(self._iter)      # the device-side count the captured kernels read
            torch.cuda.synchronize()
            before = int(self._lib.ori_kernel_launches())
            g = torch.cuda.CUDAGraph()
            gen0, it0 = self._gen, self._iter
            with torch.cuda.graph(g):
                self.update_variational_parameters()
                self.update_prior_hyper_parameters()
            self._gen, self._iter = gen0, it0             # capture executed nothing: undo the host-side bookkeeping
            self._graphs[key] = g
            self._graph_kernels = int(self._lib.ori_kernel_launches()) - before
        g.replay()
        self.graph_replays += 1
        self._pending_mstep = False
        self._gen ^= 1
        self._iter += 1
        self._pi_stale = self._dropout
        self._D_cache = None

    @property
    def graph_kernel_launches(self):
        """Kernels of this library launched through graph replays so far (ori_kernel_launches() counts launch calls,
        i.e. a captured step only once)."""
        return self.graph_replays * self._graph_kernels

    def update_variational_parameters(self):
        """E-step (zigap.py:97-141 / gap.py:82-115)."""
        self._check_trace_room()
        if self._dirty:
            self._refresh()
        if self._timers is None:
            self._call('ori_cavi_step_local', self._gen)
        else:   # same launches, with CUDA events around the two kernels that stream X
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            self._call('ori_zero_accumulators', 1)
            ev[0].record(); self._call('ori_pass_rows', self._gen); ev[1].record()
            self._call('ori_row_update', self._gen, 1)
            ev[2].record(); self._call('ori_pass_genes', self._gen); ev[3].record()
            self._timers.append(ev)
        if self._shard.enabled:
            self._shard.allreduce_sum(self._red32)
            self._shard.allreduce_sum(self._red64)
        self._call('ori_gene_update', 1)
        self._pending_mstep = True

    def update_prior_hyper_parameters(self):
        """M-step (zigap.py:143-158 / gap.py:117-129).  At construction: on the initial expectations."""
        if not self._started:
            mode = _lib.ORI_M_INIT_KEEP if getattr(self, '_keep_hyper', False) else _lib.ORI_M_INIT
            self._call('ori_mstep', mode)
            self._started = True
            self._pi_stale = False
            return
        if not getattr(self, '_pending_mstep', False):
            raise RuntimeError('update_prior_hyper_parameters() follows update_variational_parameters()')
        self._call('ori_mstep', _lib.ORI_M_STEP)
        self._pending_mstep = False
        self._gen ^= 1
        self._iter += 1
        self._pi_stale = self._dropout
        self._D_cache = None

    def _check_trace_room(self):
        """The ELBO trace is a fixed device buffer: a model that records it refuses to run past its capacity (build it
        with a larger `trace_cap`); models without the ELBO terms (elbo=False, SparseZIGaP) have no iteration limit,
        like the reference."""
        if (self._flags & _lib.ORI_F_ELBO) and self._iter + 1 >= self._trace_cap:
            raise RuntimeError('elbo trace capacity %d exhausted; build the model with a larger trace_cap'
                               % self._trace_cap)

    def _refresh(self):
        """Parameters were edited through `model.a1[:] = ...`: re-derive expectations and ELBO terms."""
        self._red64.zero_()
        self._call('ori_init_expectations', self._gen)
        self._shard.allreduce_sum(self._red64)
        self._call('ori_mstep', _lib.ORI_M_REFRESH)
        self._dirty = False
        self._D_cache = None
        self._ll_cache = None

    def _finalize(self):
        """Flush the one-pass lag: pi(t) and ELBO(t) of the current state (one extra sweep of X)."""
        if self._dirty:
            self._refresh()
        if self._dropout and self._pi_stale:
            self._pi_gen = self._pi.clone()
        self._call('ori_finalize_local', self._gen)
        self._shard.allreduce_sum(self._red64)
        self._call('ori_mstep', _lib.ORI_M_FINALIZE)
        self._pi_stale = False

    def enable_kernel_timing(self, on=True):
        """Record CUDA events around the row pass and the gene pass of every following step."""
        self._timers = [] if on else None

    def kernel_times_ms(self):
        """Mean device time of (row pass, gene pass) over the steps timed so far (synchronises)."""
        torch.cuda.synchronize()
        if not self._timers:
            return None
        rows = [e[0].elapsed_time(e[1]) for e in self._timers]
        genes = [e[2].elapsed_time(e[3]) for e in self._timers]
        return dict(pass_rows=sum(rows) / len(rows), pass_genes=sum(genes) / len(genes), steps=len(rows))

    # ------------------------------------------------------------------------------------------------
    def elbo(self):
        """Evidence lower bound of the current state (float64 accumulation on the device)."""
        self._finalize()
        return float(self._scal[_lib.ORI_SC_ELBO_LAST].item())

    @property
    def elbo_trace(self):
        """ELBO after construction and after each completed step: array of length iterations + 1."""
        self._finalize()
        return self._trace[:self._iter + 1].cpu().numpy()

    @property
    def iterations(self):
        return self._iter

    @property
    def U_hat(self):
        return self._Uhat[self._gen][:, :self.k].to(torch.float64).cpu().numpy()

    @property
    def V_hat(self):
        return self._Vhat[:, :self.k].to(torch.float64).cpu().numpy()

    def _meanlog(self, h1, h2):
        """E[log .] = psi(a) - log(b) as float32 (gamma.py:48-61).  The kernels keep exp(E[log .]) only; the
        log-expectation itself is re-derived on request (it can be below the float32 exp underflow)."""
        a = h1[:, :self.k].contiguous(); b = h2[:, :self.k].contiguous()
        out = torch.empty_like(a)
        _lib.check(self._lib.ori_gamma_expect_f32(a.data_ptr(), b.data_ptr(), None, out.data_ptr(), None,
                                                  a.numel(), _lib.stream_ptr()))
        return out.cpu().numpy()

    @property
    def log_U_hat(self):
        if self._dirty:
            self._refresh()
        return self._meanlog(self._a1, self._a2)

    @property
    def log_V_hat(self):
        if self._dirty:
            self._refresh()
        return self._meanlog(self._b1, self._b2)

    def device_state(self):
        """Zero-copy views of the device-resident state (torch CUDA tensors).  `eU` / `eV` are exp(E[log .]) rescaled per
        cell / gene by 2^58 / max_k exp(E[log .]) (csrc/special.cuh): only their ratios within a row are meaningful."""
        K = self.k
        out = dict(X=self._X, a1=self._a1[:, :K], a2=self._a2[:, :K], b1=self._b1[:, :K], b2=self._b2[:, :K],
                   U_hat=self._Uhat[self._gen][:, :K], V_hat=self._Vhat[:, :K],
                   eU=self._eU[self._gen][:, :K], eV=self._eV[:, :K],
                   alpha1=self._hyper[0], alpha2=self._hyper[1], beta1=self._hyper[2], beta2=self._hyper[3])
        if self._dropout:
            out.update(lp=self._lp, pi_d=self._pi)
        return out

    def factors(self):
        """base.py:97-98."""
        return self.U_hat, self.V_hat

    def state_dict(self):
        """The state vector of SURVEY.md section 8c as host float64 arrays (checkpoint / parity hand-off)."""
        s = {k: getattr(self, k).asarray() for k in ('a1', 'a2', 'b1', 'b2', 'alpha1', 'alpha2', 'beta1', 'beta2')}
        s['iterations'] = self._iter
        return s

    def load_state(self, state):
        """Seed the model from a state vector copied out of a reference model (or `state_dict()`)."""
        K = self.k
        for name, dst in (('a1', self._a1), ('a2', self._a2), ('b1', self._b1), ('b2', self._b2)):
            v = np.asarray(state[name], dtype=np.float64)
            if v.shape != (dst.shape[0], K):
                raise ValueError('%s has shape %s, expected %s' % (name, v.shape, (dst.shape[0], K)))
            dst.zero_()
            dst[:, :K] = torch.as_tensor(v, device=self._dev).to(torch.float32)
        for i, name in enumerate(('alpha1', 'alpha2', 'beta1', 'beta2')):
            self._hyper[i] = torch.as_tensor(np.asarray(state[name], dtype=np.float64), device=self._dev)
        self._keep_hyper = self._keep_hyper_arg
        self._ll_cache = None
        self._started = False
        self._gen = 0
        self._iter = 0
        self.update_expectations()
        self.update_prior_hyper_parameters()
        self._after_load_state(state)
        # the device-side iteration count (ORI_F_DEVICE_ITER: index of the next ELBO trace entry under graph replay) and
        # the trace follow the host-side count of the loaded state
        self._scal[_lib.ORI_SC_ITER] = float(self._iter)
        self._trace.zero_()
        if self._graphs is not None:
            self._graphs.clear()

    def _after_load_state(self, state):
        pass

    # -- reference metrics that are out of the hot path (base.py:58-95) -------------------------------
    def frobenius_norm(self):
        """base.py:84-87, evaluated in row slabs on the device (no n x p float64 temporary)."""
        tot = torch.zeros((), dtype=torch.float64, device=self._dev)
        U = self._Uhat[self._gen][:, :self.k]; V = self._Vhat[:, :self.k]
        step = max(1, self._X_SLAB_ENTRIES // max(1, self.p))
        for r0, X in self._x_slabs(step):
            for r in range(r0, r0 + X.shape[0], step):
                d = (U[r:r + step] @ V.T) - X[r - r0:r - r0 + step]
                tot += (d.double() ** 2).sum()
        tot = self._shard.allreduce_sum(tot.reshape(1))[0]
        return float(torch.sqrt(tot).item())

    def loglikelihood(self):
        """base.py:89-95: log p(U) + log p(V) + log p(X | U V^T) at the current expectations, summed by the graph nodes
        themselves (the reference's own per-node formulas).  Like the reference this materialises U V^T as an n x p
        float64 array (here on the device, released before returning), so it is for small problems; and like the
        reference it only exists where the X node is probabilistic (GaP): ZIGaP's X is a `Multiply` node, which has no
        `loglikelihood` (AttributeError in the reference too).  The node formulas are the reference's, quirks included:
        Gamma terms summed over every (factor column, parameter column) pair, Poisson terms without log x! and
        truncated to integers when the count matrix came in an integer dtype (tests/golden/loglik.npz)."""
        x_ll = self.X.loglikelihood                                   # AttributeError for deterministic X, before any work
        self.U.buffer = self._Uhat[self._gen][:, :self.k].double()
        self.V.buffer = self._Vhat[:, :self.k].double()
        self.UV.forward()
        try:
            if self._flags & _lib.ORI_F_X_U16:
                # the Poisson terms of uint16 counts, slab by slab from a float32 widening (the node's own formula)
                uv, xl = self.UV.tensor, 0.
                for r, X in self._x_slabs(max(1, self._X_SLAB_ENTRIES // max(1, self.p))):
                    xl += float(torch.nan_to_num(self.X._logp(X, uv[r:r + X.shape[0]])).sum().item())
            else:
                xl = x_ll()
            local = torch.tensor([self.U.loglikelihood() + xl], dtype=torch.float64, device=self._dev)
        finally:
            self.UV._t = None
        return float(self._shard.allreduce_sum(local)[0].item()) + self.V.loglikelihood()

    # ------------------------------------------------------------------------------------------------
    @abstractmethod
    def build_u_node(self):
        pass

    @abstractmethod
    def build_v_node(self):
        pass

    @abstractmethod
    def build_x_node(self, cmatrix, UV):
        pass

    @abstractmethod
    def define_variational_distribution(self):
        pass

    @abstractmethod
    def initialize_variational_parameters(self):
        pass
