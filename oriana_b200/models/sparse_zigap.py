"""SparseZIGaP -- PCMF with the spike-and-slab sparsity layer on V (oriana/models/sparse_zigap.py:15-204), the model
the reference's drivers run (main.py:29, experiments/clustering.py:19).

V_jk = S_jk * V'_jk,  S_jk ~ Bernoulli(pi_s_j),  V'_jk ~ Gamma(beta1_k, beta2_k); everything else as ZIGaP.
One CAVI iteration is the ZIGaP iteration with three changes (sparse_zigap.py:118-196):
  * the multinomial step runs on exp(E[log V']) masked by S_tilde = (p_s > tau) and returns a third gene-side sum
    (:100-116);
  * the gene side updates V' AND S (:144-163) and the M-step also refreshes pi_s (:196);
  * the dropout posterior multiplies the NEW U_hat with the effective V_hat = S_hat * V'_hat of the iteration's START
    (:140, :166) -- so the kernels that rebuild D_hat on the fly keep one older generation of it (`Vh_old`).
K <= 64 (tensor kernels: K <= 32); no ELBO (the reference's convergence trace for this model is the deviance, `reconstruction_deviance()` /
`explained_deviance()`, base.py:58-82, evaluated on the device).

Kernel family.  The S update is a sigmoid of the difference of two large gene-side sums (:157-160), so p_s amplifies
ABSOLUTE errors of those sums exponentially: parity with the reference needs fp32-grade sums.  Problems large enough to
fill the machine (>= 2^21 entries) therefore run the tcgen05 kernels in their fp32-grade mode (`precise=True`, the
default here: R, D_hat and the factor operands of the gene- and row-side sums split hi/lo, csrc/kernels_tc.cu PRECISE)
-- the same two passes with the masked operands plus a second, dropout-free gene sweep for the third sum; smaller ones
run the CUDA-core kernels (csrc/kernels_simt.cu, fp32 FMA).  Both are checked against the reference's recorded
trajectories at the same tolerances (tests/test_sparse_gpu.py).  `precise=False` opts into the TF32-operand kernels
(~1.4x faster, 2^-12 / sqrt(cells) noise on each gene-side sum: not comparable step by step, DESIGN.md 4.4).
"""
import numpy as np
import torch

from .. import _lib
from ..nodes import Bernoulli, Gamma, Multiply
from .base import DeviceView, FactorModel
from .zigap import ZIGaP


class SparseZIGaP(ZIGaP):

    _sparse = True

    def __init__(self, *args, tau=0.5, **kwargs):
        if kwargs.get('compat_quirk'):
            raise ValueError('compat_quirk is a ZIGaP switch (zigap.py:94); sparse_zigap.py:115 has the correct index')
        kwargs['elbo'] = False
        kwargs.setdefault('precise', True)                        # fp32-grade sums (see the module docstring)
        self._col_mean = None
        ZIGaP.__init__(self, *args, tau=tau, **kwargs)

    # -- device state ----------------------------------------------------------------------------------
    def _extra_fields(self, rowf, genef):
        self._ps, self._logV, self._Vh_old = genef(), genef(), genef()
        self._pis = torch.ones((self.p,), dtype=torch.float64, device=self._dev)
        K_ = self.k
        self.p_s = DeviceView(self, lambda: self._ps[:, :K_])
        self.pi_s = DeviceView(self, lambda: self._pis, on_write=False)
        return dict(p_s=self._ps, logV=self._logV, eVd=genef(), eVz=genef(), Vh_old=self._Vh_old, eUl=[rowf(), rowf()],
                    pi_s=self._pis, tau=float(self.tau))

    # -- model graph (sparse_zigap.py:21-40) -------------------------------------------------------------
    def build_v_node(self):
        np.random.rand(self.m)                                                                  # :27 (RNG order)
        self.S = Bernoulli(self.pi_s, self.dims('m,k ~ d,s'), name='S')
        self._hyper[2] = torch.as_tensor(np.random.gamma(2., size=self.k), device=self._dev)    # :29
        self._hyper[3] = 1.
        self.Vprime = Gamma(self.beta1, self.beta2, self.dims('m,k ~ s,d'), name='Vprime')
        return Multiply(self.S, self.Vprime)

    def define_variational_distribution(self):
        self.S_q = Bernoulli(self.p_s, self.dims('m,k ~ d,d'))                                  # :56-57
        self.p_d = DeviceView(self, self._materialize_D, on_write=False)
        self.D_q = Bernoulli(self.p_d, self.dims('n,p ~ d,d'))
        np.random.gamma(2., size=(self.n, self.k))                                              # :64 (RNG order)
        self.U_q = Gamma(self.a1, self.a2, self.dims('n,k ~ d,d'))
        np.random.gamma(2., size=(self.m, self.k))                                              # :69
        self.Vprime_q = Gamma(self.b1, self.b2, self.dims('m,k ~ d,d'))

    def initialize_variational_parameters(self):
        ZIGaP.initialize_variational_parameters(self)
        self._ps.zero_()
        self._ps[:, :self.k] = 1.                                                               # :95
        self._pis.fill_(1.)          # the constructor's M-step: row means of p_s (base.py:52 -> :196)

    # -- expectations ------------------------------------------------------------------------------------
    @property
    def S_hat(self):
        if self._dirty:
            self._refresh()
        return self._ps[:, :self.k].to(torch.float64).cpu().numpy()

    @property
    def Vprime_hat(self):
        if self._dirty:
            self._refresh()
        return (self._b1[:, :self.k].double() / self._b2[:, :self.k].double()).cpu().numpy()

    @property
    def log_Vprime_hat(self):
        return self.log_V_hat

    def device_state(self):
        out = ZIGaP.device_state(self)
        K = self.k
        out.update(p_s=self._ps[:, :K], pi_s=self._pis, log_Vprime_hat=self._logV[:, :K], V_eff_prev=self._Vh_old[:, :K])
        return out

    # -- state hand-off ----------------------------------------------------------------------------------
    def state_dict(self):
        s = ZIGaP.state_dict(self)
        s['p_s'] = self.p_s.asarray()        # float32 precision: the kernels keep S_hat = float32(p_s)
        s['pi_s'] = self._pis.cpu().numpy()
        s['V_eff_prev'] = self._Vh_old[:, :self.k].to(torch.float64).cpu().numpy()
        return s

    def load_state(self, state):
        K = self.k
        ps = np.asarray(state['p_s'], dtype=np.float64)
        if ps.shape != (self.p, K):
            raise ValueError('p_s has shape %s, expected %s' % (ps.shape, (self.p, K)))
        self._ps.zero_()
        self._ps[:, :K] = torch.as_tensor(ps, device=self._dev).to(torch.float32)
        self._pis.copy_(torch.as_tensor(np.asarray(state['pi_s'], dtype=np.float64), device=self._dev))
        FactorModel.load_state(self, state)

    def _after_load_state(self, state):
        ZIGaP._after_load_state(self, state)
        if state.get('pi_prev') is not None:
            if state.get('V_eff_prev') is None:
                raise ValueError('a mid-run SparseZIGaP snapshot must carry "V_eff_prev" (sparse_zigap.py:140, :166)')
            self._Vh_old.zero_()
            self._Vh_old[:, :self.k] = torch.as_tensor(np.asarray(state['V_eff_prev']), device=self._dev).to(torch.float32)

    # -- the reference's convergence metrics (base.py:58-82, sparse_zigap.py:44-51) ------------------------
    def _loglikelihood_sums(self, want_f64=True):
        """(int64-truncated, float64) sums of the zero-inflated Poisson log-likelihood at the three rates:
        masked U_hat V_hat^T, X itself, column means of X."""
        if self._dirty:
            self._refresh()
        # the reference's drivers print both metrics every iteration (main.py:37-44): one sweep of X serves both calls
        key = (self._iter, self._gen, bool(want_f64))
        cached = getattr(self, '_ll_cache', None)
        if cached is not None and cached[0] == key and self._D_cache_valid_for_ll():
            return cached[1]
        pi = self._current_pi()
        dev = self._dev
        if self._col_mean is None:
            cs = torch.zeros((self.p,), dtype=torch.float64, device=dev)
            _lib.check(self._lib.ori_column_sums_f64(self._X.data_ptr(), self._ldx, self.n, self.p, cs.data_ptr(),
                                                     _lib.stream_ptr()))
            self._shard.allreduce_sum(cs)
            self._col_mean = cs / float(self.n_total)
        out_i = torch.zeros((3,), dtype=torch.int64, device=dev)
        out_f = torch.zeros((3,), dtype=torch.float64, device=dev)
        self._call('ori_deviance_sums', self._gen, pi.data_ptr(), self._col_mean.data_ptr(), out_i.data_ptr(),
                   out_f.data_ptr() if want_f64 else None)
        self._shard.allreduce_sum(out_i)
        self._shard.allreduce_sum(out_f)
        res = (out_i.cpu().numpy(), out_f.cpu().numpy())
        self._ll_cache = (key, res)
        self._ll_epoch = self._state_epoch()
        return res

    def _state_epoch(self):
        # changes whenever the state the metrics are computed from may have changed: steps, reloads, parameter edits
        return (self._iter, self._gen, self._started, id(self._graphs) if self._graphs is not None else 0, self.graph_replays)

    def _D_cache_valid_for_ll(self):
        return getattr(self, '_ll_epoch', None) == self._state_epoch() and not self._dirty

    def reconstruction_deviance(self, int_quirk=True):
        """base.py:58-69.  `int_quirk=True` reproduces the reference's integer log-likelihood buffer
        (sparse_zigap.py:45: every entry truncated toward zero before the sum); False gives the float64 sum."""
        li, lf = self._loglikelihood_sums(want_f64=not int_quirk)
        ll = li.astype(np.float64) if int_quirk else lf
        return float(-2. * (ll[0] - ll[1]))

    def explained_deviance(self, int_quirk=True):
        """base.py:71-82 (with the rate mask of the current state, i.e. right after reconstruction_deviance())."""
        li, lf = self._loglikelihood_sums(want_f64=not int_quirk)
        ll = li.astype(np.float64) if int_quirk else lf
        return float((ll[0] - ll[2]) / (ll[1] - ll[2]))
