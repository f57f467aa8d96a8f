"""ZIGaP -- zero-inflated Gamma-Poisson factor model, i.e. PCMF without the sparsity layer
(oriana/models/zigap.py:15-165).

X_ij = L_ij * D_ij,  L_ij ~ Poisson(sum_k U_ik V_jk),  D_ij ~ Bernoulli(pi_j)   (D = 1: expressed)
U_ik ~ Gamma(alpha1_k, alpha2_k),  V_jk ~ Gamma(beta1_k, beta2_k).

`compat_quirk=True` reproduces zigap.py:94, where the gene-side latent counts are weighted by
D_hat[i, k] (the dropout posterior of gene number k) instead of D_hat[i, j]; the default is the correct
index (as in sparse_zigap.py:115), for which the ELBO is monotone.
"""
import numpy as np
import torch

from ..nodes import Bernoulli, Gamma, Multiply, Poisson
from ..problem import logit_pi
from .base import DeviceView, FactorModel


class ZIGaP(FactorModel):

    _dropout = True

    def __init__(self, *args, tau=0.5, **kwargs):
        self.tau = tau            # unused by the reference's ZIGaP as well (zigap.py:17-18)
        self._pi_gen = None
        FactorModel.__init__(self, *args, **kwargs)

    def build_u_node(self):
        self._hyper[0] = torch.as_tensor(np.random.gamma(2., size=self.k), device=self._dev)   # zigap.py:22
        self._hyper[1] = 1.
        return Gamma(self.alpha1, self.alpha2, self.dims('n,k ~ s,d'), name='U')

    def build_v_node(self):
        self._hyper[2] = torch.as_tensor(np.random.gamma(2., size=self.k), device=self._dev)   # zigap.py:27
        self._hyper[3] = 1.
        return Gamma(self.beta1, self.beta2, self.dims('m,k ~ s,d'), name='V')

    def build_x_node(self, cmatrix, UV):
        # the reference draws pi_d ~ U(0,1) here (zigap.py:32) and replaces it by the column means of
        # (X > 0) before the first step (base.py:52 -> zigap.py:158)
        np.random.rand(self.p)
        self.pi_d = DeviceView(self, self._current_pi, on_write=False)
        self.D = Bernoulli(self.pi_d, self.dims('n,p ~ s,d'), name='D')
        self.L = Poisson(UV, self.dims('n,m ~ d,d'), name='X')
        X = Multiply(self.L, self.D)
        X.buffer = self._X
        return X

    def define_variational_distribution(self):
        self.p_d = DeviceView(self, self._materialize_D, on_write=False)     # zigap.py:42-43
        self.D_q = Bernoulli(self.p_d, self.dims('n,p ~ d,d'))
        np.random.gamma(2., size=(self.n, self.k))                           # zigap.py:46 (RNG order only)
        self.U_q = Gamma(self.a1, self.a2, self.dims('n,k ~ d,d'))
        np.random.gamma(2., size=(self.m, self.k))                           # zigap.py:51
        self.V_q = Gamma(self.b1, self.b2, self.dims('m,k ~ d,d'))

    def initialize_variational_parameters(self):
        self._draw_factor_inits()                                            # zigap.py:55-75
        self._lp.fill_(float('-inf'))                                        # p_d = (X > 0), zigap.py:77
        self._pfloor.zero_()

    # -- dropout posterior -------------------------------------------------------------------------
    def _current_pi(self):
        if self._pi_stale:
            self._finalize()
        return self._pi

    def _materialize_D(self):
        """D_hat = float32(p_d) (zigap.py:131-136), recomputed from (U_hat, V_hat, pi) on request."""
        if self._dirty:
            self._refresh()
        if self._D_cache is None:
            out = torch.empty((self.n, self.p), dtype=torch.float32, device=self._dev)
            self._call('ori_dropout_posterior_f32', self._gen, out.data_ptr(), self.p, 0, self.n)
            self._D_cache = out
        return self._D_cache

    @property
    def D_hat(self):
        return self._materialize_D().cpu().numpy()

    def state_dict(self):
        s = FactorModel.state_dict(self)
        s['pi_d'] = self.pi_d.asarray()
        if self._iter > 0 or self._pi_gen is not None:
            s['pi_prev'] = self._pi_gen.cpu().numpy()
        return s

    def _set_generating_pi(self, pi_prev):
        pi = torch.as_tensor(np.asarray(pi_prev, dtype=np.float64), device=self._dev)
        lp, pfloor = logit_pi(pi)
        self._lp.copy_(lp); self._pfloor.copy_(pfloor)
        self._pi_gen = pi.clone()
        # `_finalize()` snapshots `_pi` as the generating pi before it refreshes it: keep the two in step, so that a
        # state_dict() taken right after a load (no step in between) carries the same pi_prev it was loaded with
        self._pi.copy_(pi)
        self._pi_stale = True
        self._D_cache = None

    def _after_load_state(self, state):
        if state.get('pi_prev') is not None:
            # mid-run snapshot: D_hat = sigmoid(logit(pi_prev) - U_hat V_hat^T) (zigap.py:131-132)
            self._set_generating_pi(state['pi_prev'])
            self._iter = int(state.get('iterations', 0))
        elif 'p_d' in state:
            pd = np.asarray(state['p_d'])
            X = self.cmatrix.as_array()
            zero = X == 0
            if pd.shape != X.shape or (pd[zero] != 0).any() or (pd[~zero] < 0.5).any():
                raise ValueError('state["p_d"] is not the indicator (X > 0) of a freshly constructed model; '
                                 'a mid-run snapshot must carry "pi_prev" (SURVEY.md section 8c)')
