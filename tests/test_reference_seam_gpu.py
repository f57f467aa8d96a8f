"""GPU: the operator seam exercised inside the reference's CAVI step.

`ZIGaP.compute_Z_q_expectations` / `GaP.compute_Z_q_expectations` (zigap.py:79-95, gap.py:67-80) are replaced by the
ctypes stubs of INTEGRATION.md section 1, i.e. by `ori_*_compute_Z_q_expectations_host` of liboriana_b200.so, called
with host numpy arrays the way the reference calls its numba kernel.  The rest of the step is the oracle's restatement
of the reference's `update_variational_parameters` (zigap.py:97-141, oracle/cavi_numpy.py, pinned against the
reference by tests/test_oracle.py), so the O(n p K) loop runs on the B200 and everything else on the host.  It is
stepped against the unmodified reference stepped on its own numba kernel from the same state (tests/golden/seam_*.npz,
oracle/make_golden.py: the counts and the initial state are regenerated from their seeds and checked by digest).

Tolerance: the reference accumulates the latent-count sums sequentially in float32; the device sums them in tiles.
Over 5 steps the parameters agree to 2e-4 relative (floor 1e-6 max), D_hat to 2e-5 absolute on the CUDA-core kernels
(small problems); a slab of >= 2^21 entries runs the tcgen05 kernels with TF32 operands: 2e-3 / 2e-4 after 2 steps.
"""
import ctypes

import numpy as np
import pytest

from conftest import load_golden, relerr

pytestmark = pytest.mark.gpu


def _stubs(lib):
    fp = ctypes.c_void_p

    keep = []

    def ptr(a, out=False):
        if a.dtype != np.float32 or a.ndim != 2:                   # the numba signature f4[:, :] raises TypeError too
            raise TypeError('2-D float32 array expected (zigap.py:79)')
        if not a.flags.c_contiguous:
            # f4[:, :] accepts any layout, and the reference does pass one: X[:] comes out of a DataFrame column-major
            # (cmatrix.py:31-37) and .astype keeps that order (zigap.py:112).  The C ABI takes row-major arrays.
            assert not out, 'outputs are np.empty arrays (zigap.py:102-104): always C-contiguous'
            a = np.ascontiguousarray(a)
            keep.append(a)
        return fp(a.ctypes.data)

    def check(rc):
        if rc:
            buf = ctypes.create_string_buffer(512)
            lib.ori_last_error(buf, 512)
            raise RuntimeError(buf.value.decode())

    calls = {'zigap': 0, 'gap': 0}

    def zigap_z(DZ_hat_i, DZ_hat_j, DZ_exp_logsum_hat, log_U_hat, log_V_hat, D_hat, X):   # zigap.py:80
        n, p = X.shape
        K = log_U_hat.shape[1]
        calls['zigap'] += 1
        check(lib.ori_zigap_compute_Z_q_expectations_host(
            ptr(DZ_hat_i, True), ptr(DZ_hat_j, True), ptr(DZ_exp_logsum_hat, True), ptr(log_U_hat), ptr(log_V_hat),
            ptr(D_hat), ptr(X), n, p, K, 1))            # 1 = keep the D_hat[i, k] indexing of zigap.py:94
        keep.clear()

    def gap_z(Z_hat_i, Z_hat_j, log_U_hat, log_V_hat, X):                                  # gap.py:68
        n, p = X.shape
        K = log_U_hat.shape[1]
        calls['gap'] += 1
        check(lib.ori_gap_compute_Z_q_expectations_host(ptr(Z_hat_i, True), ptr(Z_hat_j, True), ptr(log_U_hat),
                                                        ptr(log_V_hat), ptr(X), n, p, K))
        keep.clear()
    return zigap_z, gap_z, calls


@pytest.mark.parametrize('model_name,shape', [('ZIGaP', (300, 220, 5)), ('GaP', (257, 190, 7)),
                                              ('ZIGaP', (2100, 1100, 12))])     # the last: tensor-path sized slab
def test_reference_step_with_the_b200_operator(cuda_lib, monkeypatch, model_name, shape):
    from oracle import cavi_numpy as cn, make_golden as mg
    name = {(300, 220, 5): 'seam_zigap', (257, 190, 7): 'seam_gap', (2100, 1100, 12): 'seam_zigap_tc'}[shape]
    model, K, X, s, steps, st = mg.seam_problem(name)
    assert model == model_name and K == shape[2]
    g = load_golden(name)
    assert mg.seam_digest(s) == str(g['digest']) and steps == int(g['steps'])
    zigap_z, gap_z, calls = _stubs(cuda_lib)

    def device_z(log_U_hat, log_V_hat, X, D_hat=None, quirk=True, dtype=np.float32):
        # the reference's call: outputs allocated by the caller, X[:] as a column-major float32 copy (zigap.py:102-111)
        assert quirk and dtype == np.float32
        n, K = log_U_hat.shape
        p = log_V_hat.shape[0]
        Zi, Zj = np.empty((n, K), np.float32), np.empty((p, K), np.float32)
        X32 = np.asfortranarray(X, dtype=np.float32)
        if D_hat is None:
            gap_z(Zi, Zj, log_U_hat, log_V_hat, X32)
        else:
            zigap_z(Zi, Zj, np.empty((p, K), np.float32), log_U_hat, log_V_hat, D_hat, X32)
        return Zi, Zj

    monkeypatch.setattr(cn, 'z_expectations', device_z)
    for _ in range(steps):
        cn.step(s, quirk=True)
    assert calls['zigap' if model_name == 'ZIGaP' else 'gap'] == steps
    names = ('a1', 'a2', 'b1', 'b2', 'alpha1', 'alpha2', 'beta1', 'beta2') + (('pi_d',) if model_name == 'ZIGaP' else ())
    tensor = X.size >= (1 << 21)         # slabs of this size run the tcgen05 kernels: TF32 operands (measured 3.5e-4)
    for k in names:
        got = s[k][::st[k[0]]] if s[k].ndim == 2 else s[k]
        e = relerr(got, g[k])
        assert e < (2e-3 if tensor else 2e-4), (model_name, k, e)
    if model_name == 'ZIGaP':
        D = s['p_d'].astype(np.float32).ravel()[::st['D']]
        assert np.max(np.abs(D - g['D_hat'])) < (2e-4 if tensor else 2e-5)
