"""CPU: how the drivers describe the device state (oriana_b200/problem.py) -- kernel plan, buffer sizes, the
`ori_problem_t` builder, logit(pi_prev) -- and the escape list the two compact count formats share."""
import ctypes

import numpy as np
import pytest
import torch

from oriana_b200 import _lib
from oriana_b200.problem import build_problem, gene_buffers, kernel_plan, logit_pi, row_pitch

E = 1 << 21                               # matrix entries from which the tensor path is the default
PREC, SIMT = _lib.ORI_F_PRECISE, _lib.ORI_F_NO_TENSOR

# (k, entries, options) -> (tensor, KP, flags), or ValueError
PLANS = [
    (5, E - 1, {}, (False, 8, 0)),
    (5, E, {}, (True, 32, 0)),
    (32, E - 1, {}, (False, 32, 0)),
    (32, E, {}, (True, 32, 0)),
    (33, E, {}, (True, 64, 0)),
    (40, E - 1, {}, (False, 64, 0)),
    (40, E, {}, (True, 64, 0)),
    (64, E, {}, (True, 64, 0)),
    (65, E, {}, ValueError),
    (65, E - 1, {}, ValueError),
    # precise: the split-operand tensor kernels for k <= 32, the CUDA-core kernels above
    (5, E - 1, dict(precise=True), (False, 8, 0)),
    (5, E, dict(precise=True), (True, 32, PREC)),
    (32, E, dict(precise=True), (True, 32, PREC)),
    (33, E, dict(precise=True), (False, 64, 0)),
    (40, E, dict(precise=True), (False, 64, 0)),
    (40, E, dict(precise=True, tensor=True), (False, 64, 0)),
    # force_simt
    (5, E, dict(force_simt=True), (False, 8, SIMT)),
    (40, E, dict(force_simt=True), (False, 64, SIMT)),
    (5, E, dict(force_simt=True, precise=True), (False, 8, SIMT)),
    (5, E, dict(force_simt=True, tensor=True), ValueError),
    # an explicit choice of kernel family
    (5, E - 1, dict(tensor=True), (True, 32, 0)),
    (64, 1, dict(tensor=True), (True, 64, 0)),
    (65, E, dict(tensor=True), ValueError),
    (5, E, dict(tensor=False), (False, 8, 0)),
    # SparseZIGaP (precise by default): tensor plans for k <= 32 only
    (5, E - 1, dict(sparse=True, precise=True), (False, 8, 0)),
    (5, E, dict(sparse=True, precise=True), (True, 32, PREC)),
    (32, E, dict(sparse=True, precise=True), (True, 32, PREC)),
    (33, E, dict(sparse=True, precise=True), (False, 64, 0)),
    (40, E, dict(sparse=True), (False, 64, 0)),
    (40, E, dict(sparse=True, force_simt=True), (False, 64, SIMT)),
    (40, E, dict(sparse=True, tensor=True), ValueError),
    (64, E, dict(sparse=True), (False, 64, 0)),
    (65, E - 1, dict(sparse=True), ValueError),
    (65, E, dict(sparse=True, tensor=False), ValueError),
    # the host-streamed step: slab x p entries, precise as asked, never force_simt
    (40, 32768 * 20000, dict(precise=True), (False, 64, 0)),
    (40, 32768 * 20000, {}, (True, 64, 0)),
    (20, 32768 * 20000, dict(precise=True), (True, 32, PREC)),
]


@pytest.mark.parametrize('k, entries, opts, want', PLANS)
def test_kernel_plan(k, entries, opts, want):
    if want is ValueError:
        with pytest.raises(ValueError):
            kernel_plan(k, entries, **opts)
    else:
        assert kernel_plan(k, entries, **opts) == want


def test_row_pitch_and_gene_buffer_sizes():
    assert [row_pitch(p) for p in (1, 4, 5, 977, 20000)] == [4, 4, 8, 980, 20000]
    p, K, KP = 10, 3, 8
    for dropout, sparse in ((True, False), (False, True)):
        g = gene_buffers(p, K, KP, 'cpu', dropout=dropout, sparse=sparse, trace_cap=7)
        for name in ('b1', 'b2', 'V_hat', 'eV'):
            assert g[name].shape == (p, KP) and g[name].dtype == torch.float32
        assert g['red32'].shape == (3 if sparse else 2, p, KP)
        assert g['red64'].shape == (p + 2 * KP + _lib.R64_NSLOTS,) and g['red64'].dtype == torch.float64
        assert g['gsum'].shape == (2 * KP + 8,) and g['scal'].shape == (_lib.SCAL_SLOTS,)
        assert g['hyper'].shape == (4, K) and bool((g['hyper'] == 1).all()) and g['elbo_trace'].shape == (7,)
        if dropout:
            assert g['lp'].shape == g['pfloor'].shape == g['pi_d'].shape == (p,) and bool(torch.isinf(g['lp']).all())
        else:
            assert g['lp'] is None and g['pfloor'] is None and g['pi_d'] is None


def test_build_problem_fills_every_field():
    fields = dict(_lib.OriProblem._fields_)
    pointers = [f for f, ty in fields.items() if ty is ctypes.c_void_p]
    pairs = [f for f, ty in fields.items() if ty is ctypes.c_void_p * 2]
    assert {'X', 'b1', 'red64', 'tc_ws', 'det_ws', 'p_s', 'thrV'} <= set(pointers) and set(pairs) == {'U_hat', 'eU', 'eUl'}
    arrays = {f: torch.zeros((i + 1,)) for i, f in enumerate(pointers)}
    arrays.update({f: [torch.zeros((2,)), torch.zeros((3,))] for f in pairs})
    scalars = dict(n_rows=7, n_total=9, ldx=12, p=10, K=3, KP=8, flags=5, trace_cap=4, tau=0.5)
    P = build_problem(**scalars, **arrays)
    for f in pointers:
        assert getattr(P, f) == arrays[f].data_ptr(), f
    for f in pairs:
        assert [getattr(P, f)[g] for g in (0, 1)] == [t.data_ptr() for t in arrays[f]], f
    assert P.tc_ws_floats == arrays['tc_ws'].numel() and P.det_ws_doubles == arrays['det_ws'].numel()
    for f, v in scalars.items():
        assert getattr(P, f) == v, f
    assert P.iter == 0

    P = build_problem(**{f: None for f in pointers}, **{f: (None, None) for f in pairs})
    assert all(getattr(P, f) is None for f in pointers)
    assert all(getattr(P, f)[g] is None for f in pairs for g in (0, 1))
    assert P.tc_ws_floats == 0 and P.det_ws_doubles == 0
    for bad in ('Xq', 'tc_ws_floats', 'U0'):
        with pytest.raises(TypeError):
            build_problem(**{bad: torch.zeros(1)})


def test_logit_pi():
    pi = torch.tensor([0., 1e-20, 0.3, 1. - 1e-17, 1.], dtype=torch.float64)
    lp, pfloor = logit_pi(pi)
    assert lp.dtype == pfloor.dtype == torch.float32
    want = np.array([-np.inf, np.log(1e-15 / (1. - 1e-15)), np.log(0.3 / 0.7), np.inf, np.inf], dtype=np.float32)
    assert np.array_equal(lp.numpy(), want)
    assert np.array_equal(pfloor.numpy(), np.array([1e-10, 0., 0., 0., 0.], dtype=np.float32))


def test_both_compact_formats_share_the_escape_list():
    from oriana_b200.host_step import CompactCounts, SparseCounts
    X = torch.zeros((6, 40))
    X[1, 3], X[1, 39], X[4, 0], X[5, 7], X[2, 2] = 255., 70000., 300., 254., 9.
    for cls in (CompactCounts, SparseCounts):
        c = cls.from_tensor(X, chunk_rows=4, pin=False)
        assert c.row.tolist() == [1, 1, 4] and c.col.tolist() == [3, 39, 0] and c.val.tolist() == [255., 70000., 300.]
        assert [c.escapes(r0, r1) for r0, r1 in ((0, 1), (0, 2), (2, 5), (5, 6))] == [(0, 0), (0, 2), (2, 3), (3, 3)]
        assert torch.equal(c.dense(), X)
