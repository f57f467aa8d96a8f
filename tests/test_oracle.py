"""CPU: the oracle port against the golden trajectories made by the UNMODIFIED reference
(oracle/make_golden.py), i.e. the pin of the oracle (task section 3)."""
import numpy as np
import pytest

from conftest import GOLDEN_CASES, golden_state, load_golden, relerr, relerr_quantile
from oracle import cavi_numpy as cn, zloop

PARAMS = ('a1', 'a2', 'b1', 'b2', 'alpha1', 'alpha2', 'beta1', 'beta2')


@pytest.mark.parametrize('name', GOLDEN_CASES)
def test_z_kernel_matches_reference_numba_kernel(name):
    """zigap.py:79-95 / gap.py:67-80: C triple loop (same order) and the ratio form vs the numba output."""
    g = load_golden(name)
    s = golden_state(g, 0)
    e = cn.expectations(s)
    assert np.array_equal(e['log_U_hat'], g['z_log_U_hat'])      # gamma.py:48-61 is reproduced bit for bit
    assert np.array_equal(e['log_V_hat'], g['z_log_V_hat'])
    X32 = s['X'].astype(np.float32)
    if 'p_d' in s:
        Zi, Zj = zloop.zigap_z(e['log_U_hat'], e['log_V_hat'], e['D_hat'], X32, quirk=True)
    else:
        Zi, Zj = zloop.gap_z(e['log_U_hat'], e['log_V_hat'], X32)
    assert relerr(Zi, g['z_Zi']) < 2e-6 and relerr(Zj, g['z_Zj']) < 2e-6
    Zi, Zj = cn.z_expectations(e['log_U_hat'], e['log_V_hat'], s['X'], e.get('D_hat'), quirk=True)
    assert relerr(Zi, g['z_Zi']) < 2e-5 and relerr(Zj, g['z_Zj']) < 2e-5


@pytest.mark.parametrize('name', GOLDEN_CASES)
def test_trajectory_matches_reference(name):
    """base.py:54-56 stepped from the reference's own post-construction state."""
    g = load_golden(name)
    s = golden_state(g, 0)
    steps = [int(t) for t in g['steps']]
    for t in range(1, max(steps) + 1):
        cn.step(s, quirk=True)
        if t in steps:
            r = golden_state(g, t)
            for k in PARAMS + (('pi_d',) if 'pi_d' in s else ()):
                assert relerr(s[k], r[k]) < 5e-5, (name, t, k)
            if 'p_d' in s:
                assert np.max(np.abs(s['p_d'].astype(np.float32) - r['p_d'])) < 1e-5


def test_elbo_monotone_without_quirk():
    """The ELBO (new; parity unpinned in the reference) must not decrease under the de-quirked CAVI."""
    X = cn.synth_counts(120, 90, 4, seed=5)
    for model in ('zigap', 'gap'):
        s = cn.init_state(X, 4, np.random.default_rng(3), model)
        prev = cn.elbo(s)
        for _ in range(15):
            cn.step(s, quirk=False, dtype=np.float64)
            cur = cn.elbo(s)
            assert cur >= prev - 1e-7 * abs(prev), (model, prev, cur)
            prev = cur


def test_special_functions_against_reference_kats():
    g = load_golden('special')
    assert relerr(cn.digamma(g['x']), g['digamma']) < 1e-14
    assert relerr(cn.inverse_digamma(g['y']), g['inverse_digamma']) < 1e-12
    assert np.allclose(cn.sigmoid(g['z']), g['sigmoid'], rtol=1e-15, atol=0)
    assert np.allclose(cn.logit(g['q']), g['logit'], rtol=1e-15, atol=0)
    # test/test.py:13-32
    x = np.asarray([-2.3, 1.5, 0.45, -0.78, 5.3, -.2, 0.])
    np.testing.assert_almost_equal(cn.logit(cn.sigmoid(x)), x)
    x = np.asarray([0.54, 6.2, 1.2, 0.3, 7.9, 4.5, 2.1])
    np.testing.assert_almost_equal(cn.inverse_digamma(cn.digamma(x)), x)
    np.testing.assert_almost_equal(cn.digamma(cn.inverse_digamma(x)), x)


def test_port_matches_live_reference():
    """The port next to the reference's own run on a problem of its own (ZIGaP 60 x 70, K = 3, recorded by
    oracle/make_golden.py port): 3 steps from the reference's post-construction state."""
    g = load_golden('zigap_port')
    s = golden_state(g, 0)
    assert np.array_equal(s['X'], cn.synth_counts(60, 70, 3, seed=11))
    for _ in range(3):
        cn.step(s, quirk=True)
    r = golden_state(g, 3)
    for k in PARAMS + ('pi_d',):
        assert relerr(s[k], r[k]) < 2e-5, k


@pytest.mark.parametrize('name', ['zigap_nmf', 'gap_nmf'])
def test_nmf_initialised_trajectory_matches_reference(name):
    """The reference's default construction path (`use_factors=True`, base.py:38-40): NMF factors with tiny and exactly
    zero entries put E[log U], E[log V] at -100 ... -1e15.  The ratio form only survives there because each factor is
    rescaled per row (`cn.centred_exp`); without it a1, b1 overflow in the first step."""
    g = load_golden(name)
    s = golden_state(g, 0)
    assert (s['a1'] <= 1e-15).any() or (s['b1'] <= 1e-15).any()          # exact zeros of the NMF factors, clamped
    steps = [int(t) for t in g['steps']]
    for t in range(1, max(steps) + 1):
        cn.step(s, quirk=True)
        if t in steps:
            r = golden_state(g, t)
            for k in PARAMS + (('pi_d',) if 'pi_d' in s else ()):
                assert np.isfinite(s[k]).all(), (t, k)
                q, worst = relerr_quantile(s[k], r[k])
                # 99.8 % of the entries to 2e-4; the rest are fed by denormal-range terms of the reference (conftest.py)
                assert q < 2e-4 and worst < 0.5, (t, k, q, worst)
            if 'p_d' in s:
                assert np.max(np.abs(s['p_d'] - r['p_d'])) < 1e-5, t


def test_centred_ratio_form_against_the_sequential_loop_in_the_underflow_regime():
    """Log-expectations between -95 and +5 with sparse supports (what NMF-seeded factors produce): exp(lU) and exp(lV)
    under- and overflow float32 on their own, exp(lU + lV) mostly does not.  The plain ratio form blew up here; the
    per-row centred form (cn.centred_exp) must agree with the C restatement of the reference's triple loop
    (oracle/zloop.c: exp of the SUM, float32, sequential) wherever the reference's terms are normal float32 numbers."""
    rng = np.random.default_rng(12)
    n, p, K = 90, 120, 6
    lU = rng.uniform(-6., 3., size=(n, K)); lV = rng.uniform(-6., 5., size=(p, K))
    lU[rng.random((n, K)) < 0.35] -= rng.uniform(60., 90.)        # components ~e^-80 below the row's largest
    lV[rng.random((p, K)) < 0.35] -= rng.uniform(60., 90.)
    lU[rng.random((n, K)) < 0.05] = -1e15; lV[rng.random((p, K)) < 0.05] = -1e15      # exact zeros of the NMF factors
    lU = lU.astype(np.float32); lV = lV.astype(np.float32)
    X = rng.poisson(3., size=(n, p)).astype(np.float32)
    with np.errstate(all='ignore'):
        plain = np.exp(lU) @ np.exp(lV).T
    assert (plain == 0).any() or np.isinf(1. / plain[plain > 0]).any()     # the uncentred form is out of range here
    Zi, Zj = cn.z_expectations(lU, lV, X, None)
    rZi, rZj = zloop.gap_z(lU, lV, X)
    assert np.isfinite(Zi).all() and np.isfinite(Zj).all()
    for got, ref in ((Zi, rZi), (Zj, rZj)):
        q, worst = relerr_quantile(got, ref, q=0.99)
        assert q < 1e-4, (q, worst)            # the rest: sums fed by denormal-range or fully underflowed terms of the reference
    # the counts are conserved wherever the reference assigns them at all
    alive = rZi.sum(axis=1) > 0.999 * X.sum(axis=1)
    np.testing.assert_allclose(Zi.sum(axis=1)[alive], X.sum(axis=1)[alive], rtol=1e-4)
