"""GPU: the tcgen05/TMA tensor path (csrc/kernels_tc.cu) of the two X-streaming passes against

  * the golden trajectories recorded from the UNMODIFIED reference (compat_quirk=True, zigap.py:94),
  * the oracle port for the de-quirked update and the ELBO,
  * the CUDA-core path of the same library at sizes where work items, chunks and ring wrap-around all occur.

Stated tolerances of the tensor path.  den = eU.eV^T and U_hat.V_hat^T are split-precision (hi.hi in TF32 plus the two
cross terms in one bf16 chain: relative error about 2^-21, fp32-grade); the two
accumulating contractions R.eV, D.V_hat (and their transposes) take R, D and the factor operand rounded to
TF32 (11-bit significand, round to nearest), so a sum of m terms carries a relative error of about
2^-12 / sqrt(m) * few:
  parameters a1,a2,b1,b2 : 3e-3 relative (floor 1e-6*max) on the 100 x 500 fixtures, 1e-3 at 3000 x 1500 (2e-3 for K > 32)
  alpha, beta, pi        : 5e-4
  D_hat                  : 3e-4 absolute (measured <= 1.3e-4 on the fixtures, 2e-5 on the benchmark slabs)
  ELBO                   : 1e-4 relative (north_star's bound; measured <= 1.6e-5 everywhere, 6e-6 on the benchmark slabs)
Measured values per fixture and step: `scripts/gpu_parity_report.py` (log kept under profiles/).
"""
import numpy as np
import pytest

from conftest import GOLDEN_CASES, golden_state, load_golden, relerr

pytestmark = pytest.mark.gpu
FACTORS = ('a1', 'a2', 'b1', 'b2')
HYPER = ('alpha1', 'alpha2', 'beta1', 'beta2')


def make_model(s, quirk, **kw):
    from oriana.models import GaP, ZIGaP
    from oriana.singlecell import CountMatrix
    cls = ZIGaP if ('p_d' in s or 'pi_d' in s) else GaP
    K = s['a1'].shape[1]
    return cls(CountMatrix(s['X']), k=K, use_factors=False, state=s, compat_quirk=quirk, **kw)


@pytest.mark.parametrize('name', GOLDEN_CASES)
def test_tensor_trajectory_matches_reference(cuda_lib, name):
    """Every recorded step of every fixture (up to 50 steps on the config-1 fixtures), not only the early ones: the
    parameters stay inside the stated TF32 envelope -- measured drift at t = 50 (scripts/gpu_parity_report.py): a1..b2
    3.6e-4 / 4.2e-4, alpha / beta / pi 1.9e-4 / 1.2e-4, D_hat 3.5e-5 (zigap_c1 / gap_c1) -- and the ELBO of the device
    model follows the float64 ELBO of the reference's own recorded states to 1e-4 (measured <= 1.6e-5)."""
    from oracle import cavi_numpy as cn
    g = load_golden(name)
    s = golden_state(g, 0)
    steps = [int(t) for t in g['steps']]
    m = make_model(s, quirk=True, tensor=True, trace_cap=max(steps) + 8)
    assert m.uses_tensor_path
    for t in range(1, max(steps) + 1):
        m.step()
        if t in steps:
            r = golden_state(g, t)
            for k in FACTORS:
                e = relerr(getattr(m, k).asarray(), r[k])
                assert e < 3e-3, (name, t, k, e)
            htol = 5e-4       # measured up to 3.3e-4 (pi_d of zigap_c1 at t = 50; K > 32 at t = 3: 3.0e-4)
            for k in HYPER + (('pi_d',) if 'pi_d' in s else ()):
                e = relerr(getattr(m, k).asarray(), r[k])
                assert e < htol, (name, t, k, e)
            if 'p_d' in s:
                assert np.max(np.abs(m.D_hat - r['p_d'])) < 3e-4, (name, t)
            want = cn.elbo(r)
            got = m.elbo()
            assert abs(got - want) < 1e-4 * abs(want), (name, t, got, want)


@pytest.mark.parametrize('cfg,shape,z', [('c3', (2048, 20000, 20), 0.5), ('c4', (2048, 20000, 32), 0.5),
                                         ('c5', (2048, 30000, 64), 0.12)])
def test_tensor_path_on_the_benchmark_workloads_matches_oracle(cuda_lib, cfg, shape, z):
    """BASELINE.json configs[2], [3] (the bench's own workload: exactly the 2048-row slab `bench.py` feeds the oracle for
    `cpu_baseline`) and [4] (K = 64, ~90 % zeros) at a row slab with the full gene axis and latent dimension: six steps of
    the tensor path against the oracle port -- factors, hyper-parameters, pi, D_hat and the whole ELBO trace.
    Measured (scripts/gpu_parity_report.py): a1..b2 2.2e-3 / 1.8e-3 / 2.7e-3 after six steps, alpha, beta, pi 6e-5,
    D_hat 2e-5, ELBO trace 6e-6; the CUDA-core kernels on the same slabs: 8e-6, 5e-6, 1e-6, 6e-7."""
    from oracle import cavi_numpy as cn
    n, p, K = shape
    X = cn.synth_counts(n, p, K, seed=0, z=z)
    if cfg == 'c5':
        assert 0.85 < float((X == 0).mean()) < 0.95
    s = cn.init_state(X, K, np.random.default_rng(0), 'zigap')
    m = make_model(s, quirk=False, tensor=True)
    assert m.uses_tensor_path and m._KP == (32 if K <= 32 else 64)
    ref = {k: v.copy() for k, v in s.items()}
    want = [cn.elbo(ref, guard32=True)]
    for _ in range(6):
        m.step(); cn.step(ref, quirk=False)
        want.append(cn.elbo(ref))
    for k in FACTORS:
        assert relerr(getattr(m, k).asarray(), ref[k]) < 4e-3, (cfg, k)
    for k in HYPER + ('pi_d',):
        assert relerr(getattr(m, k).asarray(), ref[k]) < 2e-4, (cfg, k)
    assert np.max(np.abs(m.D_hat.astype(np.float64) - ref['p_d'])) < 1e-4, cfg
    got = m.elbo_trace
    assert np.max(np.abs(got - np.asarray(want)) / np.abs(want)) < 2e-5, (got, want)
    assert (np.diff(got) > 0).all()


def test_tensor_path_gene_without_zeros(cuda_lib):
    """A gene every cell expresses has pi = 1 (logit = +inf) after the first step: its entropy terms are exact zeros, not
    0 * inf (the ELBO of the tensor path used to come back NaN from such a column)."""
    from oracle import cavi_numpy as cn
    X = cn.synth_counts(2100, 1100, 6, seed=21)
    X[:, 7] = np.maximum(X[:, 7], 1); X[:, 300] = np.maximum(X[:, 300], 2)
    s = cn.init_state(X, 6, np.random.default_rng(3), 'zigap')
    m = make_model(s, quirk=False, tensor=True)
    assert m.uses_tensor_path
    ref = {k: v.copy() for k, v in s.items()}
    want = [cn.elbo(ref, guard32=True)]
    for _ in range(4):
        m.step(); cn.step(ref, quirk=False)
        want.append(cn.elbo(ref))
    got = m.elbo_trace
    assert np.isfinite(got).all()
    assert np.max(np.abs(got - np.asarray(want)) / np.abs(want)) < 1e-4, (got, want)
    assert m.pi_d.asarray()[7] > 1 - 1e-9


@pytest.mark.parametrize('name', ['zigap_ragged', 'gap_ragged', 'zigap_k10'])
def test_tensor_dequirked_update_and_elbo_match_oracle(cuda_lib, name):
    from oracle import cavi_numpy as cn
    g = load_golden(name)
    s = golden_state(g, 0)
    m = make_model(s, quirk=False, tensor=True)
    ref = {k: v.copy() for k, v in s.items()}
    want = [cn.elbo(ref, guard32=True)]
    for t in range(1, 7):
        m.step()
        cn.step(ref, quirk=False)
        want.append(cn.elbo(ref))
    for k in FACTORS:
        assert relerr(getattr(m, k).asarray(), ref[k]) < 3e-3, k
    for k in HYPER + (('pi_d',) if 'pi_d' in s else ()):
        assert relerr(getattr(m, k).asarray(), ref[k]) < 3e-4, k
    got = m.elbo_trace
    assert np.max(np.abs(got - np.asarray(want)) / np.abs(want)) < 1e-4, (got, want)


@pytest.mark.parametrize('shape', [(3000, 1500, 10), (5000, 2100, 32), (1111, 777, 5), (20000, 4500, 20),
                                   (2500, 1900, 40), (3100, 1301, 64)])      # K > 32: the KP = 64 plan (32-wide sweep tiles)
def test_tensor_path_matches_cuda_core_path(cuda_lib, shape):
    """Many work items per SM, split sweeps, ragged last tiles on both axes, every ring wrapping around."""
    from oriana.models import GaP, ZIGaP
    from oriana.singlecell import synth_counts_device
    n, p, K = shape
    X = synth_counts_device(n, p, K, seed=5)
    for cls in (ZIGaP, GaP):
        np.random.seed(3)
        m0 = cls(X[:, :p], k=K, use_factors=False, tensor=False)
        st = m0.state_dict(); st['X'] = X[:, :p]
        ms = cls(X[:, :p], k=K, use_factors=False, state=st, tensor=False)
        mt = cls(X[:, :p], k=K, use_factors=False, state=st, tensor=True)
        assert mt.uses_tensor_path and not ms.uses_tensor_path
        for t in range(3):
            mt.step(); ms.step()
        ftol = 1e-3 if K <= 32 else 2e-3     # more components: fewer counts per (gene, component) sum, same TF32 noise
        for k in FACTORS:
            assert relerr(getattr(mt, k).asarray(), getattr(ms, k).asarray()) < ftol, (cls.__name__, k)
        for k in HYPER + (('pi_d',) if cls is ZIGaP else ()):
            assert relerr(getattr(mt, k).asarray(), getattr(ms, k).asarray()) < 1e-4, (cls.__name__, k)
        et, es = mt.elbo_trace, ms.elbo_trace
        assert np.max(np.abs(et - es) / np.abs(es)) < 1e-4, (et, es)


def test_tensor_all_zero_gene_and_cell(cuda_lib):
    """Columns with pi = 0 take the 1e-10 override (zigap.py:133) on the tensor path too."""
    from oracle import cavi_numpy as cn
    X = cn.synth_counts(150, 70, 3, seed=2)
    X[:, 5] = 0; X[:, 64] = 0; X[17, :] = 0
    s = cn.init_state(X, 3, np.random.default_rng(0), 'zigap')
    m = make_model(s, quirk=False, tensor=True)
    ref = {k: v.copy() for k, v in s.items()}
    for _ in range(4):
        m.step(); cn.step(ref, quirk=False)
    for k in FACTORS + HYPER + ('pi_d',):
        got = getattr(m, k).asarray()
        assert np.isfinite(got).all()
        assert relerr(got, ref[k]) < 3e-3, k
    assert abs(m.pi_d[5] - ref['pi_d'][5]) < 1e-12 and m.pi_d[5] < 1e-9


def test_tensor_path_config2_matches_oracle(cuda_lib):
    """BASELINE.json configs[1] (10k x 2k, K=10) at full size: two CAVI steps of the tensor path against the
    oracle port on the same counts and initial state."""
    from oracle import cavi_numpy as cn
    X = cn.synth_counts(10_000, 2_000, 10, seed=4)
    s = cn.init_state(X, 10, np.random.default_rng(2), 'zigap')
    m = make_model(s, quirk=False, tensor=True)
    assert m.uses_tensor_path
    ref = {k: v.copy() for k, v in s.items()}
    want = [cn.elbo(ref, guard32=True)]
    for _ in range(2):
        m.step(); cn.step(ref, quirk=False)
        want.append(cn.elbo(ref))
    for k in FACTORS:
        assert relerr(getattr(m, k).asarray(), ref[k]) < 1e-3, k
    for k in HYPER + ('pi_d',):
        assert relerr(getattr(m, k).asarray(), ref[k]) < 1e-4, k
    got = m.elbo_trace
    assert np.max(np.abs(got - np.asarray(want)) / np.abs(want)) < 1e-4, (got, want)


def test_host_streamed_step_on_the_tensor_path(cuda_lib):
    """`HostStreamedCAVI` (what bench.py reports as e2e) with slabs large enough for the tcgen05 kernels, host counts
    kept as uint16: same results as the device-resident model, slab by slab (3 ragged slabs)."""
    import torch
    from oriana.models import ZIGaP
    from oriana.singlecell import synth_counts_device
    from oriana_b200.host_step import HostStreamedCAVI
    n, p, K = 5000, 2300, 12
    X = synth_counts_device(n, p, K, seed=6)
    np.random.seed(4)
    m = ZIGaP(X[:, :p], k=K, use_factors=False, tensor=True)
    s = m.state_dict()
    Xh = X[:, :p].to(torch.uint16).cpu().pin_memory()
    h = HostStreamedCAVI(Xh, K, s, dropout=True, slab_rows=2048)
    assert h._tensor and m.uses_tensor_path
    elbos = []
    for _ in range(3):
        m.step(); elbos.append(h.step())
    hs = h.state_dict()
    for k in FACTORS:
        assert relerr(hs[k], getattr(m, k).asarray()) < 1e-3, k
    for k in HYPER:
        assert relerr(hs[k], getattr(m, k).asarray()) < 1e-4, k
    want = m.elbo_trace[:3]
    assert np.max(np.abs(np.asarray(elbos) - want) / np.abs(want)) < 1e-5
    # a host-streamed run resumed from the device model's mid-run state reports, with its first step, the ELBO of that state
    # (slabs shorter than the kernels' accumulation chunk are chained differently from the resident matrix: 2e-5; slabs that
    # are multiples of the chunk -- the default -- agree to 1e-7, bench.py `elbo_first_vs_device`)
    h2 = HostStreamedCAVI(Xh, K, m.state_dict(), dropout=True, slab_rows=2048)
    e2 = h2.step()
    assert abs(e2 - m.elbo()) < 2e-5 * abs(e2), (e2, m.elbo())


def test_config5_slab_tensor_path_matches_cuda_core_path(cuda_lib):
    """BASELINE.json configs[4] (2M x 30k, K = 64, ~90 % zeros, 8 GPUs) at one slab of its cells: full gene axis and
    latent dimension (the KP = 64 plan with 32-wide sweep tiles), the sparsity of that configuration."""
    import torch
    from oriana.models import ZIGaP
    from oriana.singlecell import synth_counts_device
    n, p, K = 3072, 30_000, 64
    X = synth_counts_device(n, p, K, seed=12, zero_level=0.12)
    zeros = float((X[:, :p] == 0).float().mean())
    assert 0.85 < zeros < 0.95, zeros
    np.random.seed(6)
    m0 = ZIGaP(X[:, :p], k=K, use_factors=False, tensor=False)
    st = m0.state_dict(); st['X'] = X[:, :p]
    ms = ZIGaP(X[:, :p], k=K, use_factors=False, state=st, tensor=False)
    mt = ZIGaP(X[:, :p], k=K, use_factors=False, state=st, tensor=True)
    assert mt.uses_tensor_path and mt._KP == 64
    for _ in range(2):
        mt.step(); ms.step()
    for k in FACTORS:
        assert relerr(getattr(mt, k).asarray(), getattr(ms, k).asarray()) < 2e-3, k
    for k in HYPER + ('pi_d',):
        assert relerr(getattr(mt, k).asarray(), getattr(ms, k).asarray()) < 1e-4, k
    et, es = mt.elbo_trace, ms.elbo_trace
    assert np.max(np.abs(et - es) / np.abs(es)) < 1e-4, (et, es)
    assert (np.diff(et) > 0).all()


@pytest.mark.parametrize('shape,kw', [((4000, 1700, 12), {}), ((40000, 600, 8), {}), ((6000, 900, 20), dict(precise=True)),
                                      ((3000, 1000, 40), {})])
@pytest.mark.parametrize('model', ['zigap', 'gap'])
def test_deterministic_mode_repeats_bit_for_bit(cuda_lib, model, shape, kw):
    """ORI_F_DETERMINISTIC: chunk items add their accumulators in chunk order (tickets), ELBO terms and factor sums go through
    per-item / per-block slots summed in index order.  Three runs from the same state agree in every bit of every
    parameter after 6 steps (the plain kernels differ between runs by up to 1e-4 in single entries: float atomics), and
    agree with the plain kernels to the tensor path's tolerance.  Shapes: one chunk per gene block; three chunks (tickets
    at work); the fp32-grade plan (2048-cell chunks); the K = 64 plan."""
    from oracle import cavi_numpy as cn
    from oriana.models import GaP, ZIGaP
    from oriana.singlecell import CountMatrix
    n, p, K = shape
    X = cn.synth_counts(n, p, K, seed=n % 97)
    s = cn.init_state(X, K, np.random.default_rng(1), model)
    cls = ZIGaP if model == 'zigap' else GaP
    names = ('a1', 'a2', 'b1', 'b2', 'alpha1', 'alpha2', 'beta1', 'beta2') + (('pi_d',) if model == 'zigap' else ())

    def run(**extra):
        m = cls(CountMatrix(X), k=K, use_factors=False, state=s, tensor=True, **kw, **extra)
        assert m.uses_tensor_path
        for _ in range(6):
            m.step()
        return {k: getattr(m, k).asarray().copy() for k in names}, np.asarray(m.elbo_trace).copy()

    runs = [run(deterministic=True) for _ in range(3)]
    for got, tr in runs[1:]:
        for k in names:
            assert np.array_equal(got[k], runs[0][0][k]), (k, float(np.max(np.abs(got[k] - runs[0][0][k]))))
        # the trace also carries sum lgamma(X + 1), a constant formed once per model with double-precision atomics
        np.testing.assert_allclose(tr, runs[0][1], rtol=1e-13)
    plain, ptr = run()
    for k in names:
        assert relerr(plain[k], runs[0][0][k]) < 5e-3, k
    np.testing.assert_allclose(ptr, runs[0][1], rtol=1e-5)


@pytest.mark.parametrize('case', ['cuda_core_zigap', 'cuda_core_gap_chunks', 'sparse_cuda_core', 'sparse_tensor'])
def test_deterministic_mode_on_the_other_kernel_families(cuda_lib, case):
    """The same switch on the CUDA-core kernels (one CTA per row block, per-CTA / per-row-chunk slots summed in order) and
    on the sparse model (its gene update sums by a fixed shuffle tree): bit-identical repeats."""
    from oracle import cavi_numpy as cn, sparse_numpy as sn
    from oriana.models import GaP, SparseZIGaP, ZIGaP
    from oriana.singlecell import CountMatrix
    if case == 'cuda_core_zigap':
        n, p, K, cls, kw = 700, 450, 6, ZIGaP, dict(tensor=False)
    elif case == 'cuda_core_gap_chunks':
        n, p, K, cls, kw = 20000, 60, 9, GaP, dict(tensor=False)          # three row chunks in the gene pass
    elif case == 'sparse_cuda_core':
        n, p, K, cls, kw = 500, 300, 5, SparseZIGaP, dict(tensor=False)
    else:
        n, p, K, cls, kw = 4000, 1700, 12, SparseZIGaP, dict(tensor=True)
    X = cn.synth_counts(n, p, K, seed=n % 89)
    sparse = cls is SparseZIGaP
    s = sn.init_state(X, K, np.random.default_rng(2)) if sparse else \
        cn.init_state(X, K, np.random.default_rng(2), 'gap' if cls is GaP else 'zigap')
    names = ('a1', 'a2', 'b1', 'b2', 'alpha1', 'alpha2', 'beta1', 'beta2') + (() if cls is GaP else ('pi_d',)) \
        + (('p_s', 'pi_s') if sparse else ())

    def run(**extra):
        m = cls(CountMatrix(X), k=K, use_factors=False, state=s, **kw, **extra)
        assert m.uses_tensor_path == kw['tensor']
        for _ in range(5):
            m.step()
        return {k: getattr(m, k).asarray().copy() for k in names}

    runs = [run(deterministic=True) for _ in range(3)]
    for got in runs[1:]:
        for k in names:
            assert np.array_equal(got[k], runs[0][k]), (case, k, float(np.max(np.abs(got[k] - runs[0][k]))))
    plain = run()
    for k in names:
        # the sparse model's S-step (a sigmoid of a difference of large sums) amplifies the plain kernels' own run-to-run
        # spread to ~1e-2 after five steps
        assert relerr(plain[k], runs[0][k]) < (3e-2 if sparse else 1e-4), (case, k)


def test_deterministic_mode_size_limit_of_the_cuda_core_kernels(cuda_lib):
    from oriana.models import ZIGaP
    from oriana.singlecell import CountMatrix
    X = np.zeros((70000, 1000), dtype=np.uint8)                                   # 7e7 entries > 2^26
    with pytest.raises(ValueError):
        ZIGaP(CountMatrix(X), k=2, use_factors=False, tensor=False, deterministic=True)
