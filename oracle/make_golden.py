"""Generate tests/golden/*.npz by running the UNMODIFIED reference (a checkout of it, or its install under oracle/_ref).

    [ORIANA_REFERENCE_CHECKOUT=<checkout>] python -m oracle.make_golden [seam | port | generator | nmf | ...]

For each case: seeded synthetic counts (oracle.cavi_numpy.synth_counts), `np.random.seed(1)`,
construct the reference model with `use_factors=False` (zigap.py:55-77, base.py:15-52), copy the
state vector out (this is the hand-off point of every parity run, SURVEY.md 8c/8d), then call the
reference's own `step()` (base.py:54-56) and record the trajectory.  Also records one raw call of
the reference's numba Z kernels (zigap.py:79-95, gap.py:67-80) and the special-function KATs of
test/test.py:13-32.
"""
import os
import sys
import numpy as np
from oracle import refshim, cavi_numpy as cn

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')

# name, model, n, p, K, steps recorded, zinb
CASES = [
    ('zigap_c1', 'ZIGaP', 100, 500, 2, (1, 2, 5, 50), True),     # BASELINE.json configs[0]
    ('gap_c1', 'GaP', 100, 500, 2, (1, 2, 5, 50), True),
    ('zigap_ragged', 'ZIGaP', 193, 331, 5, (1, 3, 10), False),   # nothing divides a tile; K odd
    ('gap_ragged', 'GaP', 131, 257, 7, (1, 3, 10), False),
    ('zigap_k10', 'ZIGaP', 300, 260, 10, (1, 4), True),          # K of configs[1]
]


GENERATOR_CASES = [((30, 50, 4), {}), ((17, 23, 7), dict(n_groups=3, sparsity_degree_in_v=0.3, zero_inflation_level=0.7)),
                   ((100, 500, 2), {})]    # the last one is the call of experiments/clustering.py:47 at configs[0] size


def write_generator_fixture():
    """The reference's synthetic-data generator (singlecell/generation.py:68-86) under a fixed seed."""
    refshim.import_reference()
    from oriana.singlecell import generate_factor_matrices
    out = {}
    for i, (args, kw) in enumerate(GENERATOR_CASES):
        np.random.seed(100 + i)
        X, U, V, labels = generate_factor_matrices(*args, **kw)
        out.update({'c%d_X' % i: X.astype(np.int64), 'c%d_U' % i: U, 'c%d_V' % i: V, 'c%d_labels' % i: labels.astype(np.int64)})
    np.savez_compressed(os.path.join(OUT, 'generator.npz'), **out)
    refshim.release_reference()
    print('generator written')


def write_sparse_generator_fixture():
    """The reference's own experiment (experiments/clustering.py:18-57): SparseZIGaP, use_factors=False, on a matrix from
    its block generator (counts up to ~1e5) -- trajectory and the deviance trace its driver prints."""
    refshim.import_reference()
    from oriana.models import SparseZIGaP
    from oriana.singlecell import CountMatrix, generate_factor_matrices
    np.random.seed(3)
    X, _, _, _ = generate_factor_matrices(100, 800, 2, sparsity_degree_in_v=0.9, beta=80, theta=0.5, n_groups=2,
                                          zero_inflation_level=0.5)
    rec = (1, 3, 6)
    np.random.seed(1)
    m = SparseZIGaP(CountMatrix(X), k=2, use_factors=False)
    out = {'model': 'SparseZIGaP', 'K': 2, 'tau': 0.5, 'steps': np.asarray(rec)}
    s0 = refshim.snapshot(m)
    out['X'] = s0.pop('X').astype(np.int32)
    for k, v in s0.items():
        out['s0_' + k] = v.astype(np.float32) if k == 'p_d' else v
    out['s0_deviance'] = np.float64(m.reconstruction_deviance())       # clustering.py:20, before any step
    for t in range(1, max(rec) + 1):
        m.step()
        if t in rec:
            st = refshim.snapshot(m); st.pop('X')
            for k, v in st.items():
                out['s%d_%s' % (t, k)] = v.astype(np.float32) if k == 'p_d' else v
            out['s%d_deviance' % t] = np.float64(m.reconstruction_deviance())
            out['s%d_explained' % t] = np.float64(m.explained_deviance())
    np.savez_compressed(os.path.join(OUT, 'sparse_gen.npz'), **out)
    refshim.release_reference()
    print('sparse_gen written')


def write_large_k_fixtures():
    """Latent dimensions of BASELINE.json configs[3] and configs[4] (K = 32, 64) at small n, p: the reference's own
    trajectories for the padded-K plans of the device kernels (KP = 32 with 64-wide sweep tiles, KP = 64 with 32-wide)."""
    refshim.import_reference()
    from oriana.models import ZIGaP, GaP
    from oriana.singlecell import CountMatrix
    for name, cls, n, p, K, rec in (('zigap_k32', ZIGaP, 150, 210, 32, (1, 3)), ('zigap_k64', ZIGaP, 130, 170, 64, (1, 3)),
                                    ('gap_k40', GaP, 140, 190, 40, (1, 3))):
        X = cn.synth_counts(n, p, K, seed=len(name) * 3 + K)
        np.random.seed(1)
        m = cls(CountMatrix(X), k=K, use_factors=False)
        out = {'model': cls.__name__, 'K': K, 'steps': np.asarray(rec)}
        s0 = refshim.snapshot(m)
        out['X'] = s0.pop('X').astype(np.int32)
        for k, v in s0.items():
            out['s0_' + k] = v.astype(np.float32) if k == 'p_d' else v
        # one raw call of the numba kernel on the initial expectations
        lU = np.ascontiguousarray(m.log_U_hat); lV = np.ascontiguousarray(m.log_V_hat)
        X32 = m.X[:].astype(np.float32)
        Zi = np.empty((n, K), np.float32); Zj = np.empty((p, K), np.float32)
        if cls is ZIGaP:
            ZIGaP.compute_Z_q_expectations(Zi, Zj, np.empty((p, K), np.float32), lU, lV, m.D_hat, X32)
        else:
            GaP.compute_Z_q_expectations(Zi, Zj, lU, lV, X32)
        out.update(z_log_U_hat=lU, z_log_V_hat=lV, z_Zi=Zi, z_Zj=Zj)
        for t in range(1, max(rec) + 1):
            m.step()
            if t in rec:
                st = refshim.snapshot(m); st.pop('X')
                for k, v in st.items():
                    out['s%d_%s' % (t, k)] = v.astype(np.float32) if k == 'p_d' else v
                out['s%d_U_hat' % t] = np.asarray(m.U_hat); out['s%d_V_hat' % t] = np.asarray(m.V_hat)
                out['s%d_log_U_hat' % t] = np.asarray(m.log_U_hat)
                out['s%d_log_V_hat' % t] = np.asarray(m.log_V_hat)
        np.savez_compressed(os.path.join(OUT, name + '.npz'), **out)
        print(name, 'written')
    refshim.release_reference()


def write_sparse_nmf_fixture():
    """main.py:29 exactly: SparseZIGaP(counts, k, use_factors=True) -- NMF-seeded factors with exact zeros -- with the
    deviance its loop prints (main.py:30, :42)."""
    refshim.import_reference()
    from oriana.models import SparseZIGaP
    from oriana.singlecell import CountMatrix
    X = cn.synth_counts(300, 400, 4, seed=13)
    rec = (1, 2, 4)
    np.random.seed(2)
    m = SparseZIGaP(CountMatrix(X), k=4, use_factors=True)
    out = {'model': 'SparseZIGaP', 'K': 4, 'tau': 0.5, 'steps': np.asarray(rec)}
    s0 = refshim.snapshot(m)
    out['X'] = s0.pop('X').astype(np.int32)
    for k, v in s0.items():
        out['s0_' + k] = v.astype(np.float32) if k == 'p_d' else v
    out['s0_deviance'] = np.float64(m.reconstruction_deviance())
    for t in range(1, max(rec) + 1):
        m.step()
        if t in rec:
            st = refshim.snapshot(m); st.pop('X')
            for k, v in st.items():
                out['s%d_%s' % (t, k)] = v.astype(np.float32) if k == 'p_d' else v
            out['s%d_deviance' % t] = np.float64(m.reconstruction_deviance())
            out['s%d_explained' % t] = np.float64(m.explained_deviance())
    np.savez_compressed(os.path.join(OUT, 'sparse_nmf.npz'), **out)
    refshim.release_reference()
    print('sparse_nmf written')


def write_loglik_fixture():
    """FactorModel.loglikelihood() (base.py:89-95) of the reference's GaP along the trajectories of the gap_* cases
    above (same seeds, so the states are the recorded ones).  ZIGaP has no such value: its X node is a Multiply node
    without `loglikelihood` (AttributeError in the reference), which the fixture records as a flag."""
    refshim.import_reference()
    from oriana.models import ZIGaP, GaP
    from oriana.singlecell import CountMatrix
    out = {}
    for name, model, n, p, K, rec, zinb in CASES:
        if model != 'GaP':
            continue
        X = cn.synth_counts(n, p, K, seed=len(name) * 7 + n, zinb=zinb)
        np.random.seed(1)
        m = GaP(CountMatrix(X), k=K, use_factors=False)
        for t in range(1, max(rec) + 1):
            m.step()
            if t in rec:
                out['%s_s%d' % (name, t)] = np.float64(m.loglikelihood())
    X = cn.synth_counts(20, 30, 2, seed=3)
    np.random.seed(1)
    z = ZIGaP(CountMatrix(X), k=2, use_factors=False)
    try:
        z.loglikelihood(); out['zigap_raises'] = np.bool_(False)
    except AttributeError:
        out['zigap_raises'] = np.bool_(True)
    # node-level logp() with the reference's own broadcasting (gamma.py:63-68, bernoulli.py:50-52, poisson.py:64-73)
    from oriana import Dimensions, Parameter
    from oriana.nodes import Gamma, Bernoulli, Poisson
    rng = np.random.default_rng(11)
    dims = Dimensions({'n': 6, 'k': 3, 'm': 4})
    al, be = rng.uniform(0.5, 4., 3), rng.uniform(0.5, 3., 3)
    g = Gamma(Parameter(al), Parameter(be), dims('n,k ~ s,d'))
    gs = rng.gamma(2., size=(6, 3)); g.buffer = gs
    out.update(node_gamma_alpha=al, node_gamma_beta=be, node_gamma_samples=gs, node_gamma_logp=g.logp())
    pi = rng.uniform(0.05, 0.95, 4)
    b = Bernoulli(Parameter(pi), dims('n,m ~ s,d'))
    bs = (rng.uniform(size=(6, 4)) < 0.5).astype(np.float64); b.buffer = bs
    out.update(node_bern_pi=pi, node_bern_samples=bs, node_bern_logp=b.logp())
    lam = rng.gamma(2., size=(6, 4)); lam[0, 0] = 0.; lam[1, 2] = 0.
    po = Poisson(Parameter(lam), dims('n,m ~ d,d'))
    ps = rng.poisson(2., size=(6, 4)).astype(np.float64); ps[0, 0] = 0.; ps[1, 2] = 3.; po.buffer = ps
    out.update(node_pois_lambda=lam, node_pois_samples=ps, node_pois_logp=po.logp())
    np.savez_compressed(os.path.join(OUT, 'loglik.npz'), **out)
    print('loglik written', {k: (float(v) if np.ndim(v) == 0 else np.shape(v)) for k, v in out.items()})


def write_nmf_fixture():
    """The reference's DEFAULT construction path, `use_factors=True` (base.py:38-40: a1, b1 seeded with sklearn NMF
    factors, many of them tiny or exactly 0, so E[log U] reaches -100 ... -1e15 and exp(E log U) underflows float32 on
    its own while the reference's exp(lU + lV) does not).  Post-construction state + trajectory, ZIGaP and GaP."""
    refshim.import_reference()
    from oriana.models import ZIGaP, GaP
    from oriana.singlecell import CountMatrix
    for name, cls, (n, p, K), seed in (('zigap_nmf', ZIGaP, (400, 300, 5), 9), ('gap_nmf', GaP, (260, 340, 6), 10)):
        rec = (1, 2, 4)
        X = cn.synth_counts(n, p, K, seed=seed, zinb=cls is ZIGaP)
        np.random.seed(0)
        m = cls(CountMatrix(X), k=K, use_factors=True)
        out = {'model': cls.__name__, 'K': K, 'steps': np.asarray(rec)}
        s0 = refshim.snapshot(m)
        out['X'] = s0.pop('X').astype(np.int32)
        for k, v in s0.items():
            out['s0_' + k] = v.astype(np.float32) if k == 'p_d' else v
        for t in range(1, max(rec) + 1):
            m.step()
            if t in rec:
                st = refshim.snapshot(m); st.pop('X')
                for k, v in st.items():
                    out['s%d_%s' % (t, k)] = v.astype(np.float32) if k == 'p_d' else v
        np.savez_compressed(os.path.join(OUT, name + '.npz'), **out)
        print(name, 'written')
    refshim.release_reference()


SEAM_CASES = [('seam_zigap', 'ZIGaP', (300, 220, 5)), ('seam_gap', 'GaP', (257, 190, 7)),
              ('seam_zigap_tc', 'ZIGaP', (2100, 1100, 12))]      # the last: a slab the device runs on the tcgen05 kernels
SEAM_ROWS, SEAM_D = 512, 8192          # at most this many rows of a1, a2 / b1, b2 and entries of D_hat are stored


def seam_problem(name):
    """Counts, initial state (the port's seeded `use_factors=False` bootstrap, oracle.cavi_numpy.init_state), number of
    steps and the row / entry strides of the stored sample of one case of SEAM_CASES."""
    model, (n, p, K) = {c[0]: c[1:] for c in SEAM_CASES}[name]
    X = cn.synth_counts(n, p, K, seed=11)
    s0 = cn.init_state(X, K, np.random.default_rng(3), model.lower())
    strides = dict(a=-(-n // SEAM_ROWS), b=-(-p // SEAM_ROWS), D=-(-n * p // SEAM_D))
    return model, K, X, s0, (5 if n * p < 1_000_000 else 2), strides


def seam_digest(s0):
    import hashlib
    h = hashlib.sha256()
    for k in sorted(s0):
        h.update(k.encode()); h.update(np.ascontiguousarray(s0[k]).tobytes())
    return h.hexdigest()


def write_seam_fixtures():
    """The reference stepped on its own numba Z kernel (zigap.py:79-95, gap.py:67-80): the twin that
    tests/test_reference_seam_gpu.py steps the B200 operator against.  The test regenerates the counts and the initial
    state from their seeds (checked by digest); the reference's state after the last step is stored on fixed strides:
    every a-th cell, every b-th gene and every D-th entry of D_hat, row-major."""
    import warnings
    refshim.import_reference()
    import oriana.models as ref_models
    from oriana.singlecell import CountMatrix
    for name, _, _ in SEAM_CASES:
        model, K, X, s0, steps, st = seam_problem(name)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            m = getattr(ref_models, model)(CountMatrix(X.copy()), k=K, use_factors=False)
            for k, v in s0.items():
                if k != 'X':
                    getattr(m, k)[:] = v
            m.update_expectations()
            assert np.array_equal(refshim.snapshot(m)['a1'], s0['a1'])
            for _ in range(steps):
                m.step()
        r = refshim.snapshot(m)
        out = {'model': model, 'K': K, 'steps': steps, 'digest': seam_digest(s0)}
        out.update({k: v for k, v in r.items() if v.ndim == 1})
        out.update({k: r[k][::st[k[0]]].astype(np.float32) for k in ('a1', 'a2', 'b1', 'b2')})
        if model == 'ZIGaP':
            out['D_hat'] = np.asarray(m.D_hat, dtype=np.float32).ravel()[::st['D']]
        np.savez_compressed(os.path.join(OUT, name + '.npz'), **out)
        print(name, 'written')
    refshim.release_reference()


def write_port_fixture():
    """ZIGaP 60 x 70, K = 3 from `np.random.seed(4)`: post-construction state and the state after 3 reference steps."""
    refshim.import_reference()
    from oriana.models import ZIGaP
    from oriana.singlecell import CountMatrix
    X = cn.synth_counts(60, 70, 3, seed=11)
    np.random.seed(4)
    m = ZIGaP(CountMatrix(X), k=3, use_factors=False)
    out = {'model': 'ZIGaP', 'K': 3, 'steps': np.asarray([3])}
    s0 = refshim.snapshot(m)
    out['X'] = s0.pop('X').astype(np.int32)
    out.update({'s0_' + k: v for k, v in s0.items()})
    for _ in range(3):
        m.step()
    st = refshim.snapshot(m); st.pop('X')
    out.update({'s3_' + k: v for k, v in st.items()})
    np.savez_compressed(os.path.join(OUT, 'zigap_port.npz'), **out)
    refshim.release_reference()
    print('zigap_port written')


def main():
    if sys.argv[1:] == ['seam']:
        return write_seam_fixtures()
    if sys.argv[1:] == ['port']:
        return write_port_fixture()
    if sys.argv[1:] == ['generator']:
        return write_generator_fixture()
    if sys.argv[1:] == ['nmf']:
        return write_nmf_fixture()
    if sys.argv[1:] == ['loglik']:
        return write_loglik_fixture()
    if sys.argv[1:] == ['sparse_gen']:
        return write_sparse_generator_fixture()
    if sys.argv[1:] == ['sparse_nmf']:
        return write_sparse_nmf_fixture()
    if sys.argv[1:] == ['large_k']:
        return write_large_k_fixtures()
    ref = refshim.import_reference()
    from oriana.models import ZIGaP, GaP
    from oriana.singlecell import CountMatrix
    from oriana import utils as rutils
    os.makedirs(OUT, exist_ok=True)

    for name, model, n, p, K, rec, zinb in CASES:
        X = cn.synth_counts(n, p, K, seed=len(name) * 7 + n, zinb=zinb)
        np.random.seed(1)
        m = (ZIGaP if model == 'ZIGaP' else GaP)(CountMatrix(X), k=K, use_factors=False)
        out = {'model': model, 'K': K, 'steps': np.asarray(rec)}
        s0 = refshim.snapshot(m)
        out['X'] = s0.pop('X').astype(np.int32)
        for k, v in s0.items():
            out['s0_' + k] = v.astype(np.float32) if k == 'p_d' else v
        # one raw call of the numba kernel on the initial expectations
        lU = np.ascontiguousarray(m.log_U_hat); lV = np.ascontiguousarray(m.log_V_hat)
        X32 = m.X[:].astype(np.float32)
        Zi = np.empty((n, K), np.float32); Zj = np.empty((p, K), np.float32)
        if model == 'ZIGaP':
            Z3 = np.empty((p, K), np.float32)
            ZIGaP.compute_Z_q_expectations(Zi, Zj, Z3, lU, lV, m.D_hat, X32)
        else:
            GaP.compute_Z_q_expectations(Zi, Zj, lU, lV, X32)
        out.update(z_log_U_hat=lU, z_log_V_hat=lV, z_Zi=Zi, z_Zj=Zj)
        for t in range(1, max(rec) + 1):
            m.step()
            if t in rec:
                st = refshim.snapshot(m); st.pop('X')
                for k, v in st.items():
                    out['s%d_%s' % (t, k)] = v.astype(np.float32) if k == 'p_d' else v
                out['s%d_U_hat' % t] = np.asarray(m.U_hat); out['s%d_V_hat' % t] = np.asarray(m.V_hat)
                out['s%d_log_U_hat' % t] = np.asarray(m.log_U_hat)
                out['s%d_log_V_hat' % t] = np.asarray(m.log_V_hat)
        np.savez_compressed(os.path.join(OUT, name + '.npz'), **out)
        print(name, 'written', {k: getattr(v, 'shape', None) for k, v in list(out.items())[:4]})

    # SparseZIGaP (sparse_zigap.py): trajectories + the reference's own convergence metrics (base.py:58-82)
    from oriana.models import SparseZIGaP
    for name, n, p, K, rec in (('sparse_k4', 120, 300, 4, (1, 2, 5)), ('sparse_ragged', 157, 203, 6, (1, 3, 8))):
        X = cn.synth_counts(n, p, K, seed=len(name) * 5 + p)
        np.random.seed(2)
        m = SparseZIGaP(CountMatrix(X), k=K, use_factors=False, tau=0.5)
        out = {'model': 'SparseZIGaP', 'K': K, 'tau': 0.5, 'steps': np.asarray(rec)}
        s0 = refshim.snapshot(m)
        out['X'] = s0.pop('X').astype(np.int32)
        for k, v in s0.items():
            out['s0_' + k] = v.astype(np.float32) if k == 'p_d' else v
        lU = np.ascontiguousarray(m.log_U_hat); lV = np.ascontiguousarray(m.log_Vprime_hat)
        St = (m.p_s[:] > m.tau).astype(np.float32)
        Z1 = np.empty((n, K), np.float32); Z2 = np.empty((p, K), np.float32); Z3 = np.empty((p, K), np.float32)
        SparseZIGaP.compute_Z_q_expectations(Z1, Z2, Z3, lU, lV, St, np.ascontiguousarray(m.S_hat), m.D_hat,
                                             m.X[:].astype(np.float32))
        out.update(z_log_U_hat=lU, z_log_Vp_hat=lV, z_S_tilde=St, z_S_hat=np.asarray(m.S_hat), z_DSZ=Z1, z_DZ=Z2, z_DZl=Z3)
        for t in range(1, max(rec) + 1):
            m.step()
            if t in rec:
                st = refshim.snapshot(m); st.pop('X')
                for k, v in st.items():
                    out['s%d_%s' % (t, k)] = v.astype(np.float32) if k == 'p_d' else v
                dev = m.reconstruction_deviance()          # mutates node buffers only (base.py:58-69)
                out['s%d_deviance' % t] = np.float64(dev)
                out['s%d_explained' % t] = np.float64(m.explained_deviance())
        np.savez_compressed(os.path.join(OUT, name + '.npz'), **out)
        print(name, 'written')

    # special-function known answers, produced by the reference's own utils (utils.py:9-51)
    x = np.concatenate([np.asarray([0.54, 6.2, 1.2, 0.3, 7.9, 4.5, 2.1]),          # test/test.py:24
                        np.logspace(-15, 8, 70), np.asarray([1.0, 2.0, 0.5, 1e-3, 3.0, 5.999, 6.0, 6.001])])
    y = np.concatenate([np.asarray([0.54, 6.2, 1.2, 0.3, 7.9, 4.5, 2.1]), np.linspace(-30, 12, 85)])
    z = np.concatenate([np.asarray([-2.3, 1.5, 0.45, -0.78, 5.3, -.2, 0.]), np.linspace(-40, 40, 81)])  # test.py:14
    q = np.concatenate([np.asarray([0.45, 0.001, 0.9987, 0.63, 0.745, 0.521, 0.32]),                    # test.py:19
                        np.asarray([0., 1., 1e-20, 1 - 1e-17, 1e-10, 1 - 1e-10])])
    np.savez_compressed(os.path.join(OUT, 'special.npz'),
                        x=x, digamma=rutils.digamma(x), trigamma=rutils.digamma_prime(x),
                        y=y, inverse_digamma=rutils.inverse_digamma(y),
                        z=z, sigmoid=rutils.sigmoid(z), q=q, logit=rutils.logit(q))
    print('special written')
    write_generator_fixture()
    write_nmf_fixture()
    write_sparse_generator_fixture()
    write_sparse_nmf_fixture()
    write_large_k_fixtures()
    write_seam_fixtures()
    write_port_fixture()


if __name__ == '__main__':
    main()
