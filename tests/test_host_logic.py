"""CPU: host-side mirror of the reference interface, and the C-ABI surface (no compute without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT


def test_dimensions_examples_from_reference_docstring():
    """dims.py:91-102."""
    from oriana_b200 import Dimensions, IncompatibleShapeException
    d = Dimensions({'n': 10, 'm': 5, 'p': 5, 'k': 3, 'l': 4})
    assert repr(d('m,k ~ d,s')) == 'Dimension mapping (5, 3) <-> (3, 5, 1)'
    assert repr(d('n,k ~ s,d')) == 'Dimension mapping (10, 3) <-> (10, 3, 1)'
    assert repr(d('n,m,k ~ d,d,d')) == 'Dimension mapping (10, 5, 3) <-> (1, 150, 1)'
    assert repr(d('n,k,l,l ~ s,d,c,c')) == 'Dimension mapping (10, 3, 4, 4) <-> (10, 3, 16)'
    with pytest.raises(IncompatibleShapeException):
        d('n,k ~ s')
    rel = d('m,k ~ d,s')
    x = np.arange(15.).reshape(3, 5, 1)
    y = rel.reshape_func(x)
    assert y.shape == (5, 3) and np.array_equal(rel.inv_reshape_func(y), x)
    assert y[4, 2] == x[2, 4, 0]


def test_parameter_semantics():
    """parameters.py:8-32: float64 storage, [:] get/set, shape, asarray, in-place idiom."""
    from oriana_b200 import Parameter
    p = Parameter([[1, 2], [3, 4]])
    assert p.shape == (2, 2) and p[:].dtype == np.float64
    p[:] = p[:] + 1
    p[0, :] += 1
    assert np.array_equal(p.asarray(), [[3., 4.], [4., 5.]])
    assert np.array_equal(np.asarray(p), p[:])


def test_alias_package_import_paths():
    """The reference's import lines (test/test.py:5-7, zigap.py:5-9) work unchanged."""
    from oriana import Dimensions, Parameter  # noqa
    from oriana.nodes import Poisson, Gamma, Bernoulli, Multinomial, Multiply, Einsum, Transpose  # noqa
    from oriana.utils import digamma, inverse_digamma, sigmoid, logit  # noqa
    from oriana.models import FactorModel, GaP, ZIGaP  # noqa
    from oriana.inference import VariationalDistribution
    from oriana.singlecell import CountMatrix  # noqa
    v = VariationalDistribution()
    assert len(v) == 0


def test_bernoulli_and_multinomial_means():
    """test/test.py:35-57 (no special function involved: runs without a GPU)."""
    from oriana import Dimensions, Parameter
    from oriana.nodes import Bernoulli, Multinomial
    dims = Dimensions({'n': 2, 'm': 2, 'k': 2})
    p = Parameter([[0.02, 0.34], [0.62, 0.79]])
    y = Bernoulli(p, dims('m,k ~ d,d')).mean()
    np.testing.assert_almost_equal(np.asarray([[0.02, 0.34], [0.62, 0.79]]), y)
    assert y.dtype == np.float32                                   # bernoulli.py:45
    n = Parameter([[0, 1], [3, 1]])
    q = Parameter([[[0.50, 0.50], [0.21, 0.79]], [[0.43, 0.57], [0.89, 0.11]]])
    x = Multinomial(n, q, dims('n,m,k ~ d,d,c')).mean()
    np.testing.assert_almost_equal(x, q.asarray() * n.asarray()[..., None])


def test_node_forward_is_lazy():
    """test/test.py:82-96: a deterministic node changes only when forward() is called."""
    from oriana import Dimensions, Parameter
    from oriana.nodes import Multinomial, Multiply
    n = Parameter([[0, 1], [3, 1]])
    p = Parameter([[[0.50, 0.50], [0.21, 0.79]], [[0.43, 0.57], [0.89, 0.11]]])
    dims = Dimensions({'n': 2, 'm': 2, 'k': 2})
    m1 = Multinomial(n, p, dims('n,m,k ~ d,d,c'))
    m2 = Multinomial(n, Parameter(1 - p.asarray()), dims('n,m,k ~ d,d,c'))
    prod = Multiply(m1, m2)
    prod.forward()
    before = np.array(prod[:], copy=True)
    for _ in range(50):                      # the draws are random: resample until the inputs' product has moved
        m1.sample(); m2.sample()
        if not np.allclose(before, m1[:] * m2[:]):
            break
    assert np.array_equal(prod[:], before)   # untouched until forward() is called
    assert not np.allclose(prod[:], m1[:] * m2[:])
    prod.forward()
    np.testing.assert_almost_equal(prod[:], m1[:] * m2[:])


def test_count_matrix_types():
    from oriana.singlecell import CountMatrix
    from oriana import DatatypeException
    c = CountMatrix(np.arange(6).reshape(2, 3))
    assert c.shape == (2, 3) and c.T.shape == (3, 2)
    with pytest.raises(DatatypeException):
        CountMatrix([[1, 2], [3, 4]])                              # cmatrix.py:25-29


def test_count_matrix_reference_interface(tmp_path):
    """cmatrix.py:39-121: csv ingest, labels, label-based column access, row filtering, sparse export."""
    import pandas as pd
    from oriana.singlecell import CountMatrix
    df = pd.DataFrame(np.arange(12).reshape(4, 3), index=['c0', 'c1', 'c2', 'c3'], columns=['gA', 'gB', 'gC'])
    path = tmp_path / 'counts.csv'
    df.to_csv(path)
    c = CountMatrix.from_csv(str(path))
    assert c.shape == (4, 3)
    assert list(c.row_names) == ['c0', 'c1', 'c2', 'c3'] and list(c.col_names) == ['gA', 'gB', 'gC']
    np.testing.assert_array_equal(c.as_array(), df.values)
    np.testing.assert_array_equal(c['gB'], df['gB'].values)
    c['gB'] = np.array([7, 7, 7, 7])
    assert (c.as_array()[:, 1] == 7).all()
    sub = c.filter_rows(['c3', 'c1'], inplace=False)
    assert sub.shape == (2, 3) and list(sub.row_names) == ['c3', 'c1'] and c.shape == (4, 3)
    np.testing.assert_array_equal(sub.as_array()[:, 0], [9, 3])
    assert c.filter_rows(['c0', 'c2']) is c and c.shape == (2, 3)
    t = c.T
    assert t.shape == (3, 2) and list(t.row_names) == ['gA', 'gB', 'gC']
    assert c.as_sparse_matrix().shape == (2, 3) and c.as_sparse_matrix('csr').format == 'csr'
    with pytest.raises(KeyError):
        c['nope']
    plain = CountMatrix(np.zeros((2, 5), dtype=np.int64))
    assert list(plain.col_names) == [0, 1, 2, 3, 4] and list(plain.row_names) == [0, 1]


def test_block_generator_matches_reference_fixture():
    """singlecell/generation.py:68-86 under fixed seeds, against matrices recorded from the reference
    (oracle/make_golden.py generator): same draws in the same order, bit for bit."""
    from conftest import load_golden
    from oracle.make_golden import GENERATOR_CASES
    from oriana.singlecell import generate_factor_matrices
    g = load_golden('generator')
    for i, (args, kw) in enumerate(GENERATOR_CASES):
        np.random.seed(100 + i)
        X, U, V, labels = generate_factor_matrices(*args, **kw)
        np.testing.assert_array_equal(X, g['c%d_X' % i])
        np.testing.assert_array_equal(U, g['c%d_U' % i])
        np.testing.assert_array_equal(V, g['c%d_V' % i])
        np.testing.assert_array_equal(labels, g['c%d_labels' % i])
    with pytest.raises(ValueError):
        generate_factor_matrices(10, 10, 2, n_groups=3)      # fewer components than groups: the reference raises too


def test_count_matrix_ingest_helpers():
    """Row blocks of a sharded matrix tile it exactly; the narrow storage type follows the largest count."""
    import torch
    from oriana.singlecell import CountMatrix
    X = np.random.default_rng(0).poisson(3., size=(103, 7))
    c = CountMatrix(X)
    for world in (1, 2, 3, 8):
        blocks = [c.row_block(r, world) for r in range(world)]
        assert sum(b.shape[0] for b in blocks) == 103
        assert max(b.shape[0] for b in blocks) - min(b.shape[0] for b in blocks) <= 1
        np.testing.assert_array_equal(np.concatenate([b.as_array() for b in blocks]), X)
    assert CountMatrix.row_range(10, 3, 4) == (8, 10)
    assert c.narrow_dtype() == torch.uint8
    Y = X.copy(); Y[5, 2] = 300
    assert CountMatrix(Y).narrow_dtype() == torch.uint16
    Y[5, 2] = 70000
    assert CountMatrix(Y).narrow_dtype() is None
    assert CountMatrix(X + 0.5).narrow_dtype() is None
    cc = CountMatrix(np.minimum(Y, 1000)).to_compact(pin=False)
    np.testing.assert_array_equal(cc.dense().numpy(), np.minimum(Y, 1000))
    assert cc.row.numel() == 1
    sc = CountMatrix(np.minimum(Y, 1000)).to_sparse_counts(pin=False)
    np.testing.assert_array_equal(sc.dense().numpy(), np.minimum(Y, 1000))
    assert sc.row.numel() == 1 and sc.nz.numel() == int((Y != 0).sum())


def test_sparse_counts_round_trip():
    """SparseCounts (bitmap + non-zero bytes + escapes, the streaming format of the host-facing step) is lossless: ragged
    widths, all-zero rows and matrices, chunk boundaries inside the matrix, counts at and beyond the byte range."""
    import torch
    from oriana_b200.host_step import SparseCounts
    rng = np.random.default_rng(0)
    for n, p in ((7, 33), (50, 100), (33, 64), (5, 1), (64, 2049)):
        X = (rng.poisson(20, (n, p)) * (rng.random((n, p)) < 0.5)).astype(np.float32)
        X[rng.integers(0, n), rng.integers(0, p)] = 300.
        X[0, p - 1] = 255.; X[n - 1, 0] = 1000.; X[n // 2] = 0.
        sp = SparseCounts.from_tensor(torch.from_numpy(X), chunk_rows=3, pin=False)
        assert np.array_equal(sp.dense().numpy(), X), (n, p)
        assert sp.bitmap.shape == (n, (p + 31) // 32) and int(sp.rowoff[-1]) == int((X != 0).sum())
        lo, hi = sp.byte_range(n // 2, n // 2 + 1)
        assert lo == hi                                            # the empty row owns no bytes
        # bit l of word w = gene 32 w + l
        w = sp.bitmap.numpy().view(np.uint32)
        j = p - 1
        assert ((w[0, j // 32] >> np.uint32(j % 32)) & 1) == 1
    sp = SparseCounts.from_tensor(torch.zeros((4, 40)), pin=False)
    assert sp.nz.numel() == 0 and not sp.dense().any()
    assert SparseCounts.smaller_than_bytes(torch.zeros((4, 40))) and not SparseCounts.smaller_than_bytes(torch.ones((4, 40)))


def test_reference_driver_imports_resolve():
    """Every `from oriana... import ...` line of the reference's drivers and tests (main.py:5-6,
    experiments/clustering.py:5-6, test/test.py:5-7) resolves against the alias package."""
    import importlib
    wanted = {'oriana.models': ['GaP', 'SparseGaP', 'ZIGaP', 'SparseZIGaP', 'FactorModel'],
              'oriana.singlecell': ['CountMatrix', 'generate_factor_matrices', 'generate_u', 'generate_v'],
              'oriana': ['Dimensions', 'Parameter', 'DatatypeException', 'IncompatibleShapeException'],
              'oriana.nodes': ['Poisson', 'Gamma', 'Bernoulli', 'Multinomial', 'Multiply', 'Einsum', 'Transpose'],
              'oriana.utils': ['digamma', 'inverse_digamma', 'sigmoid', 'logit'],
              'oriana.inference': ['VariationalDistribution']}
    for mod, names in wanted.items():
        m = importlib.import_module(mod)
        for name in names:
            assert hasattr(m, name), (mod, name)
    from oriana.models import SparseGaP
    with pytest.raises(NotImplementedError):
        SparseGaP(None)


def test_header_is_plain_c(tmp_path):
    """include/oriana_b200.h is the drop-in boundary: it must compile as C99 (no C++ / torch types), and the struct
    mirrored by ctypes must have the size the C compiler gives it."""
    import subprocess
    src = tmp_path / 'hdr.c'
    src.write_text('#include <stdio.h>\n#include "oriana_b200.h"\n'
                   'int main(void) { printf("%zu\\n", sizeof(ori_problem_t)); return 0; }\n')
    exe = tmp_path / 'hdr'
    subprocess.run(['gcc', '-std=c99', '-Wall', '-Wextra', '-pedantic', '-Werror', '-I', os.path.join(ROOT, 'include'),
                    str(src), '-o', str(exe)], check=True)
    size = int(subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout)
    from oriana_b200 import _lib
    assert size == ctypes.sizeof(_lib.OriProblem)


def test_library_exports_every_declared_symbol():
    """The C-ABI library loads and exports exactly what include/oriana_b200.h declares."""
    from oriana_b200 import _lib
    header = open(os.path.join(ROOT, 'include', 'oriana_b200.h')).read()
    declared = sorted(set(re.findall(r'^(?:int|int64_t|unsigned long long)\s+(ori_\w+)\s*\(', header, flags=re.M)))
    assert declared == _lib.exported_symbols()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert _lib.load().ori_version() >= 100
    # struct layout agreed between the header and the ctypes mirror
    n_ptr = len(re.findall(r'^\s+(?:const\s+)?(?:float|double)\s*\*', header.split('typedef struct ori_problem')[1].split('} ori_problem_t')[0], flags=re.M))
    assert ctypes.sizeof(_lib.OriProblem) == 3 * 8 + 6 * 4 + 24 * 8 + 8 + 9 * 8 + 2 * 8 + 2 * 8 + 2 * 8 and n_ptr >= 20   # + the sparse block + xrow, xcol + thrU, thrV + det_ws, det_ws_doubles


def test_no_cpu_fallback():
    """Without a GPU every compute entry point raises; nothing silently runs on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from oriana_b200 import _lib
    from oriana.models import ZIGaP
    from oriana.utils import digamma
    with pytest.raises(_lib.OrianaB200Error):
        ZIGaP(np.ones((4, 5)), k=2, use_factors=False)
    with pytest.raises(_lib.OrianaB200Error):
        digamma(np.ones(3))
    # the product never imports the oracle
    import subprocess, sys
    out = subprocess.run([sys.executable, '-c', 'import oriana, oriana.models, sys; '
                          'print(any(m == "oracle" or m.startswith("oracle.") for m in sys.modules))'],
                         cwd=ROOT, capture_output=True, text=True)
    assert out.stdout.strip() == 'False', out


def test_row_blocks_cover_all_cells():
    from oriana_b200.sharding import RowSharding
    for n, w in ((10, 3), (1_000_000, 8), (7, 8), (0, 2)):
        blocks = [RowSharding.row_block(n, r, w) for r in range(w)]
        assert blocks[0][0] == 0 and blocks[-1][1] == n
        assert all(blocks[i][1] == blocks[i + 1][0] for i in range(w - 1))
        sizes = [b - a for a, b in blocks]
        assert max(sizes) - min(sizes) <= 1


def test_bench_initial_state_does_not_depend_on_the_sharding():
    """bench.py starts every world size from the same model: the row-side draws are keyed by the GLOBAL row block."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    n, p, K = 30_000, 50, 4
    whole = bench.initial_state(n, p, K, 0, n)
    for world in (2, 3, 8):
        parts = []
        for r in range(world):
            r0, r1 = n * r // world, n * (r + 1) // world
            s = bench.initial_state(n, p, K, r0, r1)
            parts.append(s['a1'])
            for k in ('b1', 'alpha1', 'beta1'):
                assert np.array_equal(s[k], whole[k])
        assert np.array_equal(np.concatenate(parts), whole['a1'])
    assert bench.elbo_vs_n1('no-such-config', 1, 1, 1, -5.0) == 0.0 and bench.elbo_vs_n1('no-such-config', 1, 1, 2, -5.0) is None


def test_bench_dump_outputs_writes_a_fixed_sample_of_the_state(tmp_path, monkeypatch):
    """bench.py --dump-outputs: state_dict() and the ELBO trace as float32 / float64 .npy files, the cell-side factors
    sampled on the same cells in every run, and the cell indices beside them."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setattr(bench, 'DUMP_CELLS', 64)
    rng = np.random.default_rng(0)
    n, p, K, r0 = 300, 40, 3, 1000
    state = dict(a1=rng.random((n, K)), a2=rng.random((n, K)), b1=rng.random((p, K)), b2=rng.random((p, K)),
                 alpha1=rng.random(K), pi_d=rng.random(p), iterations=7)

    class Model:
        def state_dict(self):
            return {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in state.items()}
    for d in ('one', 'two'):
        bench.dump_outputs(str(tmp_path / d), Model(), np.arange(8.), n, r0)
    names = sorted(os.listdir(tmp_path / 'one'))
    assert names == ['a1.npy', 'a2.npy', 'alpha1.npy', 'b1.npy', 'b2.npy', 'cells.npy', 'elbo_trace.npy', 'pi_d.npy']
    out = {f[:-4]: np.load(tmp_path / 'one' / f) for f in names}
    for f in names:
        assert np.array_equal(out[f[:-4]], np.load(tmp_path / 'two' / f))
    cells = out['cells'].astype(np.int64) - r0
    assert out['cells'].dtype == np.float64 and len(np.unique(cells)) == 64 and cells.min() >= 0 and cells.max() < n
    assert out['a1'].dtype == np.float32 and np.array_equal(out['a1'], state['a1'][cells].astype(np.float32))
    assert np.array_equal(out['b2'], state['b2'].astype(np.float32)) and out['pi_d'].dtype == np.float64


def test_reference_install_is_importable_and_steps():
    """The reference arm of bench.py runs the UNMODIFIED reference from oracle/_ref (installed by
    __graft_entry__.build(), oracle/refshim.py): it imports under the alias shim and steps."""
    import warnings
    from oracle import refshim, cavi_numpy as cn
    if not refshim.available():
        pytest.skip('no reference install and no checkout here')
    X = cn.synth_counts(40, 30, 3, seed=1)
    refshim.import_reference()
    try:
        from oriana.models import ZIGaP
        from oriana.singlecell import CountMatrix
        import oriana
        assert os.path.realpath(oriana.__file__).startswith(os.path.realpath(refshim.REFERENCE_ROOT))
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            np.random.seed(0)
            m = ZIGaP(CountMatrix(X), k=3, use_factors=False)
            m.step()
        assert np.isfinite(m.a1[:]).all() and m.a1[:].shape == (40, 3)
    finally:
        refshim.release_reference()
    import oriana as ours                        # the repo's alias package is importable again
    assert hasattr(ours, 'models') and 'oriana_b200' in ours.models.__name__
