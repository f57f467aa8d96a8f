"""Edge-weighted probes of the X-streaming passes against the float64 oracle (oracle/cavi_numpy.py, oracle/sparse_numpy.py,
oracle/zloop.c).

Random counts cannot see a boundary mistake at the TF32 tolerances: removing one ordinary entry of a 1111 x 777 problem
moves a1 / b1 by about 1e-3.  The problems built here put counts of 5000 and dominant factors on the rows and genes that
sit on an edge of the kernels -- own tile, CTA pair, sweep tile, 16-entry group, accumulation chunk, row pitch -- and
rare-path cases (dead cells, genes with pi <= 0 or pi = 1, zeros whose U_hat.V_hat passes the ELBO clamp) at group offsets
0, 15, 16 and in the last ragged tile.  The edges are read from the kernel sources, so they move when the code moves.

Each problem also runs with X stored as uint16 in HBM (ORI_F_X_U16, storage 'u16'): those are separate kernel instances,
with their own TMA boxes, swizzles, widening and an 8-count row pitch.  Widening a count is exact, so they are held to the
float32 tolerances.

`test_probes_move_their_checks_far_beyond_every_tolerance` and `test_probes_of_the_other_gpu_problems_move_their_checks`
(no GPU) apply each probe's mistake to the oracle's input on the very problems the GPU tests run, and show that it moves
what the probe is checked by at least 20 times the tolerance of the plan that checks it.

Tolerances (relative, floor 1e-6 of the array's maximum, as `relerr`), for TF32 operands / the fp32-grade mode / the
CUDA-core kernels: factors 3e-3 / 1e-4 / 2e-5; hyper-parameters and pi 2e-3 / 1e-4 / 2e-5 (beta1 of a K = 40 TF32 edge
state: 1.05e-3 measured, its mean over genes is carried by a few dominant ones); D_hat after the step 1e-3 / 2e-5 / 2e-5
absolute (it follows the factors' error times U_hat.V_hat: 4.3e-4 measured for TF32); ELBO 3e-4 / 2e-5 / 2e-5 of
`elbo_scale`.  That bound is wider than the 1e-4 of |ELBO| of test_tensor_path_gpu.py: on the TF32 edge states (counts of
5000 where U_hat.V_hat ~ 1e4) the ELBO of the loaded state was measured 1.25e-4 of |ELBO| off, and the ELBO after the
step of a small edge problem cancels to far less than its count terms.  The per-probe ELBO check (clamped zeros) is
relative to |ELBO|.  Measured on one B200 (1000 W power limit).
"""
import ctypes
import os
import re
import warnings

import numpy as np
import pytest

from conftest import ROOT, relerr

CSRC = os.path.join(ROOT, 'oriana_b200', 'csrc')
FACTORS = ('a1', 'a2', 'b1', 'b2')
HYPER = ('alpha1', 'alpha2', 'beta1', 'beta2')
BIG = 5000                # count of an edge entry
SCALE = 100.              # factor of the U_hat / V_hat of an edge cell / gene (U_hat.V_hat ~ 1e4 where two meet)


# --------------------------------------------------------------------------- kernel edges, read from the sources
def _grab(fname, pattern):
    with open(os.path.join(CSRC, fname)) as f:
        m = re.search(pattern, f.read())
    assert m, (fname, pattern)
    return [int(g) for g in m.groups()]


def kernel_constants():
    tc, simt = 'kernels_tc.cu', 'kernels_simt.cu'
    c = dict(TC_OWN=_grab(tc, r'constexpr int TC_OWN = (\d+);')[0],
             NCTA=_grab(tc, r'constexpr int NCTA = (\d+);')[0],
             GROUP=_grab(tc, r'const int nvalid = \(int\)min\(\(long long\)(\d+),')[0],
             CHUNK=_grab(tc, r'#define ORI_TC_CHUNK (\d+)')[0],
             CHUNK_PRECISE=_grab(tc, r'#define ORI_TC_CHUNK_PRECISE (\d+)')[0],
             PR_TR=_grab(simt, r'constexpr int PR_TR = (\d+);')[0],
             PR_TG=_grab(simt, r'constexpr int PR_TG = (\d+);')[0],
             PG_TG=_grab(simt, r'constexpr int PG_TG = (\d+);')[0],
             PG_TR=_grab(simt, r'constexpr int PG_TR = (\d+);')[0],
             SIMT_ROWS=_grab(simt, r'if \(rpc > (\d+)\) rpc = \1;')[0])
    c['SW_PRECISE'], c['SW_TILE'] = _grab(tc, r'static constexpr int SW = PRECISE \? (\d+) : (\d+) / KP;')
    return c


KC = kernel_constants()


def sweep_width(KP, precise):
    return KC['SW_PRECISE'] if precise else KC['SW_TILE'] // KP


def num_sms():
    """SMs of the device the tests run on (the split rules depend on it); 148, a B200's, without one."""
    try:
        import torch
        if torch.cuda.is_available():
            return torch.cuda.get_device_properties(0).multi_processor_count
    except ImportError:
        pass
    return 148


# the lines of `tc_partition` and of the deviance launcher that `tc_chunk` / `devi_chunk` restate: a change of either rule
# fails test_kernel_edges_are_read_from_the_sources instead of leaving the probes off the real seams
TC_SPLIT_RULE = [r'int tpc = (precise ? ORI_TC_CHUNK_PRECISE : (genes ? ORI_TC_CHUNK : 2 * ORI_TC_CHUNK)) / sw;',
                 r'if (tpc < 1) tpc = 1;', r'if (tpc > a.n_sw_tiles) tpc = a.n_sw_tiles;',
                 r'const int min_tpc = (128 / sw) > 1 ? 128 / sw : 1;',
                 r'while (!fixed_chain && (long long)a.n_own_units * cdiv(a.n_sw_tiles, tpc) < units / 2 && tpc > min_tpc) tpc = (tpc + 1) / 2;',
                 r'const int units = num_sms() / NCTA;',
                 r'a.tiles_per_chunk = a.n_sw_tiles;',
                 r'while ((long long)a.n_own_units * cdiv(a.n_sw_tiles, a.tiles_per_chunk) < 2LL * units && a.tiles_per_chunk > 4)',
                 r'a.tiles_per_chunk = (a.tiles_per_chunk + 1) / 2;']


def tc_chunk(own_total, sw_total, genes, sw, precise, fixed_chain=False, sms=None):
    """Sweep entries per work item of a tcgen05 pass (`tc_partition`): the nominal chunk, halved for small problems."""
    cd = lambda a, b: -(-a // b)
    sms = num_sms() if sms is None else sms
    units_own = cd(cd(own_total, KC['TC_OWN']), KC['NCTA'])
    n_sw = cd(sw_total, sw)
    tpc = (KC['CHUNK_PRECISE'] if precise else (KC['CHUNK'] if genes else 2 * KC['CHUNK'])) // sw
    tpc = min(max(tpc, 1), n_sw)
    min_tpc = max(128 // sw, 1)
    while not fixed_chain and units_own * cd(n_sw, tpc) < (sms // KC['NCTA']) // 2 and tpc > min_tpc:
        tpc = (tpc + 1) // 2
    return tpc * sw


def devi_chunk(n, p, sms=None):
    """Genes per work item of the deviance pass (its own split: one chunk per row block where that fills the machine)."""
    cd = lambda a, b: -(-a // b)
    sms = num_sms() if sms is None else sms
    sw = sweep_width(32, False)
    units_own = cd(cd(n, KC['TC_OWN']), KC['NCTA'])
    tpc = cd(p, sw)
    while units_own * cd(cd(p, sw), tpc) < 2 * (sms // KC['NCTA']) and tpc > 4:
        tpc = (tpc + 1) // 2
    return tpc * sw


# the lines of `launch_count_stats` / `launch_col_sums` (kernels_simt.cu) that `count_chunk_rows` restates (each launcher
# has its own copy of the rule, `n_rows` there, `P->n_rows` here); 148 is written into them, not read from the device
COUNT_SPLIT_RULE = [r'while (bx * chunks < 148 * 4 && P->n_rows / (chunks * 2) >= 16) chunks *= 2;',
                    r'const long long rpc = (P->n_rows + chunks - 1) / chunks;',
                    r'while (bx * chunks < 148 * 4 && n_rows / (chunks * 2) >= 16) chunks *= 2;',
                    r'const long long rpc = (n_rows + chunks - 1) / chunks;']


def count_chunk_rows(n, p):
    """Rows per chunk of k_count_stats / k_col_sums: the row range is halved until 128-gene blocks x chunks fill 4 CTAs per
    SM or a chunk would fall below 16 rows."""
    bx, chunks = -(-p // 128), 1
    while bx * chunks < 148 * 4 and n // (chunks * 2) >= 16:
        chunks *= 2
    return -(-n // chunks)


def periods(n, p, K, plan, sms=None, esz=4):
    """Tile, pair, group and chunk lengths of the plan along the cells and along the genes.  `esz`: bytes per count in
    HBM (4: float32, 2: uint16); X rows start on 16 bytes, so the row pitch is 4 or 8 counts."""
    pitch = 16 // esz
    if plan == 'simt':
        return ([KC['PR_TR'], KC['PG_TR'], KC['SIMT_ROWS']], [KC['PR_TG'], KC['PG_TG'], pitch])
    KP = 32 if K <= 32 else 64
    sw = sweep_width(KP, plan == 'precise')
    own, pair, g = KC['TC_OWN'], KC['NCTA'] * KC['TC_OWN'], KC['GROUP']
    rows = [own, pair, sw, g, tc_chunk(p, n, True, sw, plan == 'precise', sms=sms)]
    genes = [own, pair, sw, g, tc_chunk(n, p, False, sw, plan == 'precise', sms=sms), pitch]
    return rows, genes


def edges(N, pers):
    s = {0, N - 1}
    for P in pers:
        if P < N:
            for b in (P, 2 * P, (N - 1) // P * P):
                s.update(i for i in (b - 1, b) if 0 <= i < N)
    return sorted(s)


def _offsets(N, base):
    """Group offsets 0, 15, 16 after `base`, and one index in the last ragged tile."""
    g = KC['GROUP']
    return [i for i in (base, base + g - 1, base + g, N - 1 - base // (2 * g)) if 0 <= i < N]


# --------------------------------------------------------------------------- probe problems
def _pd(s, pi_prev, V_eff=None):
    """p_d generated by (pi_prev, U_hat, V_hat) with the reference's floors and the X != 0 override (zigap.py:131-136)."""
    from oracle import cavi_numpy as cn
    U = s['a1'] / s['a2']
    V = s['b1'] / s['b2'] if V_eff is None else V_eff
    with np.errstate(over='ignore'):
        pd = cn.sigmoid(cn.logit(pi_prev)[None, :] - U @ V.T)
    pd[:, pi_prev <= 0] = 1e-10
    pd[:, pi_prev >= 1] = 1. - 1e-10
    pd[s['X'] != 0] = 1. - 1e-10
    return pd


def _refresh(s, start, model):
    """Make the dropout side of a probed state consistent with its X and factors again."""
    if model == 'gap':
        return s
    if start == 'init':
        s['p_d'] = (s['X'] > 0).astype(np.float64)
        s.pop('pi_prev', None)
    else:
        s['p_d'] = _pd(s, s['pi_prev'], s.get('V_eff_prev'))
    s['pi_d'] = s['p_d'].mean(axis=0)
    return s


def _base(n, p, K, model, start, seed, steps=2, dtype=np.float64):
    from oracle import cavi_numpy as cn, sparse_numpy as sn
    X = cn.synth_counts(n, p, K, seed=seed)
    rng = np.random.default_rng(seed)
    if model == 'sparse':
        s = sn.init_state(X, K, rng)
    else:
        s = cn.init_state(X, K, rng, model)
    if start == 'mid':
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            for _ in range(steps):
                if model != 'gap':
                    pi_prev = s['pi_d'].copy()
                    if model == 'sparse':
                        V_eff = (s['p_s'].astype(np.float32).astype(np.float64)) * s['b1'] / s['b2']
                if model == 'sparse':
                    sn.step(s, dtype=dtype)
                else:
                    cn.step(s, quirk=False, dtype=dtype)
        if model != 'gap':
            s['pi_prev'] = pi_prev
        if model == 'sparse':
            s['V_eff_prev'] = V_eff
    s['X'] = np.array(s['X'], dtype=np.int64)
    return s


def edge_case(n, p, K, model, plan, start='mid', kind='edges', seed=None, steps=2, dtype=np.float64, sms=None, pers=None,
              esz=4):
    """(state, probes) of an edge-weighted problem.

    kind='edges': counts of 5000 on (edge cell, edge gene) pairs, the U_hat of one edge cell per edge gene and the V_hat
    of one edge gene per edge cell scaled by 100 (more on large axes), and every other (edge cell, edge gene) pair made a zero whose U_hat.V_hat passes the ELBO
    clamp: an edge gene's a2 share and an edge cell's b2 share come from its one count.  kind='rare': dead cells, genes with pi <= 0 and with pi = 1, and zeros past the
    clamp, each at group offsets 0, 15, 16 and in the last ragged tile.

    A probe is a dict: name, `mutate` (the mistake a kernel could make with it: the entry / row / gene dropped or given
    its neighbour's value) and `checks` [(key, index)] (what a step of the state is checked by)."""
    seed = (n * 7919 + p * 31 + K) % 100003 if seed is None else seed
    s = _base(n, p, K, model, start, seed, steps, dtype)
    X = s['X']
    sparse = model == 'sparse'
    probes = []

    def nb(i, N, taken=()):
        """The nearest index that carries no probe of the same kind."""
        for d in range(1, N):
            for c in (i - d, i + d):
                if 0 <= c < N and c not in taken:
                    return c
        return i

    if kind == 'edges':
        rp, gp = periods(n, p, K, plan, sms, esz) if pers is None else pers
        # an edge factor must dominate a sum over every cell / gene: the scale grows with the extent
        sr, sg = SCALE * max(1., n / 1024.), SCALE * max(1., p / 1024.)
        R, G = edges(n, rp), edges(p, gp)
        L = max(len(R), len(G))
        hits = {(R[k % len(R)], G[k % len(G)]) for k in range(L)}
        zeros = {(R[k % len(R)], G[(k + 1) % len(G)]) for k in range(L)} - hits if len(G) > 1 else set()
        X[np.ix_(R, G)] = 0          # every other (edge cell, edge gene) pair: a zero past the clamp
        for (i, j) in hits:
            X[i, j] = BIG
        # one dominant factor per sum: the first edge cell of each edge gene's counts and the first edge gene of each edge
        # cell's counts are scaled (a gene that took the counts of several scaled cells would share its b2 among them)
        # The new U_hat that b2 sums is formed by the step itself, so a cell's probe reaches b2 through its D_hat and its
        # share of the den ratios only: above ~4k cells that share is too small for the TF32 tolerance, and the edge cells
        # of such problems are probed by their counts alone
        SR = sorted({min(i for (i, j2) in hits if j2 == j) for j in {j for _, j in hits}}) if n <= 4096 else []
        SG = sorted({min(j for (i2, j) in hits if i2 == i) for i in {i for i, _ in hits}})
        if not sparse:
            s['a1'][SR] *= sr
            s['b1'][SG] *= sg
        hit_genes = {}
        for (i, j) in hits:
            hit_genes.setdefault(i, set()).add(j)
        for (i, j) in sorted(hits):
            def mut(t, i=i, j=j):
                k = nb(j, p, hit_genes[i])       # the nearest gene of the row without a probe count, else dropped
                t['X'][i, j] = t['X'][i, k] if k != j else 0
            probes.append(dict(name='count(%d,%d)' % (i, j), mutate=mut, checks=[('a1', (i, slice(None))), ('b1', (j, slice(None)))]))
        if model == 'zigap':         # GaP's a2 / b2 are plain sums over every gene / cell: no one factor dominates them
            for j in SG:
                def mut(t, j=j):
                    k = nb(j, p, G)
                    t['b1'][j] = t['b1'][k] if k != j else t['b1'][j] / sg
                probes.append(dict(name='V_hat(gene %d)' % j, mutate=mut, checks=[('a2', (slice(None), slice(None)))]))
            for i in SR:
                def mut(t, i=i):
                    k = nb(i, n, R)
                    t['a1'][i] = t['a1'][k] if k != i else t['a1'][i] / sr
                probes.append(dict(name='U_hat(cell %d)' % i, mutate=mut, checks=[('b2', (slice(None), slice(None)))]))
        if model != 'gap':
            for (i, j) in sorted(zeros):
                def mut(t, i=i, j=j):
                    t['X'][i, j] = max(int(t['X'][i, nb(j, p)]), 1)
                probes.append(dict(name='clamped zero(%d,%d)' % (i, j), mutate=mut,
                                   checks=[('p_d', (i, j)), ('b2', (j, slice(None))), ('elbo0', None)]))
    else:
        # each kind on at most a quarter of its axis, so that no probe leaves the problem without live cells or genes
        quarter = lambda idx, N: idx[:N // 4]
        dead = quarter(_offsets(n, 0), n)
        ulim_rows = quarter([i for i in _offsets(n, 2 * KC['GROUP']) if i not in dead], n)
        pi0 = quarter(_offsets(p, 0), p)
        pi1 = quarter([j for j in _offsets(p, 2 * KC['GROUP']) if j not in pi0], p) if model != 'gap' else []
        ulim_genes = quarter([j for j in _offsets(p, 4 * KC['GROUP']) if j not in pi0 + pi1], p)
        live = [j for j in range(p) if j not in pi0]
        X[:, pi0] = 0
        for j in pi1:
            X[:, j] = np.maximum(X[:, j], 1)
        if model != 'gap' and start == 'mid':
            s['pi_prev'][pi0] = 0.
            s['pi_prev'][pi1] = 1.
        if not sparse:
            s['a1'][ulim_rows] *= SCALE
            s['b1'][ulim_genes] *= SCALE
        for i in ulim_rows:
            X[i, ulim_genes] = 0
        s['a1'][dead] = 1e-15
        X[np.ix_(dead, live)] = np.maximum(X[np.ix_(dead, live)], 1)     # counts that a dead cell must assign to nobody
        for i in dead:
            def mut(t, i=i):
                t['a1'][i] = t['a1'][nb(i, n, dead)]
            probes.append(dict(name='dead cell %d' % i, mutate=mut, checks=[('a1', (i, slice(None)))]))
        for j in pi0:
            def mut(t, j=j):
                k = nb(j, p)
                t['X'][:, j] = t['X'][:, k] if k not in pi0 and t['X'][:, k].any() else np.maximum(t['X'][:, j], 1)
                if 'pi_prev' in t:
                    t['pi_prev'][j] = 0.5
            probes.append(dict(name='pi<=0 gene %d' % j, mutate=mut, checks=[('b1', (j, slice(None))), ('b2', (j, slice(None)))]))
        for j in pi1:
            def mut(t, j=j):
                t['X'][::2, j] = 0
                if 'pi_prev' in t:
                    t['pi_prev'][j] = 0.5
            probes.append(dict(name='pi=1 gene %d' % j, mutate=mut, checks=[('b2', (j, slice(None))), ('pi_d', j)]))
        if model != 'gap':
            for i in ulim_rows:
                for j in ulim_genes:
                    def mut(t, i=i, j=j):
                        t['X'][i, j] = max(int(t['X'][i, nb(j, p)]), 1)
                    probes.append(dict(name='clamped zero(%d,%d)' % (i, j), mutate=mut,
                                       checks=[('p_d', (i, j)), ('b2', (j, slice(None))), ('elbo0', None)]))
    return _refresh(s, start, model), probes


def oracle_step(s, model, dtype=np.float64, elbo=True):
    from oracle import cavi_numpy as cn, sparse_numpy as sn
    t = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in s.items()}
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        if model == 'sparse':
            sn.step(t, dtype=dtype)
        else:
            elbo0 = cn.elbo(s, guard32=True) if elbo else None
            cn.step(t, quirk=False, dtype=dtype)
            if elbo:
                t['elbo0'] = elbo0
    return t


def probe_error(got, want, key, idx):
    """Error of one probe's check: relative (relerr) for parameters and the ELBO, absolute for p_d / D_hat."""
    if key == 'elbo0':
        return abs(got[key] - want[key]) / abs(want[key])
    a, b = np.asarray(got[key]), np.asarray(want[key])
    if key == 'p_d':
        return float(np.max(np.abs(a[idx] - b[idx])))
    return relerr(np.atleast_1d(a[idx]), np.atleast_1d(b[idx]))


# tolerances per plan: factors, hyper-parameters / pi, D_hat (absolute), ELBO (relative)
TOL = {'tf32': (3e-3, 2e-3, 1e-3, 3e-4), 'precise': (1e-4, 1e-4, 2e-5, 2e-5), 'simt': (2e-5, 2e-5, 2e-5, 2e-5),
       'sparse_precise': (2e-5, 2e-5, 2e-5, 2e-5), 'sparse_tf32': (3e-3, 5e-3, 3e-4, 1e-4)}


def tol_of(plan, key):
    return TOL[plan][{'p_d': 2, 'pi_d': 1, 'elbo0': 3, 'elbo1': 3}.get(key, 1 if key in HYPER else 0)]


def elbo_scale(s, want):
    """|ELBO| + the total count + the number of entries.  An error in log den moves the ELBO in proportion to the counts,
    every entry adds terms of order one, and these terms cancel to a sum far smaller than themselves on the small edge
    problems (the ELBO after one step of a 128 x 15 problem is about -1300, its count terms alone are ~1e5)."""
    X = np.asarray(s['X'])
    return abs(want) + float(X.sum()) + X.size


# covering set of (n, p): every listed n and p appears, each tile / pair / group / chunk edge is crossed in both passes
SHAPES = [(1, 65), (127, 2049), (128, 15), (129, 63), (255, 17), (256, 1), (257, 64), (2049, 33), (16385, 16)]
PLANS = [('zigap', 'tf32', 20), ('zigap', 'tf32', 40), ('gap', 'tf32', 20), ('gap', 'tf32', 40),
         ('zigap', 'precise', 12), ('zigap', 'simt', 20), ('gap', 'simt', 12)]
SPARSE_SHAPES = [(257, 66, 8), (2049, 33, 20), (129, 2049, 12)]
NOMINAL = (4097, 3328, 12)       # fp32-grade gene pass: 13 gene pairs x 3 chunks fill the machine, no halving
NOMINAL_PERIODS = ([KC['CHUNK_PRECISE']], [2 * KC['TC_OWN']])      # its chunk seams (cells), its CTA pairs (genes)
# TF32 gene pass at its nominal 16384-cell chunk (configs 4 and 5 run it): 19 gene pairs x 2 chunks fill the machine
NOMINAL_TF32 = (16385, 4609)
NOMINAL_TF32_PERIODS = ([KC['CHUNK']], [2 * KC['TC_OWN']])
# storage of X in HBM: bytes per count.  uint16 (ORI_F_X_U16) runs the kernels' uint16 instances: their own TMA boxes and
# swizzles, their own widening and an 8-count row pitch
ESZ = {'f32': 4, 'u16': 2}


def with_storage(plans, ids):
    """pytest params of (plan, storage): the float32 runs keep the plan's id, the uint16 runs add '-u16'."""
    return [pytest.param(pl, st, id=ids(pl) + ('' if st == 'f32' else '-' + st)) for st in ESZ for pl in plans]


plan_id = lambda t: '%s-%s-k%d' % t


# --------------------------------------------------------------------------- CPU checks of the harness itself
def test_kernel_edges_are_read_from_the_sources():
    assert KC['TC_OWN'] == 128 and KC['NCTA'] == 2 and KC['GROUP'] == 16
    assert sweep_width(32, False) == 64 and sweep_width(64, False) == 32 and sweep_width(32, True) == 32
    assert KC['CHUNK'] == 16384 and KC['CHUNK_PRECISE'] == 2048
    assert KC['PR_TG'] == 32 and KC['PG_TG'] == 128 and KC['SIMT_ROWS'] == 8192
    # the nominal chunks of large problems, the halved chunks of small ones, the fixed chain of host-streamed slabs
    assert tc_chunk(20000, 1_000_000, True, 64, False) == 16384
    assert tc_chunk(1_000_000, 40000, False, 64, False) == 32768
    assert tc_chunk(2048, 33000, False, 64, False, fixed_chain=True) == 32768
    assert tc_chunk(64, 2049, False, 64, False) == 128
    assert tc_chunk(20000, 1_000_000, True, 32, True) == 2048
    assert edges(257, [128]) == [0, 127, 128, 255, 256]
    with open(os.path.join(CSRC, 'kernels_tc.cu')) as f:
        src = f.read()
    for line in TC_SPLIT_RULE:
        assert line in src, line
    assert devi_chunk(257, 2049, sms=148) == 192
    with open(os.path.join(CSRC, 'kernels_simt.cu')) as f:
        src = f.read()
    for line in COUNT_SPLIT_RULE:
        assert line in src, line
    assert count_chunk_rows(3000, 127) == count_chunk_rows(3000, 257) == 24 and count_chunk_rows(20, 129) == 20
    assert tc_chunk(NOMINAL[1], NOMINAL[0], True, sweep_width(32, True), True, sms=148) == KC['CHUNK_PRECISE']
    for KP in (32, 64):
        assert tc_chunk(NOMINAL_TF32[1], NOMINAL_TF32[0], True, sweep_width(KP, False), False, sms=148) == KC['CHUNK']
    assert periods(129, 63, 12, 'tf32', esz=2)[1][-1] == 8 and periods(129, 63, 12, 'simt', esz=2)[1][-1] == 8


def _power(n, p, K, model, plan, kind, start, pers=None, esz=4):
    """Probes of one problem whose mistake moves their check by less than 20x the plan's tolerance."""
    s, probes = edge_case(n, p, K, model, 'tf32' if model == 'sparse' else plan, start, kind, sms=148, pers=pers, esz=esz)
    assert probes, (n, p, kind)
    base = oracle_step(s, model)
    weak = []
    for pr in probes:
        t = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in s.items()}
        pr['mutate'](t)
        mut = oracle_step(_refresh(t, start, model), model, elbo=any(k == 'elbo0' for k, _ in pr['checks']))
        checks = [(k, idx) for k, idx in pr['checks'] if k in mut]
        moved = [probe_error(mut, base, k, idx) / tol_of(plan, k) for k, idx in checks]
        if not max(moved) >= 20:
            weak.append((n, p, pr['name'], max(moved)))
    return weak


@pytest.mark.parametrize('start', ['mid', 'init'])
@pytest.mark.parametrize('kind', ['edges', 'rare'])
@pytest.mark.parametrize('plan,storage', with_storage(PLANS, plan_id))
def test_probes_move_their_checks_far_beyond_every_tolerance(plan, storage, kind, start):
    """Over the problems of test_one_step_of_every_plan_matches_the_oracle_on_the_probes: every probe's mistake, applied to
    the oracle's input, moves what the probe is checked by at least 20x the plan's tolerance, so a kernel that drops or
    misplaces the probe cannot pass.  The uint16 problems differ by their row pitch of 8 counts."""
    model, pl, K = plan
    if model == 'gap' and start == 'init' and kind == 'edges':
        pytest.skip('the same problems as the mid-run start')
    if kind == 'rare' and storage == 'u16':
        pytest.skip('the rare-path probes do not depend on the row pitch')
    weak = []
    for (n, p) in SHAPES:
        weak += _power(n, p, K, model, pl, kind, start, esz=ESZ[storage])
    assert not weak, weak


@pytest.mark.parametrize('case', ['sparse', 'sparse-u16', 'nominal_chunk', 'tf32_nominal_chunk-k40', 'tf32_nominal_chunk-k20'])
def test_probes_of_the_other_gpu_problems_move_their_checks(case):
    """The same for the SparseZIGaP problems (both tensor modes use them; the looser TF32 tolerance counts), for the
    fp32-grade problem at its nominal 2048-cell chunk and for the TF32 problem at its nominal 16384-cell chunk (one float64
    oracle step of it at K = 40 takes ~5 s, its ELBO ~7 s: only probes checked by the ELBO compute it)."""
    weak = []
    if case.startswith('sparse'):
        for (n, p, K) in SPARSE_SHAPES:
            for kind in (('edges', 'rare') if case == 'sparse' else ('edges',)):
                for start in ('mid', 'init'):
                    weak += _power(n, p, K, 'sparse', 'sparse_tf32', kind, start, esz=2 if case == 'sparse-u16' else 4)
    elif case == 'nominal_chunk':
        n, p, K = NOMINAL
        weak += _power(n, p, K, 'zigap', 'precise', 'edges', 'mid', pers=NOMINAL_PERIODS)
    else:
        (n, p), K = NOMINAL_TF32, int(case[-2:])
        weak += _power(n, p, K, 'zigap', 'tf32', 'edges', 'mid', pers=NOMINAL_TF32_PERIODS)
    assert not weak, weak


# --------------------------------------------------------------------------- GPU: one step of every plan
def _model(s, model, plan, storage='f32', **kw):
    """The device model of state `s`.  storage='u16': X handed in as uint16 and kept as uint16 in HBM at any size (the
    models choose uint16 storage only where float32 would not fit the device, `oriana_b200.problem.counts_storage`)."""
    import torch
    from oriana.models import GaP, SparseZIGaP, ZIGaP
    from oriana.singlecell import CountMatrix
    from oriana_b200 import problem
    cls = dict(zigap=ZIGaP, gap=GaP, sparse=SparseZIGaP)[model]
    K = s['a1'].shape[1]
    kw = dict(kw)
    kw.setdefault('tensor', plan != 'simt')
    if plan == 'precise' or (model == 'sparse' and plan != 'simt' and 'precise' not in kw):
        kw.setdefault('precise', True)
    if storage == 'f32':
        return cls(CountMatrix(s['X']), k=K, use_factors=False, state=s, **kw)
    assert storage == 'u16' and 0 <= s['X'].min() and s['X'].max() <= 65535
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(problem, 'counts_storage', lambda u16, *args: torch.uint16 if u16 else torch.float32)
        m = cls(CountMatrix(s['X'].astype(np.uint16)), k=K, use_factors=False, state=s, **kw)
    # no silent float32 run
    assert m.counts_dtype == torch.uint16 and m._X.element_size() == 2 and m._ldx % 8 == 0
    return m


def _check_step(m, s, probes, model, plan, ref=None, elbo=True):
    """One device step against one oracle step from the same state: every array, the ELBO before and after the step,
    then every probe separately.  Prints the measured errors before it judges them."""
    from oracle import cavi_numpy as cn
    ref = oracle_step(s, model) if ref is None else ref
    elbo_keys = ('elbo0', 'elbo1') if model != 'sparse' and elbo else ()
    m.step()
    got = {k: getattr(m, k).asarray() for k in FACTORS + HYPER}
    keys = FACTORS + HYPER
    if model != 'gap':
        got['pi_d'] = m.pi_d.asarray()
        got['p_d'] = m.D_hat.astype(np.float64)
        keys += ('pi_d', 'p_d')
    errs, rel = {}, {}
    for k in keys:
        errs[k] = probe_error(got, ref, k, slice(None))
    if elbo_keys:
        got['elbo0'], got['elbo1'] = float(m.elbo_trace[0]), m.elbo()
        want1 = cn.elbo(ref, guard32=True)
        for k, want in (('elbo0', ref['elbo0']), ('elbo1', want1)):
            rel[k] = abs(got[k] - want) / abs(want)
            errs[k] = abs(got[k] - want) / elbo_scale(s, want)
    worst = {}
    for pr in probes:
        for k, idx in pr['checks']:
            if k in got and (k != 'elbo0' or elbo_keys):
                worst[(pr['name'], k)] = probe_error(got, ref, k, idx)
    errs['probes'] = max([e / tol_of(plan, k[1]) for k, e in worst.items()], default=0.)      # in units of the tolerance
    print('%s %s %dx%d: %s  ELBO/|ELBO| %s' % (model, plan, s['X'].shape[0], s['X'].shape[1],
                                               {k: '%.1e' % v for k, v in errs.items()}, {k: '%.1e' % v for k, v in rel.items()}))
    for k in keys + elbo_keys:
        assert np.isfinite(errs[k]) and errs[k] < tol_of(plan, k), (k, errs[k], tol_of(plan, k))
    for (name, k), e in worst.items():
        assert e < tol_of(plan, k), (name, k, e, tol_of(plan, k))
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize('start', ['mid', 'init'])
@pytest.mark.parametrize('kind', ['edges', 'rare'])
@pytest.mark.parametrize('plan,storage', with_storage(PLANS, plan_id))
def test_one_step_of_every_plan_matches_the_oracle_on_the_probes(cuda_lib, plan, storage, kind, start):
    model, pl, K = plan
    if model == 'gap' and start == 'init' and kind == 'edges':
        pytest.skip('GaP has no dropout state: the initial and the mid-run start differ only in the factors')
    for (n, p) in SHAPES:
        s, probes = edge_case(n, p, K, model, pl, start, kind, esz=ESZ[storage])
        m = _model(s, model, pl, storage)
        assert m.uses_tensor_path == (pl != 'simt')
        if pl != 'simt':
            assert m._KP == (32 if K <= 32 else 64) and m.precise == (pl == 'precise')
        _check_step(m, s, probes, model, pl)


@pytest.mark.gpu
@pytest.mark.parametrize('start', ['mid', 'init'])
@pytest.mark.parametrize('plan,storage', with_storage(['sparse_precise', 'sparse_tf32'], str))
def test_sparse_model_on_the_probes(cuda_lib, plan, storage, start):
    """SparseZIGaP, tcgen05 kernels: fp32-grade (its default) and TF32 operands.  The S update amplifies operand rounding
    (a sigmoid of a difference of large sums), so p_s is checked at 20x the factor tolerance."""
    for (n, p, K) in SPARSE_SHAPES:
        for kind in ('edges', 'rare'):
            s, probes = edge_case(n, p, K, 'sparse', 'tf32', start, kind, esz=ESZ[storage])
            m = _model(s, 'sparse', plan, storage, precise=(plan == 'sparse_precise'), tensor=True)
            assert m.uses_tensor_path and m.precise == (plan == 'sparse_precise')
            ref = _check_step(m, s, probes, 'sparse', plan)
            if plan == 'sparse_precise':      # TF32 operands: p_s is not comparable step by step (test_sparse_gpu.py)
                assert relerr(m.p_s.asarray(), ref['p_s']) < 5e-3
                assert relerr(m.pi_s.asarray(), ref['pi_s']) < 5e-3


@pytest.mark.gpu
def test_fp32_grade_gene_pass_at_its_nominal_chunk(cuda_lib):
    """A problem large enough that the fp32-grade gene pass keeps its nominal 2048-cell chunk (no halving), probed at the
    chunk seams 2047 / 2048 / 4095 / 4096 and at the gene pairs; float32 and uint16 storage against one oracle step."""
    n, p, K = NOMINAL
    assert tc_chunk(p, n, True, sweep_width(32, True), True) == KC['CHUNK_PRECISE'] < n
    s, probes = edge_case(n, p, K, 'zigap', 'precise', 'mid', 'edges', pers=NOMINAL_PERIODS)
    ref = None
    for storage in ESZ:
        m = _model(s, 'zigap', 'precise', storage)
        assert m.uses_tensor_path and m.precise
        ref = _check_step(m, s, probes, 'zigap', 'precise', ref=ref)


@pytest.mark.gpu
@pytest.mark.parametrize('K', [40, 20])
def test_tf32_gene_pass_at_its_nominal_chunk(cuda_lib, K):
    """The TF32 gene pass at its nominal 16384-cell chunk, two chunks (configs 4 and 5 run it so; every other TF32 problem
    here is small enough that `tc_partition` halves the chunk): probed at the chunk seams 16383 / 16384 and at the gene
    pairs.  K = 40 (KP = 64, config 5's plan) with float32 and uint16 storage against one oracle step, K = 20 (KP = 32)
    with uint16 storage."""
    n, p = NOMINAL_TF32
    assert tc_chunk(p, n, True, sweep_width(32 if K <= 32 else 64, False), False) == KC['CHUNK'] < n
    s, probes = edge_case(n, p, K, 'zigap', 'tf32', 'mid', 'edges', pers=NOMINAL_TF32_PERIODS)
    ref = None
    for storage in (('f32', 'u16') if K == 40 else ('u16',)):
        m = _model(s, 'zigap', 'tf32', storage)
        assert m.uses_tensor_path and not m.precise and m._KP == (32 if K <= 32 else 64)
        ref = _check_step(m, s, probes, 'zigap', 'tf32', ref=ref)
        del m


@pytest.mark.gpu
@pytest.mark.parametrize('model,storage', with_storage(['zigap', 'gap'], str))
def test_underflow_emulation_on_the_probes(cuda_lib, monkeypatch, model, storage):
    """`emulate_underflow=True`, fp32-grade: the probed state with 40 % of the cells and genes 70 below the rest (their
    float32 exp underflows where two meet, see test_underflow_gpu.py) against the oracle with the sequential float32 loop."""
    from oracle import cavi_numpy as cn, zloop

    def literal_z(lU, lV, X, D_hat=None, quirk=True, dtype=np.float32):
        if D_hat is None:
            return zloop.gap_z(lU, lV, X.astype(np.float32))
        return zloop.zigap_z(lU, lV, D_hat, X.astype(np.float32), quirk=quirk)

    for (n, p) in [(2049, 129), (257, 1025)]:
        s, probes = edge_case(n, p, 12, model, 'precise', 'init', 'edges', esz=ESZ[storage])
        rows = {idx[0] for pr in probes for k, idx in pr['checks'] if k == 'a1'}
        genes = {idx[0] for pr in probes for k, idx in pr['checks'] if k == 'b1'}
        rng = np.random.default_rng(n)
        low_i, low_j = rng.random(n) < 0.4, rng.random(p) < 0.4
        low_i[list(rows)] = False; low_j[list(genes)] = False        # the probed cells and genes keep their scale
        s['a1'][low_i] = 0.0143; s['b1'][low_j] = 0.0143
        s = _refresh(s, 'init', model)
        m = _model(s, model, 'precise', storage, emulate_underflow=True)
        assert m.uses_tensor_path and m.precise
        with monkeypatch.context() as mp:
            mp.setattr(cn, 'z_expectations', literal_z)
            ref = oracle_step(s, model)
        # the case does what it says: counts of (low cell, low gene) pairs are assigned to nobody
        assert s['X'][np.ix_(low_i, low_j)].sum() > 0
        # no ELBO check: the oracle's ELBO keeps the exact ratios, the emulating model's those of the float32 exp
        _check_step(m, s, probes, model, 'precise', ref=ref, elbo=False)


@pytest.mark.gpu
@pytest.mark.parametrize('model', ['zigap', 'gap'])
def test_deterministic_mode_on_the_probes(cuda_lib, model):
    """Deterministic mode at the edge shapes: two runs agree bit for bit and with the plain kernels within tolerance.  A
    deterministic run on uint16 storage agrees bit for bit with the float32 one: widening a count is exact, the rest is the
    same code."""
    names = FACTORS + HYPER + (('pi_d',) if model == 'zigap' else ())
    for (n, p, K, pl) in [(257, 2049, 20, 'tf32'), (16385, 63, 40, 'tf32'), (2049, 129, 12, 'precise')]:
        s, _ = edge_case(n, p, K, model, pl, 'mid', 'edges')

        def run(storage='f32', **kw):
            m = _model(s, model, pl, storage, **kw)
            for _ in range(2):
                m.step()
            return {k: getattr(m, k).asarray().copy() for k in names}, m.elbo()

        (a, ea), (b, eb) = run(deterministic=True), run(deterministic=True)
        (c, ec), (plain, ep), (plain16, ep16) = run('u16', deterministic=True), run(), run('u16')
        for k in names:
            assert np.array_equal(a[k], b[k]), (n, p, k)
            assert np.array_equal(a[k], c[k]), (n, p, k, 'u16')
            assert relerr(plain[k], a[k]) < 2 * TOL[pl][0], (n, p, k)
            assert relerr(plain16[k], a[k]) < 2 * TOL[pl][0], (n, p, k, 'u16')
        # sum lgamma(X + 1) is formed with float64 atomics in either order (test_u16_counts_gpu.py)
        assert ea == eb and abs(ec - ea) <= 1e-13 * abs(ea), (ea, ec)
        assert abs(ep - ea) < TOL[pl][3] * abs(ea) and abs(ep16 - ea) < TOL[pl][3] * abs(ea)


@pytest.mark.gpu
def test_host_streamed_slabs_cross_the_row_pass_chunk_seam(cuda_lib):
    """`HostStreamedCAVI` with p > 32768 and two slabs: slabs carry ORI_F_FIXED_CHAIN (n > slab), which keeps the row pass's
    nominal 32768-gene chunk, so the gene edges 32767 / 32768 are a chunk seam.  Against one oracle step (float32 flavour, to
    keep its host memory near 4 GB: X, p_d and the n x p intermediates of 4096 x 33000)."""
    import torch
    from oracle import cavi_numpy as cn
    from oriana_b200.host_step import HostStreamedCAVI
    n, p, K = 4096, 33000, 8
    assert tc_chunk(2048, p, False, sweep_width(32, False), False, fixed_chain=True) == 2 * KC['CHUNK'] < p
    s, probes = edge_case(n, p, K, 'zigap', 'tf32', 'mid', 'edges', steps=1, dtype=np.float32)
    assert s['X'][:, 2 * KC['CHUNK'] - 1].max() == BIG or s['X'][:, 2 * KC['CHUNK']].max() == BIG
    ref = oracle_step(s, 'zigap', dtype=np.float32)
    want0 = cn.elbo(s, guard32=True)
    Xh = torch.as_tensor(s['X'].astype(np.float32)).pin_memory()
    h = HostStreamedCAVI(Xh, K, s, dropout=True, slab_rows=2048)
    assert h._tensor and h.slab == 2048
    e0 = h.step()
    hs = h.state_dict()
    assert abs(e0 - want0) < tol_of('tf32', 'elbo0') * elbo_scale(s, want0), (e0, want0)
    for k in FACTORS:
        assert relerr(hs[k], ref[k]) < 3e-3, k
    for k in HYPER:
        assert relerr(hs[k], ref[k]) < 5e-4, k
    for pr in probes:
        for k, idx in pr['checks']:
            if k in FACTORS:
                assert probe_error(hs, ref, k, idx) < 3e-3, (pr['name'], k)


# --------------------------------------------------------------------------- GPU: the deviance pass at tensor shapes
def _ll_int(X, lam, pi):
    """sparse_numpy.loglikelihood_X(int_quirk=True) as the exact int64 sum (wrapping like the reference's buffer)."""
    Xf = X.astype(np.float64)
    P = np.broadcast_to(np.asarray(pi, dtype=np.float64)[None, :], Xf.shape)
    z = Xf == 0
    ret = np.empty(Xf.shape, dtype=np.int64)
    with np.errstate(divide='ignore', invalid='ignore', over='ignore'):
        ret[z] = np.log(P[z] * np.exp(-lam[z]) + (1. - P[z]))
        ret[~z] = np.log(P[~z]) - lam[~z] + Xf[~z] * np.log(lam[~z])
    return int(ret.sum(dtype=np.int64))


@pytest.mark.gpu
@pytest.mark.parametrize('precise,storage', with_storage([True, False], str))
@pytest.mark.parametrize('masked', [False, True])
def test_deviance_pass_at_tensor_shapes_matches_the_oracle(cuda_lib, masked, precise, storage):
    """The tensor deviance pass (DEVI) against the float64 oracle on edge-probed SparseZIGaP states: counts of 5000 on the
    edges (one truncated term is a visible share of the sum), observed counts under a rate that underflows float32 in the
    last ragged group (the float64 redo) and, `masked`, genes with p_s = 0 at group edges (an exactly zero rate: INT64_MIN
    terms, compared by their parity bit).  uint16 storage: one edge count is 65535, a count with the top bit set through
    the widening and the log x of large counts."""
    from oracle import sparse_numpy as sn
    for (n, p, K) in [(2049, 33, 20), (257, 2049, 8), (129, 65, 12), (16385, 17, 4)]:
        rp, gp = periods(n, p, K, 'tf32', esz=ESZ[storage])
        s, _ = edge_case(n, p, K, 'sparse', 'tf32', 'mid', 'edges', pers=(rp, gp + [devi_chunk(n, p)]),   # + its own chunks
                         esz=ESZ[storage])
        if storage == 'u16':
            i, j = np.argwhere(s['X'] == BIG)[-1]
            s['X'][i, j] = 65535
        g = KC['GROUP']
        last = [j for j in (p - 1, p - 2) if j >= (p - 1) // g * g]
        tiny = [i for i in (n // 2, n // 2 + 1) if i < n]
        s['a1'][tiny] = 1e-22; s['b1'][last] = 1e-22         # U_hat V_hat ~ 1e-44 there: 0 in float32, not in float64
        s['X'][np.ix_(tiny, last)] = 3
        if masked:
            mg = [j for j in (0, g - 1, g, p - 1) if j < p and j not in last] or [0]
            s['p_s'][mg] = 0.
            s['X'][:, mg] = np.maximum(s['X'][:, mg], 1)[:, :]
            s['X'][1::2, mg] = 0
        s = _refresh(s, 'mid', 'sparse')
        assert storage == 'f32' or s['X'].max() == 65535
        m = _model(s, 'sparse', 'sparse_precise' if precise else 'sparse_tf32', storage, tensor=True, precise=precise)
        assert m.uses_tensor_path and m.precise == precise
        li = [int(v) for v in m._loglikelihood_sums(want_f64=False)[0]]
        lam = sn.model_rate(s)
        X = s['X']
        assert (lam[np.ix_(tiny, last)] > 0).all() and (lam[np.ix_(tiny, last)].astype(np.float32) == 0).all()
        pi = s['pi_d']
        want = [_ll_int(X, lam, pi), _ll_int(X, X.astype(np.float64), pi),
                _ll_int(X, np.broadcast_to(X.mean(axis=0)[None, :], X.shape).copy(), pi)]
        top = lambda v: (v >> 63) & 1
        rest = lambda v: v & ((1 << 63) - 1)
        if masked:
            assert top(li[0] & ((1 << 64) - 1)) == top(want[0] & ((1 << 64) - 1)), (n, p)
            assert abs(rest(li[0]) - rest(want[0])) <= 1e-6 * abs(want[1]) + 2, (n, p, li[0], want[0])
        else:
            assert abs(li[0] - want[0]) <= 1e-6 * abs(want[0]) + 2, (n, p, li[0], want[0])
        for k in (1, 2):
            assert abs(li[k] - want[k]) <= 1e-6 * abs(want[k]) + 2, (n, p, k, li[k], want[k])
        for quirk in (True, False):
            # masked, int_quirk=True: sums that hold INT64_MIN terms, wrapped like the reference's int64 buffer (the
            # parity bit and the rest agree above, so the metrics formed from them agree as well)
            for name in ('reconstruction_deviance', 'explained_deviance'):
                w = getattr(sn, name)(s, int_quirk=quirk)
                gv = getattr(m, name)(int_quirk=quirk)
                if not np.isfinite(w):
                    assert gv == w or (np.isnan(w) and np.isnan(gv)), (name, quirk, gv, w)
                else:
                    assert abs(gv - w) <= 1e-5 * abs(w), (n, p, name, quirk, gv, w)


# --------------------------------------------------------------------------- GPU: the operator seam's staging ring
def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _seam_inputs(n, p, K, seed):
    rng = np.random.default_rng(seed)
    lU = rng.normal(-0.5, 1.0, (n, K)).astype(np.float32)
    lV = rng.normal(-0.5, 1.0, (p, K)).astype(np.float32)
    X = (rng.poisson(3.0, (n, p)) * (rng.random((n, p)) < 0.6)).astype(np.float32)
    X[0, 0] = X[-1, -1] = BIG
    D = np.where(X != 0, 1.0, rng.random((n, p))).astype(np.float32)
    return lU, lV, X, D


def _pinned(a):
    import torch
    t = torch.empty(a.shape, dtype=torch.float32).pin_memory()
    out = t.numpy()
    out[...] = a
    return out, t


def _z_call(lib, ctx, lU, lV, D, X, gap=False):
    from oriana_b200 import _lib
    n, K = lU.shape; p = lV.shape[0]
    Zi = np.full((n, K), np.nan, np.float32); Zj = np.full((p, K), np.nan, np.float32)
    if gap:
        if ctx is None:
            _lib.check(lib.ori_gap_compute_Z_q_expectations_host(_ptr(Zi), _ptr(Zj), _ptr(lU), _ptr(lV), _ptr(X), n, p, K))
        else:
            _lib.check(lib.ori_gap_compute_Z_q_expectations_ctx(ctx, _ptr(Zi), _ptr(Zj), _ptr(lU), _ptr(lV), _ptr(X), n, p, K))
        return Zi, Zj
    Z3 = np.full((p, K), np.nan, np.float32)
    if ctx is None:
        _lib.check(lib.ori_zigap_compute_Z_q_expectations_host(_ptr(Zi), _ptr(Zj), _ptr(Z3), _ptr(lU), _ptr(lV), _ptr(D),
                                                               _ptr(X), n, p, K, 0))
    else:
        _lib.check(lib.ori_zigap_compute_Z_q_expectations_ctx(ctx, _ptr(Zi), _ptr(Zj), _ptr(Z3), _ptr(lU), _ptr(lV), _ptr(D),
                                                              _ptr(X), n, p, K, 0))
    return Zi, Zj, Z3


def _against_zloop(got, lU, lV, D, X, tol):
    from oracle import zloop
    rZi, rZj, rZ3 = zloop.zigap_z(lU, lV, D, X, quirk=False, third=True)
    Zi, Zj, Z3 = got
    assert relerr(Zi, rZi) < tol and relerr(Zj, rZj) < tol, (relerr(Zi, rZi), relerr(Zj, rZj))
    assert np.max(np.abs(Z3 - rZ3)) < tol * np.max(np.abs(rZ3))          # signed terms cancel (zigap.py:95)


@pytest.mark.gpu
def test_staging_ring_wraps_over_pageable_slabs(cuda_lib):
    """Pageable inputs of 41 MB per slab (4096 x 2500 floats) go through the 32 MB pinned staging chunks, more than four per
    call, so the ring wraps, on both streams; the same call on pinned inputs takes the direct route.  Both against the
    sequential loop, and with each other to 1e-5 (only the order of the float atomics differs)."""
    from oracle import zloop
    from oriana_b200 import _lib
    n, p, K = 9000, 2500, 12
    lU, lV, X, D = _seam_inputs(n, p, K, 3)
    assert 4096 * p * 4 > 32 << 20
    ctx = ctypes.c_void_p()
    _lib.check(cuda_lib.ori_ctx_create(ctypes.byref(ctx), 4096))
    try:
        pageable = _z_call(cuda_lib, ctx, lU, lV, D, X)
        keep = [_pinned(a) for a in (lU, lV, D, X)]
        pinned = _z_call(cuda_lib, ctx, *[k[0] for k in keep])
        gp = _z_call(cuda_lib, ctx, lU, lV, D, X, gap=True)
    finally:
        _lib.check(cuda_lib.ori_ctx_destroy(ctx))
    _against_zloop(pageable, lU, lV, D, X, 1e-3)
    _against_zloop(pinned, lU, lV, D, X, 1e-3)
    for a, b in zip(pageable[:2], pinned[:2]):
        assert relerr(a, b) < 1e-5
    assert np.max(np.abs(pageable[2] - pinned[2])) < 1e-5 * np.max(np.abs(pinned[2]))
    rZi, rZj = zloop.gap_z(lU, lV, X)
    assert relerr(gp[0], rZi) < 1e-3 and relerr(gp[1], rZj) < 1e-3


@pytest.mark.gpu
def test_config2_call_through_the_default_context(cuda_lib):
    """The call bench.py times at config 2 (10000 x 2000, K = 10, the process-wide context), checked for what it returns."""
    n, p, K = 10000, 2000, 10
    lU, lV, X, D = _seam_inputs(n, p, K, 4)
    _against_zloop(_z_call(cuda_lib, None, lU, lV, D, X), lU, lV, D, X, 1e-3)


@pytest.mark.gpu
def test_row_longer_than_one_staging_chunk(cuda_lib):
    """A row of 8.5e6 genes (34 MB) does not fit one 32 MB staging chunk: the rows are sent in pieces.  Device memory: about
    9 GB of workspace for this shape."""
    n, p, K = 3, 8_500_000, 4
    assert p * 4 > 32 << 20
    lU, lV, X, D = _seam_inputs(n, p, K, 5)
    Zi, Zj, Z3 = _z_call(cuda_lib, None, lU, lV, D, X)
    # float64 reference: the sequential float32 loop itself drifts by ~1e-3 over 8.5e6 terms per row
    lU64, lV64 = lU.astype(np.float64), lV.astype(np.float64)
    eU, eV = np.exp(lU64), np.exp(lV64)
    RD = X * D / (eU @ eV.T)
    RtU = RD.T @ eU
    assert relerr(Zi, (RD @ eV) * eU) < 1e-3 and relerr(Zj, RtU * eV) < 1e-3
    rZ3 = (RD.T @ (eU * lU64) + lV64 * RtU) * eV            # zigap.py:95: sum_i D R e (lU + lV)
    assert np.max(np.abs(Z3 - rZ3)) < 1e-3 * np.max(np.abs(rZ3))
