"""Kernel launches and outputs of one call of each operator-seam variant, for comparing two builds of the library.

Variants: GaP; ZIGaP with quirk on / off, with / without the third output (quirk on without it is the call `bench.py`
times as `operator_seam`); the sparse operator.  Shapes: one on the CUDA-core kernels and tensor-sized slabs at K = 10
(KP = 32 plan) and K = 40 (KP = 64 plan; the sparse operator runs the CUDA-core kernels there).  Each variant gets its
own context and one warm-up call; the `ori_kernel_launches()` delta of the next call and its outputs are recorded.

    ORIANA_B200_LIB=... python scripts/gpu_operator_launches.py --out parent.npz
    python scripts/gpu_operator_launches.py --compare parent.npz new.npz
"""
import argparse, ctypes, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

SHAPES = (('simt 600 x 700 K=12', (600, 700, 12, 0)), ('tensor 2900 x 1500 K=10', (2900, 1500, 10, 1408)),
          ('tensor 2900 x 1500 K=40', (2900, 1500, 40, 1408)))
VARIANTS = ('gap', 'zigap quirk=1', 'zigap quirk=1 third', 'zigap quirk=0', 'zigap quirk=0 third', 'sparse')


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _arrays(n, p, K, seed):
    rng = np.random.default_rng(seed)
    X = (rng.poisson(3.0, (n, p)) * (rng.random((n, p)) < 0.6)).astype(np.float32)
    return dict(lU=rng.normal(-0.5, 1.0, (n, K)).astype(np.float32), lV=rng.normal(-0.5, 1.0, (p, K)).astype(np.float32),
                X=X, D=np.where(X != 0, np.float32(1), rng.random((n, p), dtype=np.float32)).astype(np.float32),
                St=(rng.random((p, K)) >= 0.3).astype(np.float32), Sh=rng.uniform(0.02, 0.98, (p, K)).astype(np.float32))


def _call(lib, ctx, variant, a, outs, n, p, K):
    Zi, Zj, Z3 = outs
    if variant == 'gap':
        return lib.ori_gap_compute_Z_q_expectations_ctx(ctx, _ptr(Zi), _ptr(Zj), _ptr(a['lU']), _ptr(a['lV']), _ptr(a['X']),
                                                        n, p, K)
    if variant == 'sparse':
        return lib.ori_sparse_zigap_compute_Z_q_expectations_ctx(ctx, _ptr(Zi), _ptr(Zj), _ptr(Z3), _ptr(a['lU']),
                                                                 _ptr(a['lV']), _ptr(a['St']), _ptr(a['Sh']), _ptr(a['D']),
                                                                 _ptr(a['X']), n, p, K)
    return lib.ori_zigap_compute_Z_q_expectations_ctx(ctx, _ptr(Zi), _ptr(Zj), _ptr(Z3) if 'third' in variant else None,
                                                      _ptr(a['lU']), _ptr(a['lV']), _ptr(a['D']), _ptr(a['X']), n, p, K,
                                                      int('quirk=1' in variant))


def record(out):
    from oriana_b200 import _lib
    lib = _lib.load()
    saved, launches = {}, {}
    for label, (n, p, K, slab) in SHAPES:
        a = _arrays(n, p, K, 0)
        for v in VARIANTS:
            outs = (np.full((n, K), np.nan, np.float32), np.full((p, K), np.nan, np.float32),
                    np.full((p, K), np.nan, np.float32))
            ctx = ctypes.c_void_p()
            _lib.check(lib.ori_ctx_create(ctypes.byref(ctx), slab))
            try:
                _lib.check(_call(lib, ctx, v, a, outs, n, p, K))
                l0 = lib.ori_kernel_launches()
                _lib.check(_call(lib, ctx, v, a, outs, n, p, K))
                launches['%s | %s' % (label, v)] = int(lib.ori_kernel_launches() - l0)
            finally:
                _lib.check(lib.ori_ctx_destroy(ctx))
            for name, o in zip(('Zi', 'Zj', 'Z3'), outs):
                if not np.isnan(o).all():
                    saved['%s | %s | %s' % (label, v, name)] = o
    np.savez(out, launches=json.dumps(launches), lib=_lib.LIB_PATH, **saved)
    print(json.dumps(launches, indent=1))


def compare(pa, pb):
    a, b = np.load(pa), np.load(pb)
    la, lb = json.loads(str(a['launches'])), json.loads(str(b['launches']))
    print('| shape | variant | launches %s | launches %s | max difference (Zi, Zj relative; Z3 / max abs) |' % (
        os.path.basename(pa), os.path.basename(pb)))
    print('|---|---|---|---|---|')
    worst = 0.0
    for key in la:
        diffs = []
        for name in ('Zi', 'Zj', 'Z3'):
            k = '%s | %s' % (key, name)
            if k not in a.files:
                continue
            x, y = a[k].astype(np.float64), b[k].astype(np.float64)
            if name == 'Z3':
                d = float(np.max(np.abs(x - y)) / max(np.max(np.abs(y)), 1e-30))
            else:
                d = float(np.max(np.abs(x - y) / (np.abs(y) + 1e-6 * np.max(np.abs(y)) + 1e-300)))
            worst = max(worst, d)
            diffs.append('%s %.1e' % (name, d))
        shape, variant = key.split(' | ')
        print('| %s | %s | %d | %d | %s |' % (shape, variant, la[key], lb[key], ', '.join(diffs)))
    print('largest difference %.2e' % worst)


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--out')
    ap.add_argument('--compare', nargs=2)
    args = ap.parse_args()
    if args.compare:
        compare(*args.compare)
    else:
        record(args.out)
