"""The sparse model's operator seam (`ori_sparse_zigap_compute_Z_q_expectations_ctx`, sparse_zigap.py:100-116) beside the
ZIGaP operator (`ori_zigap_compute_Z_q_expectations_ctx`, quirk on, no third output: the call `bench.py` times as
`operator_seam`) on the same pageable numpy arrays, calls of the two alternated, at config 2 and a row slab of config 3.
Entries / s of the whole call (host copies in and out included), the slab counts per kernel family, and the reference's
numba sparse kernel on a row slab when the reference is installed under oracle/_ref.

    python scripts/gpu_time_sparse_operator.py [--out profiles/r3_sparse_operator_seam.json] [--reps 5]
"""
import argparse, ctypes, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from oriana_b200 import _lib

CONFIGS = (('c2 10000 x 2000, K=10', (10_000, 2_000, 10)), ('c3 slab 8192 x 20000, K=20', (8192, 20_000, 20)))


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _stats(lib, ctx):
    c = [ctypes.c_uint64(0) for _ in range(4)]
    _lib.check(lib.ori_ctx_stats(ctx, *[ctypes.byref(x) for x in c]))
    return [int(x.value) for x in c]


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = 'unknown'
    return name, limit


def _reference_numba(n, p, K, rows, seed):
    """SparseZIGaP.compute_Z_q_expectations of the unmodified reference on a `rows`-row slab (one thread, by construction)."""
    from oracle import refshim
    if not os.path.isdir(os.path.join(refshim.INSTALLED, 'oriana', 'models')):
        return None
    a = _arrays(rows, p, K, seed)
    try:
        refshim.import_reference()
        from oriana.models import SparseZIGaP
        outs = np.empty((rows, K), np.float32), np.empty((p, K), np.float32), np.empty((p, K), np.float32)
        args = outs + (a['lU'], a['lV'], a['St'], a['Sh'], a['D'], a['X'])
        SparseZIGaP.compute_Z_q_expectations(*args)
        t0 = time.perf_counter()
        SparseZIGaP.compute_Z_q_expectations(*args)
        dt = time.perf_counter() - t0
    finally:
        refshim.release_reference()
    return {'rows': rows, 'ms_per_call': dt * 1e3, 'entries_per_s': rows * p / dt}


def _arrays(n, p, K, seed):
    rng = np.random.default_rng(seed)
    X = (rng.poisson(3.0, (n, p)) * (rng.random((n, p)) < 0.5)).astype(np.float32)
    return dict(lU=rng.normal(-0.5, 1.0, (n, K)).astype(np.float32), lV=rng.normal(-0.5, 1.0, (p, K)).astype(np.float32),
                X=X, D=np.where(X != 0, np.float32(1), rng.random((n, p), dtype=np.float32)).astype(np.float32),
                St=(rng.random((p, K)) >= 0.3).astype(np.float32), Sh=rng.uniform(0.02, 0.98, (p, K)).astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r3_sparse_operator_seam.json'))
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    args = ap.parse_args()
    lib = _lib.load()
    name, limit = _card()
    result = {'gpu': name, 'power_limit': limit, 'reps': args.reps, 'warmup': args.warmup, 'configs': []}
    for label, (n, p, K) in CONFIGS:
        a = _arrays(n, p, K, 0)
        DSZ, DZ, DZl = np.empty((n, K), np.float32), np.empty((p, K), np.float32), np.empty((p, K), np.float32)
        Zi, Zj = np.empty((n, K), np.float32), np.empty((p, K), np.float32)
        ctx = {k: ctypes.c_void_p() for k in ('zigap', 'sparse')}
        for c in ctx.values():
            _lib.check(lib.ori_ctx_create(ctypes.byref(c), 0))
        calls = {
            'zigap': lambda: lib.ori_zigap_compute_Z_q_expectations_ctx(
                ctx['zigap'], _ptr(Zi), _ptr(Zj), None, _ptr(a['lU']), _ptr(a['lV']), _ptr(a['D']), _ptr(a['X']), n, p, K, 1),
            'sparse': lambda: lib.ori_sparse_zigap_compute_Z_q_expectations_ctx(
                ctx['sparse'], _ptr(DSZ), _ptr(DZ), _ptr(DZl), _ptr(a['lU']), _ptr(a['lV']), _ptr(a['St']), _ptr(a['Sh']),
                _ptr(a['D']), _ptr(a['X']), n, p, K)}
        try:
            for _ in range(args.warmup):
                for f in calls.values():
                    _lib.check(f())
            before = {k: _stats(lib, c) for k, c in ctx.items()}
            times = {k: [] for k in calls}
            for _ in range(args.reps):              # alternated: both operators see the same host and card state
                for k, f in calls.items():
                    t0 = time.perf_counter()
                    _lib.check(f())
                    times[k].append(time.perf_counter() - t0)
            after = {k: _stats(lib, c) for k, c in ctx.items()}
        finally:
            for c in ctx.values():
                _lib.check(lib.ori_ctx_destroy(c))
        row = {'shape': label, 'host_bytes_in_per_call': int(a['X'].nbytes + a['D'].nbytes)}
        for k in calls:
            med = float(np.median(times[k]))
            d = [x - y for x, y in zip(after[k], before[k])]
            row[k] = {'ms_per_call_median': med * 1e3, 'ms_per_call_min': min(times[k]) * 1e3,
                      'entries_per_s': n * p / med, 'tensor_slabs_per_call': d[2] / args.reps,
                      'simt_slabs_per_call': d[3] / args.reps, 'allocations_in_timed_calls': d[1]}
        row['sparse_over_zigap_time'] = row['sparse']['ms_per_call_median'] / row['zigap']['ms_per_call_median']
        ref_rows = 64 if p <= 4000 else 16
        row['reference_numba_sparse_kernel'] = _reference_numba(n, p, K, ref_rows, 1)
        result['configs'].append(row)
        print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(result, f, indent=1)
    print('written', args.out, '(%s, power limit %s)' % (name, limit))


if __name__ == '__main__':
    main()
