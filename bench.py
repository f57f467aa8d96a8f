#!/usr/bin/env python
"""bench.py -- CAVI throughput of the B200 path on BASELINE.json's headline configuration.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c4] [--impl reference]

A "step" is one full CAVI iteration (`model.step()`, reference base.py:54-56: E-step + M-step, ELBO terms
included) over the synthetic zero-inflated negative-binomial count matrix of the configuration:
    c1 100 x 500 K=2 | c2 10k x 2k K=10 | c3 100k x 20k K=20 | c4 1M x 20k K=32 (default, the metric's config)
The matrix is generated in HBM (it is far larger than L2, so no flush is needed between steps) and is
sharded by cells over the N ranks (strong scaling: the total problem is fixed).  `value` is whole-job
matrix entries per second (= cells * genes * iterations / s) with everything resident in HBM; `e2e` is the
same metric through the host-buffer entry (`HostStreamedCAVI.step()`): the count matrix and the row
parameters are streamed from pinned host memory and the results copied back inside the timed region.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {
    'c1': (100, 500, 2), 'c2': (10_000, 2_000, 10), 'c3': (100_000, 20_000, 20),
    'c4': (1_000_000, 20_000, 32), 'c5': (2_000_000, 30_000, 64),
}
ZERO_LEVEL = {'c5': 0.12}          # keep-probability mean: ~90 % zeros for BASELINE configs[4], 0.5 elsewhere (SURVEY.md 8d)
# torch.matmul fp32 with TF32 tensor cores, 8192^3, sustained for 4 s on this pool's B200 (scripts/gpu_peaks.py, measured in
# round 2 the way MEASURED_PEAKS.json measured bf16: 700.0 TF burst, 614.7 TF sustained; profiles/r2_peaks.json)
TF32_PEAK_TFLOPS = 614.7
METRIC = 'cavi_matrix_entries_per_sec'
UNIT = 'entries/s'


def workload_name(cfg, n, p, K):
    return 'synthetic ZINB counts %d cells x %d genes, K=%d, ZIGaP CAVI (dropout on), config %s' % (n, p, K, cfg)


def load_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.samples, self.reasons, self.max_mhz, self._stop_evt = [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {getattr(nv, k): k for k in dir(nv) if k.startswith('nvmlClocksThrottleReason') or k.startswith('nvmlClocksEventReason')}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if isinstance(bit, int) and bit and (r & bit) and 'None' not in name and 'All' not in name:
                        self.reasons.add(name.replace('nvmlClocksThrottleReason', '').replace('nvmlClocksEventReason', ''))
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        rs = sorted({r for r in self.reasons if r not in ('GpuIdle', 'ApplicationsClocksSetting')})
        return dict(sm_mhz=(s[len(s) // 2] if s else None), sm_max_mhz=self.max_mhz, reasons=rs, samples=len(s))


def cpu_port_run(n, p, K, steps, warmup, seed=0, budget_rows=2048):
    """The oracle port of the reference's step() (oracle/cavi_numpy.py: numpy + multithreaded BLAS, float32
    ratio form) on a bounded row slab of the same workload: the "fair multi-core numpy" number of BASELINE.md
    section 3.  Returns (entries/s, cores, sample text, s/step)."""
    import numpy as np
    from oracle import cavi_numpy as cn
    rows = int(min(n, budget_rows))
    X = cn.synth_counts(rows, p, K, seed=seed)
    s = cn.init_state(X, K, np.random.default_rng(seed), 'zigap')
    for _ in range(warmup):
        cn.step(s, quirk=False)
    t0 = time.perf_counter()
    for _ in range(steps):
        cn.step(s, quirk=False)
    dt = (time.perf_counter() - t0) / max(1, steps)
    return rows * p / dt, os.cpu_count(), ('%d-row slab of the workload (%d x %d, K=%d), %d full CAVI steps of the '
                                          'numpy/BLAS oracle port, %.2f s/step' % (rows, rows, p, K, steps, dt)), dt


def cpu_reference_run(n, p, K, steps, warmup, seed=0, budget_s=150.0):
    """The UNMODIFIED reference (`oriana.models.ZIGaP.step()`, zigap.py:97-158: numba triple loop + numpy) installed
    under oracle/_ref by `__graft_entry__.build()`, on a bounded row slab of the same workload, through its own
    public API.  The slab is sized so that warmup + steps fit the time budget (the per-entry cost is flat in the
    number of rows, BASELINE.md section 2).  Returns None when the install did not travel."""
    import warnings
    import numpy as np
    from oracle import refshim, cavi_numpy as cn
    if not refshim.available():
        return None
    ns_per_entry = 25.0 * K                                 # BASELINE.md section 2: 776 ns at K = 32, 271 ns at K = 10
    rows = int(budget_s / max(1, steps + warmup) / (ns_per_entry * 1e-9) / p)
    rows = max(16, min(n, 256, rows))
    X = cn.synth_counts(rows, p, K, seed=seed)
    try:
        refshim.import_reference()
        from oriana.models import ZIGaP
        from oriana.singlecell import CountMatrix
        np.random.seed(1)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            m = ZIGaP(CountMatrix(X), k=K, use_factors=False)
            for _ in range(warmup):
                m.step()
            t0 = time.perf_counter()
            for _ in range(steps):
                m.step()
            dt = (time.perf_counter() - t0) / max(1, steps)
        ok = bool(np.isfinite(m.a1[:]).all() and np.isfinite(m.b1[:]).all())
    finally:
        refshim.release_reference()
    sample = ('%d-row slab of the workload (%d x %d, K=%d), %d steps of the unmodified reference ZIGaP.step() '
              '(oracle/_ref; numba Z-loop on ONE thread by construction = ~80 %% of the step, the two np.dot on %d BLAS '
              'threads), %.2f s/step, state finite: %s' % (rows, rows, p, K, steps, os.cpu_count() or 1, dt, ok))
    return rows * p / dt, 1, sample, dt


def initial_state(n, p, K, r0, r1, seed=4321, block=8192):
    """The `use_factors=False` initialisation of the reference (zigap.py:58-75: a1, b1 ~ Gamma(1), a2 = b2 = 1; prior
    shapes ~ Gamma(2), rates 1, zigap.py:22-27) drawn from counter-based streams keyed by the GLOBAL row block, so rows
    [r0, r1) get the same values under any sharding.  D_hat starts as the indicator (X > 0), zigap.py:77."""
    import numpy as np

    def stream(tag, idx):
        return np.random.Generator(np.random.Philox(key=[seed, tag], counter=[idx, 0, 0, 0]))
    a1 = np.empty((r1 - r0, K))
    for b in range(r0 // block, (r1 + block - 1) // block):
        lo, hi = b * block, min(n, (b + 1) * block)
        blk = stream(1, b).gamma(1., size=(hi - lo, K))
        s0, s1 = max(lo, r0), min(hi, r1)
        a1[s0 - r0:s1 - r0] = blk[s0 - lo:s1 - lo]
    g = stream(2, 0)
    return dict(a1=a1, a2=np.ones((r1 - r0, K)), b1=g.gamma(1., size=(p, K)), b2=np.ones((p, K)),
                alpha1=g.gamma(2., size=K), alpha2=np.ones(K), beta1=g.gamma(2., size=K), beta2=np.ones(K))


def elbo_vs_n1(cfg, warmup, steps, world, elbo_last):
    """Relative difference between this run's final ELBO and the one a single GPU reaches after the same number of
    steps from the same (sharding-invariant) initial state: profiles/elbo_ref.json holds the N = 1 values this repo
    measured, keyed "<config>:<warmup + steps>"; a N = 1 run with no entry reports 0 against itself, others null."""
    path = os.path.join(ROOT, 'profiles', 'elbo_ref.json')
    try:
        ref = json.load(open(path)).get('%s:%d' % (cfg, warmup + steps))
    except Exception:
        ref = None
    if ref is None:
        return 0.0 if world == 1 else None
    return abs(elbo_last - ref) / abs(ref)


def secondary_device_run(cfg, world, rank, dev, steps=5, warmup=3):
    """A short device-resident run of another BASELINE configuration in the same job (no e2e / CPU legs): used for config 5
    (2M x 30k, K = 64, ~90 % zeros), which BASELINE.json defines at 8 GPUs only, so that the driver's 8-GPU run records it."""
    import torch
    import torch.distributed as dist
    from oriana.models import ZIGaP
    from oriana.singlecell import synth_counts_device
    from oriana_b200.sharding import RowSharding
    n, p, K = CONFIGS[cfg]
    r0, r1 = RowSharding.row_block(n, rank, world)
    rows = r1 - r0
    X = synth_counts_device(rows, p, K, seed=1234, row0=r0, zero_level=ZERO_LEVEL.get(cfg, 0.5))
    zeros = float((X[: min(rows, 4096), :p] == 0).float().mean())
    st = initial_state(n, p, K, r0, r1)
    st['X'] = X[:, :p]
    m = ZIGaP(X[:, :p], k=K, use_factors=False, sharded=world > 1, state=st, keep_hyper=False, trace_cap=warmup + steps + 8)
    del st
    for _ in range(warmup):
        m.step()
    m.enable_kernel_timing()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        m.step()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    kt = m.kernel_times_ms()
    trace = m.elbo_trace
    peak, _ = load_peaks()
    alg = 4.0 * rows * p
    flops = 12.0 * K * rows * p          # SURVEY.md 8d: algorithmic flops per entry and iteration with dropout
    out = {'workload': workload_name(cfg, n, p, K), 'n_gpus': world, 'steps': steps, 'warmup': warmup, 'ms_per_step': ms,
           'iters_per_sec': 1e3 / ms, 'value': n * p / (ms * 1e-3), 'unit': UNIT, 'zero_fraction_sample': zeros,
           'KP_plan': 32 if K <= 32 else 64,
           'kernels': [{'kernel': k, 'ms': kt[k], 'hbm_gbs': alg / (kt[k] * 1e-3) / 1e9, 'hbm_frac': alg / (kt[k] * 1e-3) / 1e9 / peak}
                       for k in ('pass_rows', 'pass_genes')],
           'algorithmic_tflops_per_rank': flops / (ms * 1e-3) / 1e12,
           'tf32_peak_tflops': TF32_PEAK_TFLOPS, 'tensor_frac_of_tf32_peak': flops / (ms * 1e-3) / 1e12 / TF32_PEAK_TFLOPS,
           'elbo_monotone': bool((trace[2:] >= trace[1:-1] - 1e-6 * abs(trace[1:-1])).all()), 'elbo_last': float(trace[-1])}
    del m, X
    torch.cuda.empty_cache()
    return out


DUMP_CELLS = 65536


def dump_outputs(path, model, trace, rows, r0):
    """What the timed `model.step()` leaves its caller after the last timed step, as <path>/<name>.npy: the model's
    `state_dict()` and its ELBO trace.  The cell-side factors (a1, a2: cells x K) are a fixed sample of DUMP_CELLS of
    this rank's cells, the same in every run of a configuration (their global indices in cells.npy), so that two builds
    can be compared output for output within 64 MB.  The factors are float32 on the device and written as float32."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    cells = np.arange(rows) if rows <= DUMP_CELLS else np.sort(np.random.default_rng(0).choice(rows, DUMP_CELLS, replace=False))
    out = {'cells': (r0 + cells).astype(np.float64), 'elbo_trace': np.asarray(trace, dtype=np.float64)}
    for k, v in model.state_dict().items():
        if k == 'iterations':
            continue
        v = np.asarray(v)
        out[k] = (v[cells] if k in ('a1', 'a2') else v).astype(np.float32 if k in ('a1', 'a2', 'b1', 'b2') else np.float64)
    total = sum(v.nbytes for v in out.values())
    assert total <= 64 << 20, 'outputs of %d bytes exceed 64 MB' % total
    for k, v in out.items():
        np.save(os.path.join(path, k + '.npy'), v)


def operator_seam_rates(lib):
    """The reference's plug-in point (`ZIGaP.compute_Z_q_expectations`, zigap.py:79-95) through its C-ABI replacement with
    HOST numpy arrays in and out, at config 2 and at a row slab of config 3: entries / s of the whole call (copies in)."""
    import ctypes
    import numpy as np
    out = []
    fp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    for name, (n, p, K) in (('c2 10000 x 2000, K=10', (10_000, 2_000, 10)), ('c3 slab 8192 x 20000, K=20', (8192, 20_000, 20))):
        rng = np.random.default_rng(0)
        lU = rng.normal(-0.5, 1.0, (n, K)).astype(np.float32); lV = rng.normal(-0.5, 1.0, (p, K)).astype(np.float32)
        X = (rng.poisson(3.0, (n, p)) * (rng.random((n, p)) < 0.5)).astype(np.float32)
        D = np.where(X != 0, np.float32(1), rng.random((n, p), dtype=np.float32)).astype(np.float32)
        Zi = np.empty((n, K), np.float32); Zj = np.empty((p, K), np.float32)
        call = lambda: lib.ori_zigap_compute_Z_q_expectations_host(fp(Zi), fp(Zj), None, fp(lU), fp(lV), fp(D), fp(X), n, p, K, 1)
        assert call() == 0
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            assert call() == 0
        dt = (time.perf_counter() - t0) / reps
        out.append({'shape': name, 'ms_per_call': dt * 1e3, 'entries_per_s': n * p / dt,
                    'host_bytes_in_per_call': int(X.nbytes + D.nbytes + lU.nbytes + lV.nbytes)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default=os.environ.get('ORIANA_BENCH_CONFIG', 'c4'), choices=sorted(CONFIGS))
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the secondary measurements (operator seam, config 5 at 8 GPUs)')
    ap.add_argument('--e2e-steps', type=int, default=0)
    ap.add_argument('--e2e-x', default='auto', choices=['auto', 'sparse', 'u8esc', 'u16', 'f32'],
                    help='how the host holds X for the e2e leg: bitmap + non-zero bytes (sparse), saturating uint8 + escapes '
                         '(u8esc), uint16, float32; auto (default) = sparse when that is the smaller of the two lossless byte forms')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the model state they computed as DIR/<name>.npy (rank 0; a fixed '
                         'sample of the cell-side factors, 64 MB at most)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the device run (--impl ours)')
    n, p, K = CONFIGS[args.config]
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    W = max(args.warmup, 0)

    if args.impl == 'reference':
        if rank != 0:
            return 0
        # torchrun pins OMP_NUM_THREADS=1 for its workers: the CPU arm gets every host core (set before numpy loads)
        for var in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS', 'NUMBA_NUM_THREADS'):
            os.environ[var] = str(os.cpu_count() or 1)
        steps = max(1, args.steps)
        pval, pcores, psample, pdt = cpu_port_run(n, p, K, min(steps, 5), min(W, 1))
        port = {'value': pval, 'unit': UNIT, 'cores': pcores, 'kind': 'port', 'sample': psample}
        ref = cpu_reference_run(n, p, K, steps, W)
        if ref is not None:
            val, cores, sample, dt = ref
            kind = 'reference'
        else:   # no reference install (oracle/_ref missing): the port is what is left
            val, cores, sample, dt = cpu_port_run(n, p, K, steps, W)
            kind = 'port'
        print(json.dumps({
            'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': steps,
            'warmup': W, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
            'dtype': 'f32/f64 (reference: float32 Z loop, float64 parameters)', 'data': 'synthetic',
            'iters_per_sec_full_problem': val / (n * p),
            'config': {'workload': workload_name(args.config, n, p, K), 'n': n, 'p': p, 'K': K},
            'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cores, 'kind': kind, 'sample': sample},
            'fair_multicore_port': port,
            'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}))
        return 0

    import numpy as np
    import torch
    import torch.distributed as dist
    from oriana.models import ZIGaP
    from oriana.singlecell import synth_counts_device
    from oriana_b200.host_step import HostStreamedCAVI
    from oriana_b200.sharding import RowSharding

    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    W = max(W, 3)
    K_steps = max(1, args.steps)
    r0, r1 = RowSharding.row_block(n, rank, world)
    rows = r1 - r0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- synthetic counts, generated in HBM by this rank for its own cells
    X = synth_counts_device(rows, p, K, seed=1234, row0=r0, zero_level=ZERO_LEVEL.get(args.config, 0.5))
    # initial state keyed by the GLOBAL row (like the counts): the same model whatever the number of ranks, so that the
    # ELBO after the timed steps is a sharding check across N = 1/2/4/8 (it differs only by summation order)
    state0 = initial_state(n, p, K, r0, r1)
    state0['X'] = X[:, :p]
    model = ZIGaP(X[:, :p], k=K, use_factors=False, sharded=world > 1, state=state0, keep_hyper=False,
                  trace_cap=W + K_steps + 8)
    del state0
    uses_tc = model.uses_tensor_path
    for _ in range(W):
        model.step()
    model.enable_kernel_timing()
    sampler = ClockSampler(local)
    from oriana_b200 import _lib as _orilib
    launches0 = int(_orilib.load().ori_kernel_launches())
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K_steps):
        model.step()
    e1.record()
    barrier()
    launches = int(_orilib.load().ori_kernel_launches()) - launches0      # counted inside the C ABI library
    clocks = sampler.stop()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    ms_step = ms_total / K_steps
    value = n * p * K_steps / (ms_total * 1e-3)
    kt = model.kernel_times_ms()
    model.enable_kernel_timing(False)
    trace = model.elbo_trace
    elbo_ok = bool(np.isfinite(trace).all() and np.all(np.diff(trace[1:]) >= -1e-6 * np.abs(trace[1:-1])))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, trace, rows, r0)

    # ---- the same steps without the ELBO terms (SURVEY.md 8d: reported beside the contract number, not instead)
    state0 = model.state_dict(); state0['X'] = X[:, :p]
    lean = ZIGaP(X[:, :p], k=K, use_factors=False, sharded=world > 1, state=state0, elbo=False,
                 trace_cap=2 * (W + K_steps) + 16)      # continues the iteration count of the snapshot
    for _ in range(W):
        lean.step()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(K_steps):
        lean.step()
    f1.record()
    barrier()
    ms_step_lean = max_over_ranks(f0.elapsed_time(f1)) / K_steps
    del lean, state0

    # ---- roofline of the dominant kernel (both X-streaming kernels read this rank's X once: 4 B/entry)
    peak, peak_src = load_peaks()
    alg_bytes = 4.0 * rows * p
    kernels = []
    for name in ('pass_rows', 'pass_genes'):
        t = max_over_ranks(kt[name])
        kernels.append({'kernel': name, 'ms': t, 'achieved': alg_bytes / (t * 1e-3) / 1e9})
    dom = max(kernels, key=lambda k: k['ms'])
    # DRAM bytes per launch of the dominant kernel from an `ncu --set full` capture of THIS configuration and world
    # size (profiles/traffic.json, key "<config>:n<world>:<kernel>"); null when no such capture exists
    traffic = None
    prof = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get('%s:n%d:%s' % (args.config, world, dom['kernel']))
        except Exception:
            traffic = None
    roofline = {'bound': 'hbm', 'kernel': dom['kernel'], 'achieved': dom['achieved'], 'peak': peak, 'unit': 'GB/s',
                'frac': dom['achieved'] / peak, 'traffic': traffic, 'peak_source': peak_src,
                'algorithmic_bytes_per_launch': alg_bytes, 'kernels': kernels,
                'step_frac': (8.0 * rows * p / (ms_step * 1e-3) / 1e9) / peak}
    # second roofline of the same kernels (profiles/r2_xu_mio_bound.md): a MUFU costs 8 cycles per warp instruction and SM
    # sub-partition (16 lanes / clk / SM, measured); the row pass issues 2 per entry (ex2 + rcp), the gene pass 3 (+ lg2 of
    # the ELBO).  Floor = entries x MUFU / (SMs x 16 x the median SM clock sampled during the timed region).
    if uses_tc and clocks.get('sm_mhz'):
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        per = {'pass_rows': 2, 'pass_genes': 3}
        xu = []
        for k in kernels:
            floor_ms = rows * p * per[k['kernel']] / (sms * 16.0 * clocks['sm_mhz'] * 1e6) * 1e3
            xu.append({'kernel': k['kernel'], 'mufu_per_entry': per[k['kernel']], 'floor_ms': floor_ms, 'frac': floor_ms / k['ms']})
        step_floor = sum(x['floor_ms'] for x in xu)
        roofline['xu'] = {'bound': 'special-function (MUFU) issue, not a contract field: explains the HBM fraction', 'sm_mhz': clocks['sm_mhz'],
                          'kernels': xu, 'step_floor_ms': step_floor, 'step_frac': step_floor / ms_step,
                          'hbm_step_floor_ms': 8.0 * rows * p / (peak * 1e9) * 1e3}

    # ---- end to end through host buffers
    e2e = None
    if not args.no_e2e:
        state = model.state_dict()
        del model
        # counts are small integers: by default the host keeps them as saturating uint8 + an escape list for the
        # counts >= 255 (lossless, oriana_b200.host_step.CompactCounts): one byte per entry crosses PCIe per step
        from oriana_b200.host_step import CompactCounts, SparseCounts, bind_host_thread_to_gpu
        # pinned host buffers next to this rank's GPU: allocate them from the cores NVML calls local to it
        all_cores = os.sched_getaffinity(0)
        numa_cores = bind_host_thread_to_gpu(local)
        e2e_x = args.e2e_x
        if e2e_x == 'auto':
            e2e_x = 'sparse' if SparseCounts.smaller_than_bytes(X[:, :p]) else 'u8esc'
        if e2e_x == 'sparse':
            Xh = SparseCounts.from_tensor(X[:, :p])
            xdesc = ('bitmap (1 bit per entry) + %d non-zero bytes (%.3f bytes per entry in all) + %d escapes (counts >= 255)'
                     % (Xh.nz.numel(), Xh.nbytes / float(rows * p), Xh.row.numel()))
        elif e2e_x == 'u8esc':
            Xh = CompactCounts.from_tensor(X[:, :p])
            xdesc = 'uint8 + %d escapes (counts >= 255)' % Xh.row.numel()
        else:
            xdt = torch.uint16 if (e2e_x == 'u16' and float(X.max()) < 65536) else torch.float32
            Xh = torch.empty((rows, p), dtype=xdt, pin_memory=True)
            for r in range(0, rows, 1 << 16):
                Xh[r:r + (1 << 16)].copy_(X[r:r + (1 << 16), :p].to(xdt))
            xdesc = str(xdt).replace('torch.', '')
        del X
        torch.cuda.empty_cache()
        host = HostStreamedCAVI(Xh, K, state, dropout=True, sharded=world > 1)
        n_e2e = args.e2e_steps or max(2, min(K_steps, 4))
        e_first = host.step()                             # warm-up; returns the ELBO of the state it started from
        h0, d0 = host.h2d_bytes, host.d2h_bytes
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            host.step()
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        hb = torch.tensor([host.h2d_bytes - h0, host.d2h_bytes - d0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(hb)
        e2e = {'value': n * p * n_e2e / dt, 'unit': UNIT, 'h2d_bytes_per_step': float(hb[0]) / n_e2e,
               'd2h_bytes_per_step': float(hb[1]) / n_e2e, 'steps': n_e2e, 'ms_per_step': dt / n_e2e * 1e3,
               'host_x_dtype': xdesc, 'host_cores_bound': (None if numa_cores is None else '%d cores: %d-%d' % (len(numa_cores), numa_cores[0], numa_cores[-1])),
               # the host-streamed run continues the device run: its first step reports the ELBO of the device model's
               # last state
               'elbo_first_vs_device': abs(e_first - float(trace[-1])) / abs(float(trace[-1])),
               'api': 'oriana_b200.host_step.HostStreamedCAVI.step (pinned host X, a1, a2, b1, b2 in; results out)'}
        os.sched_setaffinity(0, all_cores)          # the CPU arm below gets every host core again

    # ---- the reference's CPU path beside it (rank 0, N=1 only): the unmodified reference on a bounded slab, and the
    #      multi-core numpy/BLAS port of the same step as the fair comparison
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        for var in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
            os.environ.setdefault(var, str(os.cpu_count() or 1))
        pval, pcores, psample, _ = cpu_port_run(n, p, K, steps=3, warmup=1)
        port = {'value': pval, 'unit': UNIT, 'cores': pcores, 'kind': 'port', 'sample': psample}
        ref = cpu_reference_run(n, p, K, steps=3, warmup=1, budget_s=12.0)
        if ref is not None:
            cpu = {'value': ref[0], 'unit': UNIT, 'cores': ref[1], 'kind': 'reference', 'sample': ref[2], 'port': port}
        else:
            cpu = port

    # ---- secondary measurements in the same job
    extra = {}
    if not args.no_extra:
        try:
            del host, Xh
        except NameError:
            pass
        import gc
        gc.collect(); torch.cuda.empty_cache()
        if world == 1 and rank == 0:
            extra['operator_seam'] = operator_seam_rates(_orilib.load())
        if world == 8 and args.config == 'c4':
            extra['config5'] = secondary_device_run('c5', world, rank, dev)

    if rank == 0:
        out = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K_steps, 'warmup': W,
            'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
            'dtype': 'tf32 operands / f32 accumulate (f32 state, f64 ELBO sums)' if uses_tc else 'f32', 'data': 'synthetic',
            'iters_per_sec': 1e3 / ms_step,
            'without_elbo': {'ms_per_step': ms_step_lean, 'iters_per_sec': 1e3 / ms_step_lean,
                             'value': n * p / (ms_step_lean * 1e-3)},
            'config': {'workload': workload_name(args.config, n, p, K), 'n': n, 'p': p, 'K': K,
                       'arithmetic': 'fp32 state; denominator and U.V^T split-precision on the tensor cores (tf32 hi.hi + bf16 cross '
                                     'terms, ~2^-21); R and D_hat as TF32 operands, fp32 accumulation in TMEM; ELBO partial sums fp64',
                       'cells_per_rank': rows, 'parallelism': 'cells sharded over %d rank(s); 2 sum-allreduces/iter' % world,
                       'l2': 'X per rank is %.1f GB, far larger than the 126 MB L2: no flush between steps' % (alg_bytes / 1e9)},
            'roofline': roofline, 'cpu_baseline': cpu, 'e2e': e2e, 'clocks': clocks,
            'gpu_launches': launches, 'tensor_path': bool(uses_tc), 'elbo_monotone': elbo_ok, 'elbo_last': float(trace[-1]),
            'elbo_vs_n1': elbo_vs_n1(args.config, W, K_steps, world, float(trace[-1])),
            'tensor_frac_of_tf32_peak': (12.0 * K * rows * p / (ms_step * 1e-3) / 1e12) / TF32_PEAK_TFLOPS,
        }
        out.update(extra)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
