"""uint16 resident counts (ORI_F_X_U16) against float32 on one GPU -> profiles/r3_u16_counts.json (or argv[1]).

Config 4 (1M x 20k, K = 32), ZIGaP and GaP: the same synthetic counts held once as float32 and once as uint16 (narrowed in
slabs, every slab checked to be integral and <= 65535); both models from the same initial state, 5 warm-up steps each,
then 20 steps timed with CUDA events around each pass, the two models stepped alternately; ms per step from events
around whole steps; the ELBO after 25 steps of each.
Config 4 fits the device as float32, so the models would store uint16 counts as float32 (oriana_b200.problem.counts_storage);
the uint16 model here is given uint16 storage explicitly.  Config 5 (2M x 30k, K = 64) on ONE GPU (240 GB as float32 would
not fit) goes through the models' own choice, which must be uint16: 10 steps, ms per step, peak memory, ELBO monotone.  `quick` as an argument: a small rehearsal of the same code."""
import gc, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
from oriana.models import GaP, ZIGaP
from oriana.singlecell import CountMatrix
from oriana_b200 import _lib, problem
from oriana_b200.problem import row_pitch
from oriana_b200.singlecell.synth import synth_counts_device

QUICK = 'quick' in sys.argv
OUT = next((a for a in sys.argv[1:] if a.endswith('.json')), os.path.join(ROOT, 'profiles', 'r3_u16_counts.json'))
C4 = (20_000, 2_000, 32) if QUICK else (1_000_000, 20_000, 32)
C5 = (40_000, 3_000, 64) if QUICK else (2_000_000, 30_000, 64)


def narrow_u16(n, p, K, seed, X32=None, chunk=16384):
    """uint16 [n, p] view of a [n, row_pitch(p, 2)] device buffer holding the synthetic counts of (seed), built slab by slab
    (from X32 when given, else synthesised per slab: the generator is keyed by the global row)."""
    out = torch.zeros((n, row_pitch(p, 2)), dtype=torch.int16, device='cuda')
    for r in range(0, n, chunk):
        rows = min(chunk, n - r)
        blk = X32[r:r + rows, :p] if X32 is not None else synth_counts_device(rows, p, K, seed=seed, row0=r)[:, :p]
        assert float(blk.max()) <= 65535 and float(blk.min()) >= 0 and bool((blk == blk.round()).all())
        out[r:r + rows, :p] = blk.to(torch.int32).to(torch.int16)        # same bits as uint16
    return out.view(torch.uint16)[:, :p]


def timed_steps(m, k):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(k):
        m.step()
    ev[1].record()
    return ev


def config4(cls, X32, X16, K):
    n, p = X32.shape
    models = {}
    rule = problem.counts_storage
    problem.counts_storage = lambda u16, *args: torch.uint16 if u16 else torch.float32
    try:
        for name, X in (('float32', X32), ('uint16', X16)):
            np.random.seed(0)
            models[name] = cls(CountMatrix(X), k=K, use_factors=False, trace_cap=64)
            assert models[name].uses_tensor_path
    finally:
        problem.counts_storage = rule
    assert models['uint16'].counts_dtype == torch.uint16 and models['uint16']._X.data_ptr() == X16.data_ptr()
    for m in models.values():
        for _ in range(5):
            m.step()
        m.enable_kernel_timing()
    step_ev = {k: [] for k in models}
    for _ in range(20):                   # alternate the two models step by step
        for k, m in models.items():
            step_ev[k].append(timed_steps(m, 1))
    torch.cuda.synchronize()
    res = {}
    for k, m in models.items():
        kt = m.kernel_times_ms()
        tr = m.elbo_trace
        res[k] = dict(pass_rows_ms=kt['pass_rows'], pass_genes_ms=kt['pass_genes'], timed_steps=kt['steps'],
                      ms_per_step=float(np.mean([e[0].elapsed_time(e[1]) for e in step_ev[k]])),
                      elbo_after_25=float(tr[25]), x_bytes=int(m._X.untyped_storage().nbytes()))
    f, u = res['float32'], res['uint16']
    res['uint16_over_float32'] = dict(pass_rows=u['pass_rows_ms'] / f['pass_rows_ms'],
                                      pass_genes=u['pass_genes_ms'] / f['pass_genes_ms'],
                                      step=u['ms_per_step'] / f['ms_per_step'])
    res['elbo_rel_diff'] = abs(u['elbo_after_25'] - f['elbo_after_25']) / abs(f['elbo_after_25'])
    print(cls.__name__, json.dumps(res), flush=True)
    del models, m
    gc.collect()                          # the models hold reference cycles (parameter views): free their HBM now
    torch.cuda.empty_cache()
    return res


def main():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                       text=True).stdout.strip().splitlines()
    out = dict(gpu=q[0] if q else torch.cuda.get_device_name(), quick=QUICK)
    n, p, K = C4
    X32 = synth_counts_device(n, p, K, seed=1)[:, :p]
    X16 = narrow_u16(n, p, K, 1, X32=X32)
    out['config4'] = dict(shape=[n, p, K], ZIGaP=config4(ZIGaP, X32, X16, K), GaP=config4(GaP, X32, X16, K))
    del X32, X16
    gc.collect()
    torch.cuda.empty_cache()

    n, p, K = C5
    torch.cuda.reset_peak_memory_stats()
    X16 = narrow_u16(n, p, K, 5)
    np.random.seed(0)
    m = ZIGaP(CountMatrix(X16), k=K, use_factors=False, trace_cap=32)
    assert m.counts_dtype == torch.uint16 and m.uses_tensor_path
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(11)]
    ev[0].record()
    for i in range(10):
        m.step()
        ev[i + 1].record()
    torch.cuda.synchronize()
    per = [ev[i].elapsed_time(ev[i + 1]) for i in range(10)]
    tr = [float(v) for v in m.elbo_trace]
    out['config5_one_gpu_uint16'] = dict(
        shape=[n, p, K], ms_per_step_all=per, ms_per_step_after_first=float(np.mean(per[1:])),
        peak_memory_gb=torch.cuda.max_memory_allocated() / 1e9, x_gb=n * row_pitch(p, 2) * 2 / 1e9,
        float32_x_gb=n * row_pitch(p) * 4 / 1e9, device_memory_gb=torch.cuda.get_device_properties(0).total_memory / 1e9,
        elbo_trace=tr, elbo_monotone=bool(all(b >= a - 1e-7 * abs(a) for a, b in zip(tr, tr[1:]))))
    print('config5', json.dumps(out['config5_one_gpu_uint16']), flush=True)
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, 'w') as f:
        json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
