"""CSR ingest and the CsrCounts host form on one GPU -> profiles/r3_csr_ingest.json (or the .json path given).

100k x 20k cells x genes at 50 %, 10 % and 3 % non-zeros (counts 1..7, float32 like a scanpy / AnnData matrix):
  * ingest: `CountMatrix(X).to_device()` of the dense float32 ndarray against the CSR of the same counts (float32 data,
    int32 indices), wall time to a device synchronise, best of 3 after one warm-up, and the host bytes of each input;
    the two device matrices are compared bit for bit.
  * host-streamed step: `HostStreamedCAVI`, ZIGaP K = 20, from `SparseCounts` against `CsrCounts` of the same counts and
    the same initial state; 2 warm-up steps, then 5 steps timed with a host clock around each (each ends in a device
    synchronise); h2d_bytes per step; the largest relative difference of the parameters after the 7 steps.
`quick` as an argument: a small rehearsal of the same code."""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, scipy.sparse as sp, torch
from oriana.singlecell import CountMatrix
from oriana_b200.host_step import HostStreamedCAVI

QUICK = 'quick' in sys.argv
OUT = next((a for a in sys.argv[1:] if a.endswith('.json')), os.path.join(ROOT, 'profiles', 'r3_csr_ingest.json'))
N, P, K = (4_000, 1_500, 20) if QUICK else (100_000, 20_000, 20)
DENSITIES = (0.5, 0.1, 0.03)


def counts(density, seed, chunk=5_000):
    """(dense float32 ndarray, CSR) of the same counts, built in row chunks."""
    rng = np.random.default_rng(seed)
    X = np.zeros((N, P), dtype=np.float32)
    for r in range(0, N, chunk):
        rows = min(chunk, N - r)
        keep = rng.random((rows, P), dtype=np.float32) < density
        X[r:r + rows][keep] = rng.integers(1, 8, size=int(keep.sum())).astype(np.float32)
    csr = sp.vstack([sp.csr_matrix(X[r:r + chunk]) for r in range(0, N, chunk)], format='csr')
    return X, csr


def host_bytes(a):
    return int(a.nbytes) if isinstance(a, np.ndarray) else int(a.data.nbytes + a.indices.nbytes + a.indptr.nbytes)


def ingest(src):
    """Best-of-3 seconds of CountMatrix(src).to_device() (one warm-up), and the device matrix of the last run."""
    out, best = None, float('inf')
    for i in range(4):
        out = None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = CountMatrix(src).to_device('cuda')
        torch.cuda.synchronize()
        if i:
            best = min(best, time.perf_counter() - t0)
    return best, out


def init_state(seed):
    rng = np.random.default_rng(seed)
    return dict(a1=rng.gamma(1., size=(N, K)), a2=np.ones((N, K)), b1=rng.gamma(1., size=(P, K)), b2=np.ones((P, K)),
                alpha1=rng.gamma(2., size=K), alpha2=np.ones(K), beta1=rng.gamma(2., size=K), beta2=np.ones(K))


def streamed(form, state, warm=2, timed=5):
    h = HostStreamedCAVI(form, K, state, dropout=True)
    for _ in range(warm):
        h.step()
    ms, by = [], []
    for _ in range(timed):
        b0 = h.h2d_bytes
        t0 = time.perf_counter()
        h.step()                                          # ends in a device synchronise
        ms.append(1e3 * (time.perf_counter() - t0))
        by.append(h.h2d_bytes - b0)
    return h, dict(ms_per_step_median=float(np.median(ms)), ms_per_step=ms, h2d_bytes_per_step=by[-1], slab_rows=h.slab,
                   host_form_bytes=int(form.nbytes))


def main():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                       text=True).stdout.strip().splitlines()
    out = dict(gpu=q[0] if q else torch.cuda.get_device_name(), quick=QUICK, shape=[N, P], K=K, cases=[])
    for d in DENSITIES:
        X, csr = counts(d, seed=int(d * 1000))
        nnz = int(csr.nnz)
        t_dense, Xd = ingest(X)
        t_csr, Xc = ingest(csr)
        same = bool(torch.equal(Xd, Xc))
        del Xd, Xc
        state = init_state(7)
        cm = CountMatrix(csr)
        spc, cc = cm.to_sparse_counts(), cm.to_csr_counts()
        del X
        hs, rs = streamed(spc, state)
        hc, rc = streamed(cc, state)
        worst = max(float(np.max(np.abs(hc.state_dict()[k] - hs.state_dict()[k]) / (np.abs(hs.state_dict()[k]) + 1e-30)))
                    for k in ('a1', 'a2', 'b1', 'b2'))
        del hs, hc, spc, cc
        torch.cuda.empty_cache()
        case = dict(density=d, nnz=nnz,
                    ingest=dict(dense_s=t_dense, csr_s=t_csr, dense_host_bytes=N * P * 4, csr_host_bytes=host_bytes(csr),
                                device_matrices_identical=same),
                    host_streamed=dict(sparse_counts=rs, csr_counts=rc, max_rel_param_diff=worst))
        out['cases'].append(case)
        print(json.dumps(case), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, 'w') as f:
        json.dump(out, f, indent=1)
    print('wrote', OUT)


if __name__ == '__main__':
    main()
