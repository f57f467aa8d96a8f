"""GPU, needs >= 2 devices (skipped on a single-GPU box): the device models row-sharded over two ranks on NCCL against
the same models unsharded -- ZIGaP on the tensor path, ZIGaP at K = 40 on uint16 storage, and SparseZIGaP with its
deviance metrics (integer sums all-reduced as int64)."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        from oracle import cavi_numpy as cn, sparse_numpy as sn
        from oriana.models import SparseZIGaP, ZIGaP
        from oriana.singlecell import CountMatrix
        from oriana_b200.sharding import RowSharding
        res = {}
        # ---- SparseZIGaP, CUDA-core kernels
        n, p, K = 901, 333, 6
        X = cn.synth_counts(n, p, K, seed=21)
        s = sn.init_state(X, K, np.random.default_rng(2))
        r0, r1 = RowSharding.row_block(n, rank, world)
        mine = {k: (v[r0:r1].copy() if k in ('X', 'a1', 'a2', 'p_d') else v.copy()) for k, v in s.items()}
        ms = SparseZIGaP(CountMatrix(mine['X']), k=K, use_factors=False, state=mine, sharded=True)
        full = SparseZIGaP(CountMatrix(X), k=K, use_factors=False, state=s) if rank == 0 else None
        for _ in range(3):
            ms.step()
            if full is not None:
                full.step()
        dev, expl = ms.reconstruction_deviance(), ms.explained_deviance()
        if rank == 0:
            for k in ('b1', 'b2', 'p_s', 'pi_s', 'pi_d', 'alpha1', 'beta2'):
                a, b = getattr(ms, k).asarray(), getattr(full, k).asarray()
                res['sparse_' + k] = float(np.max(np.abs(a - b) / (np.abs(b) + 1e-6 * np.abs(b).max())))
            a, b = ms.a1.asarray(), full.a1.asarray()[r0:r1]
            res['sparse_a1'] = float(np.max(np.abs(a - b) / (np.abs(b) + 1e-6 * np.abs(b).max())))
            d0 = full.reconstruction_deviance(); e0 = full.explained_deviance()
            res['sparse_deviance'] = abs(dev - d0) / abs(d0) if np.isfinite(d0) else float(dev != d0)
            res['sparse_explained'] = abs(expl - e0) / abs(e0) if np.isfinite(e0) else float(expl != e0)
        # ---- ZIGaP, tensor path
        n, p, K = 6000, 1500, 12
        X = cn.synth_counts(n, p, K, seed=22)
        s = cn.init_state(X, K, np.random.default_rng(3), 'zigap')
        r0, r1 = RowSharding.row_block(n, rank, world)
        mine = {k: (v[r0:r1].copy() if k in ('X', 'a1', 'a2', 'p_d') else v.copy()) for k, v in s.items()}
        mz = ZIGaP(CountMatrix(mine['X']), k=K, use_factors=False, state=mine, sharded=True, tensor=True)
        fz = ZIGaP(CountMatrix(X), k=K, use_factors=False, state=s, tensor=True) if rank == 0 else None
        for _ in range(3):
            mz.step()
            if fz is not None:
                fz.step()
        tr = mz.elbo_trace
        # graph replay is a single-rank feature (capturing the NCCL all-reduces hung on this stack): refused up front
        try:
            ZIGaP(CountMatrix(mine['X']), k=K, use_factors=False, state=mine, sharded=True, tensor=True, graphs=True)
            refused = False
        except ValueError:
            refused = True
        assert refused
        if rank == 0:
            for k in ('b1', 'b2', 'pi_d', 'alpha1', 'beta2'):
                a, b = getattr(mz, k).asarray(), getattr(fz, k).asarray()
                res['zigap_' + k] = float(np.max(np.abs(a - b) / (np.abs(b) + 1e-6 * np.abs(b).max())))
            res['zigap_elbo'] = float(np.max(np.abs(tr - fz.elbo_trace) / np.abs(fz.elbo_trace)))
        # ---- ZIGaP, tensor path, K = 40 (KP = 64), each rank's row block kept as uint16 in HBM, against the unsharded
        # float32 model.  uint16 storage is forced here, in the spawned process: the models choose it only where float32
        # would not fit the device
        import torch
        from oriana_b200 import problem
        problem.counts_storage = lambda u16, *args: torch.uint16 if u16 else torch.float32
        n, p, K = 5000, 1200, 40
        X = cn.synth_counts(n, p, K, seed=23)
        X[7, 11] = 65535
        s = cn.init_state(X, K, np.random.default_rng(4), 'zigap')
        r0, r1 = RowSharding.row_block(n, rank, world)
        mine = {k: (v[r0:r1].copy() if k in ('X', 'a1', 'a2', 'p_d') else v.copy()) for k, v in s.items()}
        mu = ZIGaP(CountMatrix(mine['X'].astype(np.uint16)), k=K, use_factors=False, state=mine, sharded=True, tensor=True)
        assert mu.counts_dtype == torch.uint16 and mu._X.element_size() == 2 and mu._ldx % 8 == 0
        fu = ZIGaP(CountMatrix(X.astype(np.float32)), k=K, use_factors=False, state=s, tensor=True) if rank == 0 else None
        assert fu is None or fu.counts_dtype == torch.float32
        for _ in range(3):
            mu.step()
            if fu is not None:
                fu.step()
        tr = mu.elbo_trace
        if rank == 0:
            for k in ('b1', 'b2', 'pi_d', 'alpha1', 'beta2'):
                a, b = getattr(mu, k).asarray(), getattr(fu, k).asarray()
                res['zigap_u16_' + k] = float(np.max(np.abs(a - b) / (np.abs(b) + 1e-6 * np.abs(b).max())))
            a, b = mu.a1.asarray(), fu.a1.asarray()[r0:r1]
            res['zigap_u16_a1'] = float(np.max(np.abs(a - b) / (np.abs(b) + 1e-6 * np.abs(b).max())))
            res['zigap_u16_elbo'] = float(np.max(np.abs(tr - fu.elbo_trace) / np.abs(fu.elbo_trace)))
            out.update(res)
    finally:
        dist.destroy_process_group()


def test_two_gpu_sharded_models_match_unsharded(cuda_lib):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
        res = dict(out)
    assert res, 'rank 0 reported nothing'
    print(res)
    for k, e in res.items():
        if k in ('zigap_elbo', 'zigap_u16_elbo'):
            tol = 1e-5
        elif k in ('sparse_deviance', 'sparse_explained'):     # integer-truncated sums masked by round(D_hat): they inherit
            tol = 2e-4                                         # the p_s differences below (measured 4e-7 ... 6e-5 between runs)
        elif k.startswith('sparse'):      # the S update amplifies the order of the float32 sums; b1, b2, a1 inherit S_hat
            tol = 5e-3 if k in ('sparse_p_s', 'sparse_pi_s') else 2e-3
        else:
            tol = 5e-4
        assert e < tol, (k, e, res)
