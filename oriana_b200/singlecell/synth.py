"""Synthetic zero-inflated negative-binomial counts generated in HBM (bench / large tests only).

The host cannot hold BASELINE.json's larger configurations, so each rank generates its row block with the
library's counter-based generator (`ori_synth_counts_f32`, csrc/synth.cu).  The reference's own generator
(oriana/singlecell/generation.py) is provided in `generation.py`; its counts are not Poisson draws (SURVEY.md
section 2 #13), so the bench does not use it.
"""
import torch

from .. import _lib
from ..problem import row_pitch


def synth_counts_device(n_rows, p, K, seed=0, zero_level=0.5, nb=True, row0=0, ldx=None, chunk_rows=None):
    """Returns a float32 CUDA tensor [n_rows, ldx] (ldx = p rounded up to 4; pad columns are zero)."""
    dev = _lib.require_cuda()
    lib = _lib.load()
    ldx = ldx or row_pitch(p)
    X = torch.empty((n_rows, ldx), dtype=torch.float32, device=dev)
    chunk = chunk_rows or max(1, min(n_rows, (1 << 28) // max(1, ldx)))
    Vs = torch.empty((p, K), dtype=torch.float32, device=dev)
    pi = torch.empty((p,), dtype=torch.float32, device=dev)
    Us = torch.empty((chunk, K), dtype=torch.float32, device=dev)
    for r in range(0, n_rows, chunk):
        rows = min(chunk, n_rows - r)
        _lib.check(lib.ori_synth_counts_f32(X[r:r + rows].data_ptr(), ldx, row0 + r, rows, p, K, seed,
                                            float(zero_level), int(bool(nb)), Us.data_ptr(), Vs.data_ptr(),
                                            pi.data_ptr(), _lib.stream_ptr()))
    return X
