"""Debug: the ELBO terms of one state as the device model's flush pass and as the first host-streamed step see them."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
from oriana.models import ZIGaP
from oriana.singlecell import synth_counts_device
from oriana_b200 import _lib
from oriana_b200.host_step import HostStreamedCAVI, CompactCounts
n, p, K = (int(a) for a in sys.argv[1:4]) if len(sys.argv) > 3 else (100_000, 20_000, 20)
X = synth_counts_device(n, p, K, seed=3)
np.random.seed(1)
m = ZIGaP(X[:, :p], k=K, use_factors=False, tensor=True)
for _ in range(5): m.step()
e_dev = m.elbo()
parts_dev = m._red64[-_lib.ORI_R64_NSLOTS:].cpu().numpy().copy()      # the ORI_R64_* partials close red64
scal_dev = m._scal.cpu().numpy().copy()
state = m.state_dict()
R64 = [(s, getattr(_lib, 'ORI_R64_' + s)) for s in ('XLOGDEN', 'ENT', 'PUV', 'HROW', 'LGAMX', 'NNZ')]
SC = [(s, getattr(_lib, 'ORI_SC_' + s)) for s in ('LGAMX', 'NNZ', 'PENDING', 'ELBO_LAST', 'ITER', 'UVSUM')]
for mode in ('u8', 'f32'):
    Xh = CompactCounts.from_tensor(X[:, :p]) if mode == 'u8' else X[:, :p].cpu().pin_memory()
    h = HostStreamedCAVI(Xh, K, state, dropout=True)
    scal_h0 = h._g['scal'].cpu().numpy().copy()
    e_h = h.step()
    parts_h = h._g['red64'][-_lib.ORI_R64_NSLOTS:].cpu().numpy().copy()
    print(mode, 'ELBO dev %.10e host %.10e rel %.2e' % (e_dev, e_h, abs(e_dev - e_h) / abs(e_dev)))
    for name, i in R64:
        print('  red64 %-8s dev %.8e host %.8e' % (name, parts_dev[i], parts_h[i]))
    for name, i in SC:
        print('  scal %-9s dev %.8e host (after init) %.8e' % (name, scal_dev[i], scal_h0[i]))
    del h
