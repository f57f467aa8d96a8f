"""The device state as the library sees it (`ori_problem_t`, include/oriana_b200.h): kernel plan, gene-side and reduction
buffers, and the problem that points at them; shared by the device models and the host-streamed step."""
import ctypes

import torch

from . import _lib


def row_pitch(p):
    """Floats per row of X in HBM: p rounded up to 4, the 16-byte row pitch the kernels read."""
    return (p + 3) // 4 * 4


def pad_k(K):
    for kp in (8, 16, 32, 64):
        if K <= kp:
            return kp
    raise ValueError('k=%d: the CUDA kernels support latent dimensions up to 64' % K)


def kernel_plan(k, entries, precise=False, tensor=None, force_simt=False, sparse=False):
    """(tensor, KP, flags) for k latent dimensions and `entries` matrix entries (of the problem, or of one slab).

    The tcgen05/TMA tensor path (k <= 64, tf32 contractions, fp32 accumulation) is the default for problems that fill the
    machine.  precise=True: on the tensor path (k <= 32) R, D_hat and the factor operands of the accumulating contractions
    are split hi/lo (ORI_F_PRECISE, about half the rate); for k > 32 the CUDA-core kernels run, as they do for the sparse
    model at k > 32.  `flags`: ORI_F_PRECISE and ORI_F_NO_TENSOR."""
    if sparse and k > 64:
        raise ValueError('SparseZIGaP supports k <= 64')
    if sparse and k > 32:
        if tensor:
            raise ValueError('SparseZIGaP: the tensor path needs k <= 32 (32 < k <= 64 runs on the CUDA-core kernels)')
        tensor = False
    if tensor is None:
        tensor = not force_simt and k <= 64 and entries >= (1 << 21)
    if tensor and (k > 64 or force_simt):
        raise ValueError('the tensor path needs k <= 64 and force_simt=False')
    tensor = bool(tensor) and not (precise and k > 32)
    KP = (32 if k <= 32 else 64) if tensor else pad_k(k)
    return tensor, KP, (_lib.ORI_F_PRECISE if precise and tensor else 0) | (_lib.ORI_F_NO_TENSOR if force_simt else 0)


def gene_buffers(p, K, KP, device, dropout, sparse, trace_cap):
    """The gene-side state and the reduction buffers under their `ori_problem_t` names; lp, pfloor and pi_d with dropout
    only, a third gene-side sum for the sparse model."""
    f32, f64 = dict(dtype=torch.float32, device=device), dict(dtype=torch.float64, device=device)
    return dict(
        b1=torch.zeros((p, KP), **f32), b2=torch.zeros((p, KP), **f32), V_hat=torch.zeros((p, KP), **f32),
        eV=torch.zeros((p, KP), **f32), red32=torch.zeros((3 if sparse else 2, p, KP), **f32),
        lp=torch.full((p,), float('-inf'), **f32) if dropout else None,
        pfloor=torch.zeros((p,), **f32) if dropout else None, pi_d=torch.zeros((p,), **f64) if dropout else None,
        hyper=torch.ones((4, K), **f64), red64=torch.zeros((p + 2 * KP + _lib.R64_NSLOTS,), **f64),
        gsum=torch.zeros((2 * KP + 8,), **f64), scal=torch.zeros((_lib.SCAL_SLOTS,), **f64),
        elbo_trace=torch.zeros((trace_cap,), **f64))


_FIELDS = dict(_lib.OriProblem._fields_)
_SIZES = {'tc_ws': 'tc_ws_floats', 'det_ws': 'det_ws_doubles'}
_PAIR = ctypes.c_void_p * 2                         # the two generations of a row-side factor


def build_problem(**fields):
    """An `OriProblem` from its scalar fields and named arrays: a tensor gives its device pointer, None gives NULL, the
    two-generation fields take a pair, and the workspaces bring their sizes.  An unknown name raises TypeError."""
    P = _lib.OriProblem()
    for name, v in fields.items():
        ty = _FIELDS.get(name)
        if ty is ctypes.c_void_p:
            setattr(P, name, None if v is None else v.data_ptr())
            if name in _SIZES and v is not None:
                setattr(P, _SIZES[name], v.numel())
        elif ty is _PAIR:
            getattr(P, name)[:] = [None if t is None else t.data_ptr() for t in v]
        elif ty is None or name in _SIZES.values():
            raise TypeError('ori_problem_t has no field %r to fill' % name)
        else:
            setattr(P, name, v)
    return P


def logit_pi(pi):
    """(lp, pfloor) of the dropout prior pi (float64 tensor): lp = float32(logit(pi)), -inf / +inf at pi <= 0 / pi >= 1,
    and the 1e-10 floor of D_hat (zigap.py:133) where pi <= 0."""
    pc = torch.clamp(pi, 1e-15, 1. - 1e-15)
    lp = torch.log(pc / (1. - pc))
    lp = torch.where(pi <= 0, torch.full_like(lp, float('-inf')), lp)
    lp = torch.where(pi >= 1, torch.full_like(lp, float('inf')), lp)
    return lp.to(torch.float32), torch.where(pi <= 0, 1e-10, 0.).to(torch.float32)
