"""ctypes binding of liboriana_b200.so (the C ABI declared in include/oriana_b200.h).

There is no CPU fallback: every compute entry point of this package goes through this library and
raises when it (or an sm_100 GPU) is missing.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('ORIANA_B200_LIB') or os.path.join(_HERE, 'lib', 'liboriana_b200.so')   # override: kernel A/B runs

ORI_F_DROPOUT, ORI_F_QUIRK, ORI_F_ELBO, ORI_F_NO_TENSOR, ORI_F_SPARSE, ORI_F_DEVICE_ITER, ORI_F_PRECISE = 1, 2, 4, 8, 16, 32, 64
ORI_F_FIXED_CHAIN = 128
ORI_F_DETERMINISTIC = 256
ORI_F_X_U16 = 512
ORI_CSR_U8, ORI_CSR_U16, ORI_CSR_F32 = 1, 2, 4       # value types of ori_expand_csr_counts (their size in bytes)
ORI_M_STEP, ORI_M_INIT, ORI_M_INIT_KEEP, ORI_M_FINALIZE, ORI_M_REFRESH = 0, 1, 2, 3, 4

# layout of the reduction buffers of `ori_problem_t` (the ORI_R64_* / ORI_GSUM_* / ORI_SC_* slots and size macros)
ORI_R64_XLOGDEN, ORI_R64_ENT, ORI_R64_PUV, ORI_R64_HROW, ORI_R64_LGAMX, ORI_R64_NNZ, ORI_R64_NSLOTS = 0, 1, 2, 3, 4, 5, 8
ORI_GSUM_HGENE, ORI_GSUM_NSLOTS = 0, 8
ORI_SC_LGAMX, ORI_SC_NNZ, ORI_SC_PENDING, ORI_SC_ELBO_LAST, ORI_SC_ITER, ORI_SC_UVSUM, ORI_SC_NSLOTS = 0, 1, 2, 4, 5, 6, 16


def ORI_RED32_FLOATS(p, KP, third):
    return (3 if third else 2) * p * KP


def ORI_RED64_DOUBLES(p, KP):
    return p + 2 * KP + ORI_R64_NSLOTS


def ORI_GSUM_DOUBLES(KP):
    return 2 * KP + ORI_GSUM_NSLOTS


_fp = C.POINTER(C.c_float)
_dp = C.POINTER(C.c_double)


class OriProblem(C.Structure):
    """Mirror of `ori_problem_t` (include/oriana_b200.h)."""
    _fields_ = [
        ('n_rows', C.c_int64), ('n_total', C.c_int64), ('ldx', C.c_int64),
        ('p', C.c_int32), ('K', C.c_int32), ('KP', C.c_int32), ('flags', C.c_uint32),
        ('iter', C.c_int32), ('trace_cap', C.c_int32),
        ('X', C.c_void_p),
        ('a1', C.c_void_p), ('a2', C.c_void_p),
        ('U_hat', C.c_void_p * 2), ('eU', C.c_void_p * 2),
        ('eUw', C.c_void_p), ('Zi', C.c_void_p), ('a2s', C.c_void_p),
        ('b1', C.c_void_p), ('b2', C.c_void_p), ('V_hat', C.c_void_p), ('eV', C.c_void_p),
        ('red32', C.c_void_p), ('lp', C.c_void_p), ('pfloor', C.c_void_p),
        ('hyper', C.c_void_p), ('red64', C.c_void_p), ('gsum', C.c_void_p), ('pi_d', C.c_void_p),
        ('scal', C.c_void_p), ('elbo_trace', C.c_void_p),
        ('tc_ws', C.c_void_p), ('tc_ws_floats', C.c_int64),
        ('p_s', C.c_void_p), ('logV', C.c_void_p), ('eVd', C.c_void_p), ('eVz', C.c_void_p), ('Vh_old', C.c_void_p),
        ('eUl', C.c_void_p * 2), ('pi_s', C.c_void_p), ('tau', C.c_double),
        ('xrow', C.c_void_p), ('xcol', C.c_void_p), ('thrU', C.c_void_p), ('thrV', C.c_void_p), ('det_ws', C.c_void_p), ('det_ws_doubles', C.c_int64),
    ]


_PP = C.POINTER(OriProblem)
_SIGNATURES = {
    'ori_version': ([], C.c_int),
    'ori_kernel_launches': ([], C.c_uint64),
    'ori_last_error': ([C.c_char_p, C.c_size_t], C.c_int),
    'ori_device_check': ([C.c_int], C.c_int),
    'ori_special_f64': ([C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p], C.c_int),
    'ori_gamma_expect_f32': ([C.c_void_p] * 5 + [C.c_int64, C.c_void_p], C.c_int),
    'ori_tc_workspace_floats': ([C.c_int64, C.c_int32, C.c_int32], C.c_int64),
    'ori_det_workspace_doubles': ([C.c_int64, C.c_int32, C.c_int32], C.c_int64),
    'ori_uses_tensor_path': ([_PP], C.c_int),
    'ori_problem_check': ([_PP], C.c_int),
    'ori_count_stats': ([_PP, C.c_void_p], C.c_int),
    'ori_init_expectations': ([_PP, C.c_int, C.c_void_p], C.c_int),
    'ori_zero_accumulators': ([_PP, C.c_int, C.c_void_p], C.c_int),
    'ori_pass_rows': ([_PP, C.c_int, C.c_void_p], C.c_int),
    'ori_row_update': ([_PP, C.c_int, C.c_int, C.c_void_p], C.c_int),
    'ori_pass_genes': ([_PP, C.c_int, C.c_void_p], C.c_int),
    'ori_gene_update': ([_PP, C.c_int, C.c_void_p], C.c_int),
    'ori_mstep': ([_PP, C.c_int, C.c_void_p], C.c_int),
    'ori_cavi_step': ([_PP, C.c_int, C.c_void_p], C.c_int),
    'ori_cavi_step_local': ([_PP, C.c_int, C.c_void_p], C.c_int),
    'ori_cavi_step_global': ([_PP, C.c_int, C.c_void_p], C.c_int),
    'ori_finalize_local': ([_PP, C.c_int, C.c_void_p], C.c_int),
    'ori_dropout_posterior_f32': ([_PP, C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p], C.c_int),
    'ori_row_sums_f32': ([C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p], C.c_int),
    'ori_column_sums_f64': ([C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p], C.c_int),
    'ori_row_sums_u16_f32': ([C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p], C.c_int),
    'ori_column_sums_u16_f64': ([C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p], C.c_int),
    'ori_deviance_sums': ([_PP, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    'ori_zigap_compute_Z_q_expectations_host': ([C.c_void_p] * 7 + [C.c_int64] * 3 + [C.c_int], C.c_int),
    'ori_gap_compute_Z_q_expectations_host': ([C.c_void_p] * 5 + [C.c_int64] * 3, C.c_int),
    'ori_ctx_create': ([C.POINTER(C.c_void_p), C.c_int64], C.c_int),
    'ori_ctx_destroy': ([C.c_void_p], C.c_int),
    'ori_ctx_stats': ([C.c_void_p] + [C.POINTER(C.c_uint64)] * 4, C.c_int),
    'ori_zigap_compute_Z_q_expectations_ctx': ([C.c_void_p] * 8 + [C.c_int64] * 3 + [C.c_int], C.c_int),
    'ori_gap_compute_Z_q_expectations_ctx': ([C.c_void_p] * 6 + [C.c_int64] * 3, C.c_int),
    'ori_sparse_zigap_compute_Z_q_expectations_host': ([C.c_void_p] * 9 + [C.c_int64] * 3, C.c_int),
    'ori_sparse_zigap_compute_Z_q_expectations_ctx': ([C.c_void_p] * 10 + [C.c_int64] * 3, C.c_int),
    'ori_widen_counts_f32': ([C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p], C.c_int),
    'ori_expand_bitmap_counts_f32': ([C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64,
                                      C.c_int32, C.c_void_p], C.c_int),
    'ori_expand_csr_counts': ([C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                               C.c_int64, C.c_int64, C.c_int32, C.c_void_p], C.c_int),
    'ori_scatter_counts_f32': ([C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int64, C.c_void_p], C.c_int),
    'ori_synth_counts_f32': ([C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_uint64,
                              C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
}

_lib = None


class OrianaB200Error(RuntimeError):
    pass


def exported_symbols():
    """Names every build of the library must export (checked by tests against include/oriana_b200.h)."""
    return sorted(_SIGNATURES)


def load():
    """Load the shared library (building is `python -m oriana_b200.build` / `__graft_entry__.build()`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OrianaB200Error(
                'liboriana_b200.so is missing (%s): run `python -m oriana_b200.build`. '
                'oriana_b200 has no CPU fallback.' % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (args, res) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = res
        _lib = lib
    return _lib


def last_error():
    buf = C.create_string_buffer(512)
    load().ori_last_error(buf, 512)
    return buf.value.decode(errors='replace')


def check(rc):
    if rc != 0:
        raise OrianaB200Error('oriana_b200 C ABI error %d: %s' % (rc, last_error()))


def require_cuda():
    """Raise unless the library is built and a CUDA device is visible to torch."""
    import torch
    load()
    if not torch.cuda.is_available():
        raise OrianaB200Error('no CUDA device: oriana_b200 computes only on sm_100a GPUs (no CPU fallback)')
    return torch.device('cuda', torch.cuda.current_device())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
