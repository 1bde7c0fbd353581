"""ctypes binding of libprogen_b200.so (the C ABI in include/progen_b200.h).

PyTorch is used for device memory and streams only; every kernel on the hot path lives in the shared library.
There is no fallback: if the library is missing, or the device is not sm_100, calls raise.
"""
import ctypes as C
import os
import torch

F32, BF16 = 0, 1
BACKEND_SIMT, BACKEND_TC = 0, 1
EPI_STORE, EPI_ROTARY, EPI_RESIDUAL, EPI_GLU, EPI_GELU, EPI_GLU_BWD, EPI_GELU_BWD, EPI_ACCUM = range(8)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libprogen_b200.so')


class ProgenError(RuntimeError):
    pass


class GemmDesc(C.Structure):
    _fields_ = [
        ('M', C.c_int32), ('N', C.c_int32), ('K', C.c_int32),
        ('a_mn_major', C.c_int32), ('b_mn_major', C.c_int32),
        ('batch', C.c_int32), ('batch_reduce', C.c_int32), ('causal', C.c_int32), ('split_k', C.c_int32),
        ('in_dtype', C.c_int32), ('out_dtype', C.c_int32), ('epi_kind', C.c_int32), ('backend', C.c_int32),
        ('seq_len', C.c_int32), ('dim_head', C.c_int32),
        ('atomic', C.c_int32), ('tril', C.c_int32), ('tril_rows', C.c_int32),
        ('lda', C.c_int64), ('ldb', C.c_int64),
        ('a_batch_rows', C.c_int64), ('b_batch_rows', C.c_int64), ('d_batch_rows', C.c_int64),
        ('ldo', C.c_int64), ('ldo2', C.c_int64), ('ldaux', C.c_int64),
        ('A', C.c_void_p), ('B', C.c_void_p), ('out', C.c_void_p), ('out2', C.c_void_p),
        ('bias', C.c_void_p), ('aux', C.c_void_p), ('rot_sin', C.c_void_p), ('rot_cos', C.c_void_p),
    ]


_lib = None

_LL, _I, _P, _F = C.c_longlong, C.c_int, C.c_void_p, C.c_float

# name -> argtypes (restype is int unless listed in _RESTYPES); must match include/progen_b200.h
PROTOTYPES = {
    'progen_version': [],
    'progen_last_error': [],
    'progen_device_check': [],
    'progen_launch_count': [],
    'progen_gemm': [C.POINTER(GemmDesc), _P],
    'progen_embed_fwd': [_P, _P, _P, _LL, _I, _I, _P],
    'progen_embed_bwd': [_P, _P, _P, _LL, _I, _I, _P],
    'progen_ln_shift_fwd': [_P, _LL, _I, _P, _P, _LL, _I, _P, _P, _LL, _I, _I, _I, _P],
    'progen_ln_shift_bwd': [_P, _LL, _I, _P, _LL, _I, _P, _P, _P, _P, _P, _LL, _P, _P, _LL, _I, _I, _I, _I, _P],
    'progen_colsum': [_P, _LL, _I, _P, _LL, _I, _P],
    'progen_ce_fwd_bwd': [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _F, _P],
    'progen_rotary_bwd': [_P, _LL, _I, _P, _P, _LL, _I, _I, _I, _P],
    'progen_local_attn_fwd_simt': [_P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    'progen_local_attn_bwd_simt': [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    'progen_local_attn_fwd': [_P, _P, _P, _I, _I, _I, _I, _I, _P],
    'progen_local_attn_fwd_tc': [_P, _P, _P, _I, _I, _I, _I, _I, _P],
    'progen_local_attn_bwd': [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    'progen_local_attn_bwd_tc': [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    'progen_local_attn_bwd_tc_ex': [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    'progen_sgu_gate_fwd': [_P, _LL, _P, _LL, _P, _P, _LL, _I, _LL, _I, _I, _P],
    'progen_sgu_gate_bwd': [_P, _LL, _P, _LL, _P, _LL, _P, _P, _LL, _P, _LL, _P, _I, _LL, _I, _I, _P],
    'progen_gelu_bwd': [_P, _P, _I, _LL, _P],
    'progen_cast_f32': [_P, _P, _I, _LL, _P],
    'progen_tril_cast': [_P, _P, _I, _I, _P],
    'progen_decode_step': [_P, _I, _P],
    'progen_decode_run': [_P, _P],
    'progen_optim_workspace_floats': [],
    'progen_grad_sqnorm': [_P, _LL, _P, _P, _P],
    'progen_adamw_step': [_P, _P, _P, _P, _P, _P, _LL, _LL, _P, _F, _F, _F, _F, _F, _F, _LL, _I, _P],
    'progen_adamw_step_dev': [_P, _P, _P, _P, _P, _P, _LL, _LL, _P, _F, _F, _F, _F, _F, _F, _I, _P, _P],
}
_RESTYPES = {'progen_version': C.c_char_p, 'progen_last_error': C.c_char_p, 'progen_launch_count': C.c_longlong}


def load():
    """Load the shared library (once).  Raises ProgenError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ProgenError(f'{LIB_PATH} not found: run `python -c "import __graft_entry__ as g; g.build()"` '
                          f'(or progen_b200/csrc/build.sh). There is no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export a declared symbol
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, C.c_int)
    _lib = lib
    return lib


def version():
    return load().progen_version().decode()


def check(rc, what=''):
    if rc != 0:
        raise ProgenError(f'{what} failed (code {rc}): {load().progen_last_error().decode()}')


def require_device():
    if not torch.cuda.is_available():
        raise ProgenError('no CUDA device: progen_b200 has no CPU fallback (sm_100a only)')
    check(load().progen_device_check(), 'progen_device_check')


def dt(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise ProgenError(f'unsupported dtype {t.dtype}')


def ptr(t):
    return 0 if t is None else t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def gemm(*, M, N, K, A, lda, B, ldb, out, ldo, epi=EPI_STORE, backend, a_mn=False, b_mn=False, in_dtype, out_dtype=F32,
         batch=1, a_batch_rows=0, b_batch_rows=0, d_batch_rows=0, batch_reduce=False, causal=0, split_k=1,
         out2=None, ldo2=0, bias=None, aux=None, ldaux=0, rot_sin=None, rot_cos=None, seq_len=0, dim_head=0,
         atomic=False, tril=False, tril_rows=0):
    """Thin wrapper over progen_gemm; tensors are passed as torch tensors (or raw ints for sub-views)."""
    d = GemmDesc()
    d.M, d.N, d.K = M, N, K
    d.a_mn_major, d.b_mn_major = int(a_mn), int(b_mn)
    d.batch, d.batch_reduce, d.causal, d.split_k = batch, int(batch_reduce), causal, split_k
    d.in_dtype, d.out_dtype, d.epi_kind, d.backend = in_dtype, out_dtype, epi, backend
    d.seq_len, d.dim_head = seq_len, dim_head
    d.atomic, d.tril, d.tril_rows = int(atomic), int(tril), tril_rows
    d.lda, d.ldb = lda, ldb
    d.a_batch_rows, d.b_batch_rows, d.d_batch_rows = a_batch_rows, b_batch_rows, d_batch_rows
    d.ldo, d.ldo2, d.ldaux = ldo, ldo2, ldaux
    as_ptr = lambda x: x if isinstance(x, int) else ptr(x)
    d.A, d.B, d.out, d.out2 = as_ptr(A), as_ptr(B), as_ptr(out), as_ptr(out2)
    d.bias, d.aux, d.rot_sin, d.rot_cos = as_ptr(bias), as_ptr(aux), as_ptr(rot_sin), as_ptr(rot_cos)
    check(load().progen_gemm(C.byref(d), stream()), 'progen_gemm')
