"""ctypes binding of libdalle_b200.so (C ABI declared in include/dalle_b200.h).

The shared library is the product: if it cannot be loaded (or built) every op raises — there is no
PyTorch/CPU fallback behind these calls.
"""
import ctypes
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('DALLE_B200_LIB') or os.path.join(_HERE, 'libdalle_b200.so')   # env override: A/B builds only
CSRC = os.path.join(_HERE, 'csrc')

c_int, c_float, c_void_p, c_int64 = ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_int64

# enums (include/dalle_b200.h)
F32, BF16 = 0, 1
ATTN_FULL, ATTN_AXIAL_ROW, ATTN_AXIAL_COL, ATTN_CONV_LIKE, ATTN_STATIC = 0, 1, 2, 3, 4
EPI_STORE, EPI_QKV, EPI_RESID, EPI_GEGLU, EPI_GEGLU_BWD = 0, 1, 2, 3, 4
GEMM_AUTO, GEMM_SIMT, GEMM_TCGEN05, GEMM_SMALLM = 0, 1, 2, 3


class LnShiftFwdParams(ctypes.Structure):
    _fields_ = [('batch', c_int), ('n', c_int), ('d', c_int), ('text_len', c_int), ('fmap', c_int),
                ('do_ln', c_int), ('do_shift', c_int), ('out_dtype', c_int), ('eps', c_float),
                ('x', c_void_p), ('gamma', c_void_p), ('beta', c_void_p), ('out', c_void_p),
                ('mean', c_void_p), ('rstd', c_void_p)]


class LnShiftBwdParams(ctypes.Structure):
    _fields_ = [('batch', c_int), ('n', c_int), ('d', c_int), ('text_len', c_int), ('fmap', c_int),
                ('do_ln', c_int), ('do_shift', c_int), ('dout_dtype', c_int),
                ('d_out', c_void_p), ('x', c_void_p), ('mean', c_void_p), ('rstd', c_void_p), ('gamma', c_void_p),
                ('dres', c_void_p), ('dx', c_void_p), ('dgamma', c_void_p), ('dbeta', c_void_p),
                ('up_y', c_void_p), ('up_scale', c_void_p), ('up_sign', c_float), ('up_dy', c_void_p), ('up_dscale', c_void_p),
                ('up_dbias', c_void_p)]


class GemmParams(ctypes.Structure):
    _fields_ = [('M', c_int), ('N', c_int), ('K', c_int), ('dtype', c_int), ('backend', c_int),
                ('A', c_void_p), ('lda', c_int64), ('a_mn_major', c_int),
                ('B', c_void_p), ('ldb', c_int64), ('b_mn_major', c_int),
                ('epilogue', c_int),
                ('C', c_void_p), ('ldc', c_int64), ('c_dtype', c_int), ('bias', c_void_p), ('split_k_ok', c_int),
                ('C_multicast', c_void_p), ('c_scale', c_float),
                ('q', c_void_p), ('k', c_void_p), ('v', c_void_p), ('cos_t', c_void_p), ('sin_t', c_void_p),
                ('seq_n', c_int), ('heads', c_int), ('dim_head', c_int), ('pos_offset', c_int), ('q_scale', c_float),
                ('resid', c_void_p), ('scale', c_void_p), ('sign', c_float), ('y_out', c_void_p), ('out', c_void_p),
                ('u_out', c_void_p), ('h_out', c_void_p), ('hidden', c_int), ('u_in', c_void_p), ('du_out', c_void_p)]


class AttnFwdParams(ctypes.Structure):
    _fields_ = [('batch', c_int), ('heads', c_int), ('n_q', c_int), ('n_k', c_int), ('dim_head', c_int),
                ('dtype', c_int), ('pattern', c_int), ('causal', c_int), ('stable', c_int),
                ('text_len', c_int), ('fmap', c_int), ('kernel_size', c_int), ('dilation', c_int), ('gather', c_int), ('kv_rows', c_int),
                ('key_mask', c_void_p), ('static_mask', c_void_p), ('static_ld', c_int64),
                ('q', c_void_p), ('k', c_void_p), ('v', c_void_p), ('out', c_void_p), ('lse', c_void_p)]


class AttnBwdParams(ctypes.Structure):
    _fields_ = [('f', AttnFwdParams), ('d_out', c_void_p), ('cos_t', c_void_p), ('sin_t', c_void_p),
                ('q_scale', c_float), ('delta', c_void_p), ('dqkv', c_void_p)]


class ScaleBwdParams(ctypes.Structure):
    _fields_ = [('rows', c_int), ('d', c_int), ('dtype', c_int), ('sign', c_float),
                ('d_out', c_void_p), ('y', c_void_p), ('scale', c_void_p), ('dy', c_void_p),
                ('dscale', c_void_p), ('dbias', c_void_p)]


class AdamParams(ctypes.Structure):
    _fields_ = [('p', c_void_p), ('g', c_void_p), ('m', c_void_p), ('v', c_void_p), ('count', c_int64),
                ('lr', c_float), ('beta1', c_float), ('beta2', c_float), ('eps', c_float), ('weight_decay', c_float),
                ('step', c_int), ('max_norm', c_float), ('gnorm_sq', c_void_p)]


_STRUCTS = (LnShiftFwdParams, LnShiftBwdParams, GemmParams, AttnFwdParams, AttnBwdParams, ScaleBwdParams, AdamParams)

_lib = None
_lock = threading.Lock()


def build(force=False, verbose=False):
    """Compile libdalle_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    if force:
        for f in os.listdir(os.path.join(CSRC, 'build')) if os.path.isdir(os.path.join(CSRC, 'build')) else []:
            if f.endswith('.o'):
                os.remove(os.path.join(CSRC, 'build', f))
    r = subprocess.run(['bash', os.path.join(CSRC, 'build.sh')], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout)
        print(r.stderr)
    if r.returncode != 0:
        raise RuntimeError('building libdalle_b200.so failed:\n' + r.stdout + r.stderr)
    return LIB_PATH


def _declare(lib):
    lib.dalle_b200_version.restype = c_int
    lib.dalle_b200_last_error.restype = ctypes.c_char_p
    lib.dalle_b200_device_ok.argtypes = [c_int]
    lib.dalle_b200_abi_sizes.argtypes = [ctypes.POINTER(c_int), c_int]
    for name, st in (('ln_shift_fwd', LnShiftFwdParams), ('ln_shift_bwd', LnShiftBwdParams), ('gemm', GemmParams),
                     ('attn_fwd', AttnFwdParams), ('attn_bwd', AttnBwdParams), ('scale_bwd', ScaleBwdParams)):
        fn = getattr(lib, 'dalle_b200_' + name)
        fn.argtypes = [ctypes.POINTER(st), c_void_p]
        fn.restype = c_int
    lib.dalle_b200_gemm_select.argtypes = [ctypes.POINTER(GemmParams)]
    lib.dalle_b200_gemm_select.restype = c_int
    lib.dalle_b200_colsum.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]
    lib.dalle_b200_qkv_rotary.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p]
    lib.dalle_b200_geglu_bwd.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]
    lib.dalle_b200_ce_fwd.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p]
    lib.dalle_b200_ce_bwd.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p]
    lib.dalle_b200_cast_bf16.argtypes = [c_void_p, c_void_p, c_int64, c_void_p]
    lib.dalle_b200_mc_add.argtypes = [c_void_p, c_void_p, c_int64, c_float, c_void_p]
    lib.dalle_b200_split_bf16x3.argtypes = [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p]
    lib.dalle_b200_resid_scale.argtypes = [c_void_p, c_int, c_void_p, c_void_p, c_float, c_void_p, c_int64, c_int, c_void_p]
    lib.dalle_b200_sample_topk_gumbel.argtypes = [c_void_p, c_int, c_int, c_int, c_int64, c_int, c_float, c_void_p, ctypes.c_uint64, ctypes.c_uint64, c_void_p, c_void_p]
    lib.dalle_b200_sample_guided_topk_gumbel.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_float, c_int, c_float, c_void_p, ctypes.c_uint64, ctypes.c_uint64,
                                                          c_void_p, c_void_p]
    lib.dalle_b200_decode_shift.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]
    lib.dalle_b200_decode_kv_append.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]
    lib.dalle_b200_dropout.argtypes = [c_void_p, c_void_p, c_int, c_int64, c_float, ctypes.c_uint64, ctypes.c_uint64, c_void_p]
    lib.dalle_b200_geglu_fwd.argtypes = [c_void_p, c_void_p, c_int64, c_int, c_void_p]
    lib.dalle_b200_axpby.argtypes = [c_void_p, c_void_p, c_float, c_void_p, c_int64, c_void_p]
    lib.dalle_b200_sumsq.argtypes = [c_void_p, c_int64, c_void_p, c_void_p]
    lib.dalle_b200_adam.argtypes = [ctypes.POINTER(AdamParams), c_void_p]
    lib.dalle_b200_embed_fwd.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]
    lib.dalle_b200_embed_bwd.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]
    sizes = (c_int * 8)()
    n = lib.dalle_b200_abi_sizes(sizes, 8)
    assert n == len(_STRUCTS)
    for i, st in enumerate(_STRUCTS):
        if ctypes.sizeof(st) != sizes[i]:
            raise RuntimeError(f'ABI mismatch for {st.__name__}: ctypes {ctypes.sizeof(st)} vs C {sizes[i]}')


def lib():
    """The loaded library (loads on first use; builds it first if the .so is missing and nvcc is present)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                build()
            l = ctypes.CDLL(LIB_PATH)
            _declare(l)
            _lib = l
    return _lib


def check(rc, what=''):
    if rc != 0:
        msg = lib().dalle_b200_last_error().decode('utf-8', 'replace')
        raise RuntimeError(f'libdalle_b200 {what} failed (status {rc}): {msg}')


EXPORTED = ['dalle_b200_version', 'dalle_b200_last_error', 'dalle_b200_device_ok', 'dalle_b200_abi_sizes',
            'dalle_b200_ln_shift_fwd', 'dalle_b200_ln_shift_bwd', 'dalle_b200_gemm', 'dalle_b200_gemm_select', 'dalle_b200_attn_fwd',
            'dalle_b200_attn_bwd', 'dalle_b200_scale_bwd', 'dalle_b200_colsum', 'dalle_b200_qkv_rotary', 'dalle_b200_geglu_bwd', 'dalle_b200_ce_fwd', 'dalle_b200_ce_bwd', 'dalle_b200_cast_bf16', 'dalle_b200_mc_add', 'dalle_b200_split_bf16x3', 'dalle_b200_resid_scale', 'dalle_b200_dropout', 'dalle_b200_sample_topk_gumbel', 'dalle_b200_sample_guided_topk_gumbel', 'dalle_b200_decode_shift', 'dalle_b200_decode_kv_append', 'dalle_b200_geglu_fwd',
            'dalle_b200_axpby', 'dalle_b200_embed_fwd', 'dalle_b200_embed_bwd', 'dalle_b200_sumsq', 'dalle_b200_adam', 'dalle_b200_debug_attn_timeline']
