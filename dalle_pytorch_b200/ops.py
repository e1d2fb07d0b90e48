"""Thin torch-tensor wrappers over the C ABI (include/dalle_b200.h).  No arithmetic happens in Python:
each function fills a POD struct with device pointers and enqueues the kernel on the current CUDA stream.
Tensors are allocated by torch (the library never owns memory, SURVEY.md §8b)."""
import contextlib
import ctypes
import os

import torch

from . import _lib, config
from ._lib import (F32, BF16, EPI_STORE, EPI_QKV, EPI_RESID, EPI_GEGLU, EPI_GEGLU_BWD, GEMM_AUTO,
                   ATTN_FULL, ATTN_AXIAL_ROW, ATTN_AXIAL_COL, ATTN_CONV_LIKE, ATTN_STATIC)

_launch_count = 0          # kernels-launching ABI calls (bench.py reports it as gpu_launches)


def launches():
    return _launch_count


def _count(n=1):
    global _launch_count
    _launch_count += n


def dt_code(dtype):
    if dtype == torch.float32:
        return F32
    if dtype == torch.bfloat16:
        return BF16
    raise TypeError(f'unsupported compute dtype {dtype}')


def _p(t):
    if t is None:
        return None
    assert t.is_cuda, 'libdalle_b200 operates on CUDA tensors only (no CPU fallback)'
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _c(t):
    assert t.is_contiguous(), 'expected a contiguous tensor'
    return t


# ------------------------------------------------------------------------------------------------
def ln_shift_fwd(x, gamma, beta, out_dtype, text_len, fmap, do_ln=True, do_shift=True, eps=1e-5):
    """x [b,n,d] fp32 -> (out [b*n,d] out_dtype, mean [b*n], rstd [b*n])"""
    b, n, d = x.shape
    _c(x)
    assert x.dtype == torch.float32
    out = torch.empty(b * n, d, device=x.device, dtype=out_dtype)
    mean = torch.empty(b * n, device=x.device, dtype=torch.float32) if do_ln else None
    rstd = torch.empty(b * n, device=x.device, dtype=torch.float32) if do_ln else None
    P = _lib.LnShiftFwdParams(batch=b, n=n, d=d, text_len=text_len, fmap=fmap, do_ln=int(do_ln), do_shift=int(do_shift),
                              out_dtype=dt_code(out_dtype), eps=eps, x=_p(x), gamma=_p(gamma), beta=_p(beta), out=_p(out),
                              mean=_p(mean), rstd=_p(rstd))
    _lib.check(_lib.lib().dalle_b200_ln_shift_fwd(ctypes.byref(P), _stream()), 'ln_shift_fwd')
    _count()
    return out, mean, rstd


def ln_shift_bwd(d_out, x, mean, rstd, gamma, dres, text_len, fmap, do_ln=True, do_shift=True, dgamma=None, dbeta=None, up=None,
                 up_zeroed=None):
    """-> dx [b,n,d] fp32 ; dgamma/dbeta accumulated in place (must be zero-initialised by the caller).
    `up` = (up_y | None, up_scale | None, up_sign): also form the upstream sub-layer's LayerScale adjoint from dx in the same pass
    (d = 1024 only) and return (dx, up_dy, up_dscale, up_dbias)."""
    b, n, d = x.shape
    dx = torch.empty_like(x)
    P = _lib.LnShiftBwdParams(batch=b, n=n, d=d, text_len=text_len, fmap=fmap, do_ln=int(do_ln), do_shift=int(do_shift),
                              dout_dtype=dt_code(d_out.dtype), d_out=_p(_c(d_out)), x=_p(_c(x)), mean=_p(mean), rstd=_p(rstd),
                              gamma=_p(gamma), dres=_p(dres), dx=_p(dx), dgamma=_p(dgamma), dbeta=_p(dbeta))
    res = None
    if up is not None:
        up_y, up_scale, up_sign = up
        assert d == 1024 and (up_y is None or (up_y.dtype == d_out.dtype and up_y.is_contiguous()))
        up_dy = torch.empty(b * n, d, device=x.device, dtype=d_out.dtype)
        acc = up_zeroed if up_zeroed is not None else torch.zeros(2, d, device=x.device, dtype=torch.float32)   # [2, d] fp32, pre-zeroed
        want_scale = up_scale is not None and up_y is not None
        P.up_y, P.up_scale, P.up_sign, P.up_dy = _p(up_y), _p(up_scale), up_sign, _p(up_dy)
        P.up_dscale, P.up_dbias = (_p(acc[0]) if want_scale else None), _p(acc[1])
        res = (up_dy, acc[0] if want_scale else None, acc[1])
    _lib.check(_lib.lib().dalle_b200_ln_shift_bwd(ctypes.byref(P), _stream()), 'ln_shift_bwd')
    _count()
    return dx if res is None else (dx,) + res


_gemm_events = None      # list of (start, end, flops, backend, shape-key) while gemm_timing is on


def gemm_timing(enable):
    """bench.py: bracket every GEMM launch with CUDA events on the launching stream.  gemm_timing(True) starts
    collecting; gemm_timing(False) synchronises and returns {'tcgen05': {flops, ms, launches}, 'simt': {...},
    'by_shape': {key: {ms, tflops, launches}}}."""
    global _gemm_events
    if enable:
        _gemm_events = []
        return None
    ev, _gemm_events = _gemm_events or [], None
    torch.cuda.synchronize()
    out = {'tcgen05': {'flops': 0.0, 'ms': 0.0, 'launches': 0}, 'simt': {'flops': 0.0, 'ms': 0.0, 'launches': 0},
           'smallm': {'flops': 0.0, 'ms': 0.0, 'launches': 0}, 'by_shape': {}}
    for s, e, flops, backend, key in ev:
        ms = s.elapsed_time(e)
        fam = out['tcgen05' if backend == _lib.GEMM_TCGEN05 else 'smallm' if backend == _lib.GEMM_SMALLM else 'simt']
        fam['flops'] += flops
        fam['ms'] += ms
        fam['launches'] += 1
        b = out['by_shape'].setdefault(key, {'ms': 0.0, 'flops': 0.0, 'launches': 0})
        b['ms'] += ms
        b['flops'] += flops
        b['launches'] += 1
    for b in out['by_shape'].values():
        b['tflops'] = b['flops'] / (b['ms'] * 1e-3) / 1e12 if b['ms'] > 0 else 0.0
        b['ms_per_launch'] = b['ms'] / b['launches']
        del b['flops']
    return out


_EPI_NAMES = {EPI_STORE: 'store', EPI_QKV: 'qkv', EPI_RESID: 'resid', EPI_GEGLU: 'geglu', EPI_GEGLU_BWD: 'geglu_bwd'}


def _gemm(P):
    if _gemm_events is None:
        _lib.check(_lib.lib().dalle_b200_gemm(ctypes.byref(P), _stream()), 'gemm')
        _count()
        return
    backend = _lib.lib().dalle_b200_gemm_select(ctypes.byref(P))
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    _lib.check(_lib.lib().dalle_b200_gemm(ctypes.byref(P), _stream()), 'gemm')
    e.record()
    _count()
    key = f"{_EPI_NAMES.get(P.epilogue, '?')}:{'M' if P.a_mn_major else 'K'}{'N' if P.b_mn_major else 'K'}:{P.M}x{P.N}x{P.K}"
    _gemm_events.append((s, e, 2.0 * P.M * P.N * P.K, backend, key))


SMALL_M = os.environ.get('DALLE_B200_SMALLM', '1') != '0'      # M <= 16 bf16 GEMMs (decoding) on the weight-streaming kernel
_small_m_rows = 16        # row limit of the rule below; small_m_rows() raises it for the duration of a block


@contextlib.contextmanager
def small_m_rows(rows):
    """Send bf16 GEMMs of up to `rows` (<= 32) rows to the weight-streaming kernel inside the block.  The guided decoder runs its
    step at batch 2b (conditional + unconditional stream) under small_m_rows(32); everywhere else the limit stays at 16."""
    global _small_m_rows
    assert 1 <= rows <= 32
    prev, _small_m_rows = _small_m_rows, rows
    try:
        yield
    finally:
        _small_m_rows = prev


def _small_m(A, N, a_mn=False, b_mn=False):
    """A [M, K] bf16 with M <= 16 (small_m_rows: up to 32): the problem db200_gemm_backend::DB200_GEMM_SMALLM covers
    (csrc/gemm_smallm.cu)."""
    return (SMALL_M and A.dtype == torch.bfloat16 and not a_mn and not b_mn and 1 <= A.shape[0] <= _small_m_rows and A.shape[1] % 256 == 0
            and N % 16 == 0)


def _base(M, N, K, A, lda, a_mn, B, ldb, b_mn, epilogue, backend=GEMM_AUTO):
    assert A.dtype == B.dtype
    return _lib.GemmParams(M=M, N=N, K=K, dtype=dt_code(A.dtype), backend=backend, A=_p(A), lda=lda, a_mn_major=int(a_mn),
                           B=_p(B), ldb=ldb, b_mn_major=int(b_mn), epilogue=epilogue)


# ------------------------------------------------------------------------------------------------
# fp32 parity mode on the tensor cores: "bf16x6"
# ------------------------------------------------------------------------------------------------
def split_bf16x3(x, operand, concat_rows):
    """fp32 [rows, cols] -> the six-fold K-concatenated bf16 operand of dalle_b200_split_bf16x3 (operand 0 = A, 1 = B)."""
    rows, cols = x.shape
    dst = torch.empty((6 * rows, cols) if concat_rows else (rows, 6 * cols), device=x.device, dtype=torch.bfloat16)
    _lib.check(_lib.lib().dalle_b200_split_bf16x3(_p(_c(x)), _p(dst), rows, cols, int(concat_rows), operand, _stream()), 'split_bf16x3')
    _count()
    return dst


def _gemm_x6(A, B, a_mn, b_mn, bias, out):
    """fp32 acc[M,N] = sum_k A(m,k) B(n,k) on gemm_tcgen05_kernel: both operands split into three bf16 pieces laid side by side
    along K (six partial products = one GEMM with K' = 6K, fp32 accumulation in tensor memory, fp32 STORE epilogue).
    Returns None if the shape does not qualify for the tcgen05 kernel (the caller then uses the CUDA-core kernel)."""
    if a_mn:
        K, M = A.shape
    else:
        M, K = A.shape
    N = B.shape[1] if b_mn else B.shape[0]
    if K % 8 or N % 8 or (a_mn and M % 8) or not (A.is_cuda and torch.cuda.get_device_capability(A.device)[0] == 10):
        return None
    A6 = split_bf16x3(A, 0, concat_rows=a_mn)
    B6 = split_bf16x3(B, 1, concat_rows=b_mn)
    P = _base(M, N, 6 * K, A6, A6.shape[1], a_mn, B6, B6.shape[1], b_mn, EPI_STORE, GEMM_AUTO)
    C = out if out is not None else torch.empty(M, N, device=A.device, dtype=torch.float32)
    P.C, P.ldc, P.c_dtype, P.bias, P.split_k_ok = _p(C), N, F32, _p(bias), 0
    if _lib.lib().dalle_b200_gemm_select(ctypes.byref(P)) != _lib.GEMM_TCGEN05:
        return None
    _gemm(P)
    return C


def _use_x6(A):
    return A.dtype == torch.float32 and config.fp32_gemm() == 'bf16x6'


def resid_scale(y, resid, scale, sign):
    """resid + sign * scale (.) y  -> fp32 [M, d]   (y fp32 or bf16)"""
    M, d = y.shape
    out = torch.empty(M, d, device=y.device, dtype=torch.float32)
    _lib.check(_lib.lib().dalle_b200_resid_scale(_p(_c(y)), dt_code(y.dtype), _p(resid), _p(scale), sign, _p(out), M, d, _stream()), 'resid_scale')
    _count()
    return out


def sample_topk_gumbel(logits, thres=0.5, temperature=1.0, seed=0, offset=0, gumbel=None):
    """logits [B, V] -> int64 [B]: top_k(logits, thres) + gumbel_sample(., temperature) of dalle_pytorch.py:43-58 in one launch."""
    B, V = logits.shape
    assert logits.stride(1) == 1
    k = max(int((1 - thres) * V), 1)
    out = torch.empty(B, device=logits.device, dtype=torch.int64)
    _lib.check(_lib.lib().dalle_b200_sample_topk_gumbel(_p(logits), dt_code(logits.dtype), B, V, logits.stride(0), k, float(temperature), _p(gumbel),
                                                        int(seed) & (2 ** 64 - 1), int(offset), _p(out), _stream()), 'sample_topk_gumbel')
    _count()
    return out


def sample_guided_topk_gumbel(logits, cond_scale, thres=0.5, temperature=1.0, seed=0, offset=0, gumbel=None):
    """logits [2b, V] = conditional rows [:b] then unconditional rows [b:] -> int64 [b]: sample_topk_gumbel of the guided logits
    null + (cond - null) * cond_scale (forward_with_cond_scale, dalle_pytorch.py:564-574), which the kernel forms row by row
    without writing them.  Same (seed, offset) (or `gumbel` [b, V]) -> the same tokens as torch's guided logits through
    sample_topk_gumbel."""
    B2, V = logits.shape
    assert B2 % 2 == 0 and logits.stride(1) == 1
    b = B2 // 2
    k = max(int((1 - thres) * V), 1)
    out = torch.empty(b, device=logits.device, dtype=torch.int64)
    if gumbel is not None:
        assert gumbel.shape == (b, V) and gumbel.dtype == torch.float32 and gumbel.is_contiguous()
    _lib.check(_lib.lib().dalle_b200_sample_guided_topk_gumbel(_p(logits[:b]), _p(logits[b:]), dt_code(logits.dtype), b, V, logits.stride(0),
                                                               float(cond_scale), k, float(temperature), _p(gumbel), int(seed) & (2 ** 64 - 1),
                                                               int(offset), _p(out), _stream()), 'sample_guided_topk_gumbel')
    _count()
    return out


def decode_shift(h, ring_top, ring_left, pos_t, text_len, fmap, out_dtype):
    """One decoding step of PreShiftToken (include/dalle_b200.h): h [b,d] fp32 (normalised token), rings fp32 [fmap,b,d/4] /
    [fmap,b,d/2-d/4], pos_t int64 [1] on the device -> y [b,d] out_dtype; the rings are updated in place."""
    b, d = h.shape
    assert h.dtype == torch.float32 and ring_top.dtype == torch.float32 and ring_left.dtype == torch.float32 and pos_t.dtype == torch.int64
    assert ring_top.shape == (fmap, b, d // 4) and ring_left.shape == (fmap, b, d // 2 - d // 4) and d % 4 == 0
    y = torch.empty(b, d, device=h.device, dtype=out_dtype)
    _lib.check(_lib.lib().dalle_b200_decode_shift(_p(_c(h)), _p(y), dt_code(out_dtype), b, d, _p(_c(ring_top)), _p(_c(ring_left)), _p(pos_t),
                                                  int(text_len), int(fmap), _stream()), 'decode_shift')
    _count()
    return y


def decode_kv_append(k_new, v_new, k_cache, v_cache, pos_t):
    """k_new, v_new [b,h,1,dh] -> row pos_t (int64 [1] on the device) of the in-place caches [b,h,rows,dh]."""
    b, h, one, dh = k_new.shape
    assert one == 1 and v_new.shape == k_new.shape and k_cache.shape == v_cache.shape and k_cache.shape[:2] == (b, h) and k_cache.shape[3] == dh
    assert k_new.dtype == v_new.dtype == k_cache.dtype == v_cache.dtype and pos_t.dtype == torch.int64
    _lib.check(_lib.lib().dalle_b200_decode_kv_append(_p(_c(k_new)), _p(_c(v_new)), _p(_c(k_cache)), _p(_c(v_cache)), dt_code(k_cache.dtype), b * h, dh,
                                                      k_cache.shape[2], _p(pos_t), _stream()), 'decode_kv_append')
    _count()


def dropout_(x, p, seed, offset):
    """In place: x[i] <- keep(i) ? x[i] / (1 - p) : 0 with the Philox mask of (seed, offset) (include/dalle_b200.h)."""
    _lib.check(_lib.lib().dalle_b200_dropout(_p(_c(x)), _p(x), dt_code(x.dtype), x.numel(), float(p), int(seed) & (2 ** 64 - 1), int(offset), _stream()),
               'dropout')
    _count()
    return x


def geglu_fwd(u):
    """fp32 u = [a | g] [M, 2H] -> a * gelu_erf(g) [M, H]"""
    M, H2 = u.shape
    h = torch.empty(M, H2 // 2, device=u.device, dtype=torch.float32)
    _lib.check(_lib.lib().dalle_b200_geglu_fwd(_p(_c(u)), _p(h), M, H2 // 2, _stream()), 'geglu_fwd')
    _count()
    return h


def gemm_store(A, B, a_mn=False, b_mn=False, out_dtype=None, bias=None, backend=GEMM_AUTO, out=None):
    """acc[M,N] = sum_k A(m,k) B(n,k).  A: [M,K] (a_mn=False) or [K,M] (a_mn=True); B: [N,K] or [K,N].
    `out` (optional, contiguous [M,N]) receives the result instead of a fresh tensor."""
    _c(A), _c(B)
    if backend == GEMM_AUTO and _use_x6(A) and (out is None or out.dtype == torch.float32) and out_dtype in (None, torch.float32):
        C6 = _gemm_x6(A, B, a_mn, b_mn, bias, out)
        if C6 is not None:
            return C6
    if a_mn:
        K, M = A.shape
    else:
        M, K = A.shape
    if b_mn:
        Kb, N = B.shape
    else:
        N, Kb = B.shape
    assert K == Kb, (A.shape, B.shape, a_mn, b_mn)
    if out is not None:
        assert out.shape == (M, N) and out.is_contiguous()
        C, out_dtype = out, out.dtype
    else:
        out_dtype = out_dtype or A.dtype
        C = None
    # weight-gradient shapes (few output tiles, very long K): let the kernel split K; it needs a zeroed fp32 C
    split_ok = out_dtype == torch.float32 and bias is None and A.dtype == torch.bfloat16 and M * N <= 4096 * 1024 and K >= 4096
    mc = getattr(out, '_b200_mc', None) if out is not None else None      # (multicast address, scale): data-parallel multimem slot
    if backend == GEMM_AUTO and mc is None and _small_m(A, N, a_mn, b_mn):
        backend, split_ok = _lib.GEMM_SMALLM, False
    if C is None:
        C = (torch.zeros if split_ok else torch.empty)(M, N, device=A.device, dtype=out_dtype)
    elif split_ok and mc is None:
        C.zero_()
    P = _base(M, N, K, A, A.shape[1], a_mn, B, B.shape[1], b_mn, EPI_STORE, backend)
    P.C, P.ldc, P.c_dtype, P.bias, P.split_k_ok = _p(C), N, dt_code(out_dtype), _p(bias), int(split_ok)
    if mc is not None:      # the epilogue ADDS scale * acc into every GPU's replica of the (pre-zeroed) flat gradient buffer
        assert out_dtype == torch.float32 and bias is None
        P.C_multicast, P.c_scale = ctypes.c_void_p(mc[0]), mc[1]
    _gemm(P)
    return C


def gemm_qkv(A, W, batch, seq_n, heads, dim_head, cos_t, sin_t, q_scale, pos_offset=0, backend=GEMM_AUTO):
    """A [batch*seq_n, d], W [3*heads*dim_head, d] -> q,k,v [batch, heads, seq_n, dim_head] (rotary + q scale fused)"""
    _c(A), _c(W)
    M, K = A.shape
    N = W.shape[0]
    if backend == GEMM_AUTO and _use_x6(A) and dim_head % 8 == 0:
        raw = _gemm_x6(A, W, False, False, None, None)           # plain product on the tensor cores, then the streaming head split
        if raw is not None:
            qkv = torch.empty(3, batch, heads, seq_n, dim_head, device=A.device, dtype=A.dtype)
            _lib.check(_lib.lib().dalle_b200_qkv_rotary(_p(raw), _p(qkv[0]), _p(qkv[1]), _p(qkv[2]), _p(cos_t), _p(sin_t), F32, M, seq_n, heads,
                                                        dim_head, pos_offset, q_scale, seq_n, _stream()), 'qkv_rotary')
            _count()
            return qkv[0], qkv[1], qkv[2]
    if backend == GEMM_AUTO and _small_m(A, N) and dim_head % 8 == 0:
        return gemm_qkv_auto(A, W, batch, seq_n, heads, dim_head, cos_t, sin_t, q_scale, pos_offset, n_alloc=seq_n)   # small-M product + head split
    qkv = torch.empty(3, batch, heads, seq_n, dim_head, device=A.device, dtype=A.dtype)
    P = _base(M, N, K, A, K, False, W, K, False, EPI_QKV, backend)
    P.q, P.k, P.v = _p(qkv[0]), _p(qkv[1]), _p(qkv[2])
    P.cos_t, P.sin_t = _p(cos_t), _p(sin_t)
    P.seq_n, P.heads, P.dim_head, P.pos_offset, P.q_scale = seq_n, heads, dim_head, pos_offset, q_scale
    _gemm(P)
    return qkv[0], qkv[1], qkv[2]


FUSE_QKV_EPILOGUE = False   # True: rotary + head split inside the GEMM epilogue (EPI_QKV); False (measured faster for bf16 on
#                             B200): plain GEMM + dalle_b200_qkv_rotary streaming pass


def gemm_qkv_auto(A, W, batch, seq_n, heads, dim_head, cos_t, sin_t, q_scale, pos_offset=0, n_alloc=None):
    """n_alloc (gathered axial layout, see GatherLayout): rows per (batch, head) of the returned q/k/v, rows >= seq_n zero."""
    if n_alloc is None and (FUSE_QKV_EPILOGUE or A.dtype != torch.bfloat16 or dim_head % 8):
        return gemm_qkv(A, W, batch, seq_n, heads, dim_head, cos_t, sin_t, q_scale, pos_offset)
    raw = gemm_store(A, W)                                      # [M, 3*h*dh]
    M = raw.shape[0]
    rows = n_alloc or seq_n
    qkv = torch.empty(3, batch, heads, rows, dim_head, device=A.device, dtype=A.dtype)
    _lib.check(_lib.lib().dalle_b200_qkv_rotary(_p(raw), _p(qkv[0]), _p(qkv[1]), _p(qkv[2]), _p(cos_t), _p(sin_t), dt_code(A.dtype), M, seq_n,
                                                heads, dim_head, pos_offset, q_scale, rows, _stream()), 'qkv_rotary')
    _count()
    return qkv[0], qkv[1], qkv[2]


def gemm_resid(A, W, bias, resid, scale, sign=1.0, keep_y=False, backend=GEMM_AUTO):
    """out[M,N] fp32 = resid + sign*scale*(A W^T + bias); optionally also returns y = A W^T + bias (A.dtype)"""
    _c(A), _c(W)
    M, K = A.shape
    N = W.shape[0]
    if backend == GEMM_AUTO and _use_x6(A):
        y6 = _gemm_x6(A, W, False, False, bias, None)            # y = A W^T + bias
        if y6 is not None:
            return resid_scale(y6, resid, scale, sign), (y6 if keep_y else None)
    out = torch.empty(M, N, device=A.device, dtype=torch.float32)
    y = torch.empty(M, N, device=A.device, dtype=A.dtype) if keep_y else None
    if backend == GEMM_AUTO and _small_m(A, N):
        backend = _lib.GEMM_SMALLM
    P = _base(M, N, K, A, K, False, W, K, False, EPI_RESID, backend)
    P.bias, P.resid, P.scale, P.sign, P.y_out, P.out = _p(bias), _p(resid), _p(scale), sign, _p(y), _p(out)
    _gemm(P)
    return out, y


def gemm_geglu(A, W1, b1, keep_u=True, backend=GEMM_AUTO):
    """A [M,d], W1 [2H,d], b1 [2H] -> (h [M,H], u [M,2H] or None)"""
    _c(A), _c(W1)
    M, K = A.shape
    N = W1.shape[0]
    H = N // 2
    if backend == GEMM_AUTO and _use_x6(A):
        u6 = _gemm_x6(A, W1, False, False, b1, None)             # u = A W1^T + b1
        if u6 is not None:
            return geglu_fwd(u6), (u6 if keep_u else None)
    h = torch.empty(M, H, device=A.device, dtype=A.dtype)
    u = torch.empty(M, N, device=A.device, dtype=A.dtype) if keep_u else None
    if backend == GEMM_AUTO and _small_m(A, N):
        backend = _lib.GEMM_SMALLM
    P = _base(M, N, K, A, K, False, W1, K, False, EPI_GEGLU, backend)
    P.bias, P.u_out, P.h_out, P.hidden = _p(b1), _p(u), _p(h), H
    _gemm(P)
    return h, u


def gemm_geglu_bwd(dy, W2, u, backend=GEMM_AUTO):
    """dy [M,d], W2 [d,H] (read N-major), u [M,2H] -> du [M,2H]"""
    _c(dy), _c(W2), _c(u)
    M, K = dy.shape
    H = W2.shape[1]
    du = torch.empty_like(u)
    P = _base(M, H, K, dy, K, False, W2, H, True, EPI_GEGLU_BWD, backend)
    P.u_in, P.du_out, P.hidden = _p(u), _p(du), H
    _gemm(P)
    return du


# ------------------------------------------------------------------------------------------------
class AttnSpec:
    """Geometry + pattern of one attention layer (maps the reference's attention classes onto db200_attn_pattern)."""

    def __init__(self, pattern=ATTN_FULL, causal=True, stable=False, text_len=0, fmap=0, kernel_size=0, dilation=1,
                 static_mask=None):
        self.pattern, self.causal, self.stable = pattern, causal, stable
        self.text_len, self.fmap, self.kernel_size, self.dilation = text_len, fmap, kernel_size, dilation
        self.static_mask = static_mask      # uint8 [n, n] on device or None


class GatherLayout:
    """Tensor layout of the gathered axial attention kernels (include/dalle_b200.h, db200_attn_fwd_params::gather):
    q/k/v carry n_alloc = text_len + fmap^2 rows per (batch, head) (the reference's zero pad token, attention.py:255-258, is
    materialised as a zero row), lse/delta n_stat entries; for axis 1 the gradient of the attention output needs one spare row."""
    __slots__ = ('n', 'n_alloc', 'n_stat', 'col', 'pad_dout')

    def __init__(self, spec, n):
        T, fm = spec.text_len, spec.fmap
        self.n, self.n_alloc, self.n_stat = n, T + fm * fm, (T + 63) // 64 * 64 + fm * fm
        self.col = spec.pattern == ATTN_AXIAL_COL
        self.pad_dout = self.col and n < T + fm * fm


GATHER_AXIAL = os.environ.get('DALLE_B200_AXIAL_GATHER', '1') != '0'    # 0: axial patterns run the dense-tile predicate kernels


def gather_layout(spec, dtype, n, dim_head=64, key_mask=None):
    """The gathered layout if axial attention of this shape can use it (bf16 tensor-core path, whole image), else None."""
    if not GATHER_AXIAL or spec is None or spec.pattern not in (ATTN_AXIAL_ROW, ATTN_AXIAL_COL):
        return None
    if dtype != torch.bfloat16 or dim_head != 64 or key_mask is not None:
        return None
    if os.environ.get('DALLE_B200_ATTN', 'tc') != 'tc' or spec.fmap not in (16, 32, 64):
        return None
    full = spec.text_len + spec.fmap * spec.fmap
    if n not in (full - 1, full):
        return None
    return GatherLayout(spec, n)


def _attn_params(spec, q, k, v, out, lse, key_mask, lay=None, n_k=None):
    b, h, n_q, dh = q.shape
    kv_rows = 0
    if n_k is not None:                 # in-place KV cache: k, v are [b, h, capacity, dh] buffers, the first n_k rows valid
        kv_rows, n_k = k.shape[2], int(n_k)
        assert n_k <= kv_rows
    else:
        n_k = k.shape[2]
    if lay is not None:
        assert n_q == n_k == lay.n_alloc, 'gathered layout: q/k/v must carry n_alloc rows per head'
        n_q = n_k = lay.n
    sm = spec.static_mask
    return _lib.AttnFwdParams(batch=b, heads=h, n_q=n_q, n_k=n_k, dim_head=dh, dtype=dt_code(q.dtype), pattern=spec.pattern,
                              causal=int(spec.causal), stable=int(spec.stable), text_len=spec.text_len, fmap=spec.fmap,
                              kernel_size=spec.kernel_size, dilation=spec.dilation, gather=int(lay is not None), kv_rows=kv_rows,
                              key_mask=_p(key_mask),
                              static_mask=_p(sm), static_ld=(sm.shape[1] if sm is not None else 0),
                              q=_p(_c(q)), k=_p(_c(k)), v=_p(_c(v)), out=_p(out), lse=_p(lse))


def attn_fwd(spec, q, k, v, key_mask=None, lay=None, n_k=None):
    """q [b,h,n_q,64], k,v [b,h,n_k,64] -> out [b,n_q,h*64], lse [b,h,n_q]
    (lay = GatherLayout: q,k,v [b,h,n_alloc,64] -> out [b,n,h*64], lse [b,h,n_stat];
     n_k = valid rows of k, v when they are [b,h,capacity,64] in-place KV-cache buffers)"""
    b, h, n_q, dh = q.shape
    if lay is not None:
        n_q = lay.n
    out = torch.empty(b, n_q, h * dh, device=q.device, dtype=q.dtype)
    lse = torch.empty(b, h, lay.n_stat if lay is not None else n_q, device=q.device, dtype=torch.float32)
    P = _attn_params(spec, q, k, v, out, lse, key_mask, lay, n_k)
    _lib.check(_lib.lib().dalle_b200_attn_fwd(ctypes.byref(P), _stream()), 'attn_fwd')
    _count()
    return out, lse


def attn_dout_buffer(lay, rows, inner, device, dtype):
    """[rows, inner] destination for the gradient of the attention output; with the column gather the buffer carries the spare
    row the strided box of the last batch reaches (the library zeroes it)."""
    if lay is not None and lay.pad_dout:
        return torch.empty(rows + 1, inner, device=device, dtype=dtype)[:rows]
    return torch.empty(rows, inner, device=device, dtype=dtype)


def attn_bwd(spec, q, k, v, out, lse, d_out, cos_t, sin_t, q_scale, key_mask=None, lay=None):
    """-> dqkv [b*n, 3*h*64] : gradient w.r.t. the to_qkv output (rotary adjoint and q scale folded in).
    With a GatherLayout whose pad_dout is set, d_out must come from attn_dout_buffer()."""
    b, h, n, dh = q.shape
    if lay is not None:
        n = lay.n
        if lay.pad_dout:
            assert d_out.untyped_storage().nbytes() - d_out.storage_offset() * d_out.element_size() >= (b * n + 1) * h * dh * d_out.element_size(), \
                'column gather: d_out needs one spare row (ops.attn_dout_buffer)'
    dqkv = torch.empty(b * n, 3 * h * dh, device=q.device, dtype=q.dtype)
    delta = torch.empty(b, h, lay.n_stat if lay is not None else n, device=q.device, dtype=torch.float32)
    P = _lib.AttnBwdParams(f=_attn_params(spec, q, k, v, out, lse, key_mask, lay), d_out=_p(_c(d_out)), cos_t=_p(cos_t), sin_t=_p(sin_t),
                           q_scale=q_scale, delta=_p(delta), dqkv=_p(dqkv))
    _lib.check(_lib.lib().dalle_b200_attn_bwd(ctypes.byref(P), _stream()), 'attn_bwd')
    _count(3)
    return dqkv


# ------------------------------------------------------------------------------------------------
def scale_bwd(d_out, y, scale, sign, dtype, want_dscale=True, want_dbias=True, zeroed=None):
    """d_out [M,d] fp32 -> dy [M,d] dtype, dscale [d] fp32 | None, dbias [d] fp32 | None.
    `zeroed` (optional) = (dscale_buf, dbias_buf): pre-zeroed fp32 [d] accumulators (callers carve them out of one pooled
    torch.zeros per sub-layer instead of launching a fill per gradient)."""
    M, d = d_out.shape
    dy = torch.empty(M, d, device=d_out.device, dtype=dtype)
    if zeroed is not None:
        dscale = zeroed[0] if (want_dscale and scale is not None) else None
        dbias = zeroed[1] if want_dbias else None
    else:
        dscale = torch.zeros(d, device=d_out.device, dtype=torch.float32) if (want_dscale and scale is not None) else None
        dbias = torch.zeros(d, device=d_out.device, dtype=torch.float32) if want_dbias else None
    P = _lib.ScaleBwdParams(rows=M, d=d, dtype=dt_code(dtype), sign=sign, d_out=_p(_c(d_out)), y=_p(y), scale=_p(scale), dy=_p(dy),
                            dscale=_p(dscale), dbias=_p(dbias))
    _lib.check(_lib.lib().dalle_b200_scale_bwd(ctypes.byref(P), _stream()), 'scale_bwd')
    _count()
    return dy, dscale, dbias


def geglu_bwd(dh, u, want_dbias=True, zeroed=None):
    """dh [M,H], u [M,2H] -> (du [M,2H], db1 [2H] fp32 | None): streaming GEGLU adjoint + bias gradient in one pass.
    `zeroed`: optional pre-zeroed fp32 [2H] accumulator for the bias gradient."""
    M, H = dh.shape
    du = torch.empty_like(u)
    db = (zeroed if zeroed is not None else torch.zeros(2 * H, device=dh.device, dtype=torch.float32)) if want_dbias else None
    _lib.check(_lib.lib().dalle_b200_geglu_bwd(_p(_c(dh)), _p(_c(u)), _p(du), _p(db), dt_code(dh.dtype), M, H, _stream()), 'geglu_bwd')
    _count()
    return du, db


def ce_fwd(logits, labels, coef, loss_acc):
    """logits [R,V], labels [R] int64; loss_acc (fp32 scalar tensor) += coef * sum(CE rows).  Returns row_lse [R]."""
    R, V = logits.shape
    lse = torch.empty(R, device=logits.device, dtype=torch.float32)
    _lib.check(_lib.lib().dalle_b200_ce_fwd(_p(_c(logits)), dt_code(logits.dtype), R, V, _p(_c(labels)), coef, _p(lse), _p(loss_acc), _stream()), 'ce_fwd')
    _count()
    return lse


def ce_bwd_(logits, labels, coef, row_lse, upstream):
    """In place: logits <- upstream * coef * (softmax(logits) - onehot(labels)) (the gradient w.r.t. the logits)."""
    R, V = logits.shape
    _lib.check(_lib.lib().dalle_b200_ce_bwd(_p(_c(logits)), dt_code(logits.dtype), R, V, _p(_c(labels)), coef, _p(row_lse), _p(upstream), _stream()), 'ce_bwd')
    _count()
    return logits


def colsum(x):
    rows, cols = x.shape
    out = torch.zeros(cols, device=x.device, dtype=torch.float32)
    _lib.check(_lib.lib().dalle_b200_colsum(_p(_c(x)), dt_code(x.dtype), rows, cols, _p(out), _stream()), 'colsum')
    _count()
    return out


def mc_add(src, mc_ptr, scale):
    """every replica of the symmetric buffer at multicast address mc_ptr += scale * src (fp32, flat)"""
    src = _c(src)
    assert src.dtype == torch.float32
    _lib.check(_lib.lib().dalle_b200_mc_add(_p(src), ctypes.c_void_p(mc_ptr), src.numel(), scale, _stream()), 'mc_add')
    _count()


def cast_bf16(src):
    src = _c(src)
    assert src.dtype == torch.float32
    dst = torch.empty(src.shape, device=src.device, dtype=torch.bfloat16)
    _lib.check(_lib.lib().dalle_b200_cast_bf16(_p(src), _p(dst), src.numel(), _stream()), 'cast_bf16')
    _count()
    return dst


def embed_fwd(ids, weight, out, seg_off):
    """out[b, seg_off + l, :] = weight[ids[b, l], :]   (ids [B, L] int64, out [B, n, d] fp32 contiguous, written in place)"""
    B, L = ids.shape
    _, n, d = out.shape
    _lib.check(_lib.lib().dalle_b200_embed_fwd(_p(_c(ids)), _p(_c(weight)), _p(out), B, L, n, seg_off, d, weight.shape[0], _stream()), 'embed_fwd')
    _count()


def embed_bwd(ids, d_out, dweight, seg_off):
    """dweight[ids[b, l], :] += d_out[b, seg_off + l, :]   (fp32 atomics)"""
    B, L = ids.shape
    _, n, d = d_out.shape
    _lib.check(_lib.lib().dalle_b200_embed_bwd(_p(_c(ids)), _p(_c(d_out)), _p(dweight), B, L, n, seg_off, d, dweight.shape[0], _stream()), 'embed_bwd')
    _count()


def sumsq_(x, out):
    """out (fp32 device scalar) += sum(x^2) over a flat fp32 tensor"""
    _lib.check(_lib.lib().dalle_b200_sumsq(_p(_c(x)), x.numel(), _p(out), _stream()), 'sumsq')
    _count()


def adam_(p, g, m, v, step, lr, beta1, beta2, eps, weight_decay=0.0, max_norm=0.0, gnorm_sq=None):
    """In-place Adam update of the flat fp32 buffers p, m, v from g (see include/dalle_b200.h::dalle_b200_adam)."""
    for t in (p, g, m, v):
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.numel() == p.numel()
    P = _lib.AdamParams(p=_p(p), g=_p(g), m=_p(m), v=_p(v), count=p.numel(), lr=lr, beta1=beta1, beta2=beta2, eps=eps,
                        weight_decay=weight_decay, step=step, max_norm=max_norm, gnorm_sq=_p(gnorm_sq))
    _lib.check(_lib.lib().dalle_b200_adam(ctypes.byref(P), _stream()), 'adam')
    _count()


def axpby(a, b, alpha):
    """a + alpha * b over fp32 tensors of equal shape"""
    _c(a), _c(b)
    y = torch.empty_like(a)
    _lib.check(_lib.lib().dalle_b200_axpby(_p(a), _p(b), alpha, _p(y), a.numel(), _stream()), 'axpby')
    _count()
    return y
