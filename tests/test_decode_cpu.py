"""Host logic of the graph-replayed decoding path (dalle_pytorch_b200/decode.py) without a GPU.

The device-indexed step differs from the host-indexed cached step only in HOW the position reaches the kernels (device index
operations instead of host integers).  That glue is plain torch, so it is checked here on the CPU with the five library calls of a
cached step replaced by torch expressions of the same contract (the stubs below are test scaffolding, not a product path): both
forms of the step must then produce the same logits at every position.  The kernels themselves, the capture and the replay are
covered by tests/test_parity_gpu.py::test_generate_images_graph_replay.
"""
from collections import deque

import pytest
import torch
import torch.nn.functional as F

import dalle_pytorch_b200 as D
from dalle_pytorch_b200 import ops, decode, functional
from dalle_pytorch_b200.transformer import PreShiftToken

NEG = -torch.finfo(torch.float32).max


def _ln_shift_fwd(x, gamma, beta, out_dtype, text_len, fmap, do_ln=True, do_shift=True, eps=1e-5):
    assert not do_shift
    b, n, d = x.shape
    out = F.layer_norm(x, (d,), gamma, beta, eps) if do_ln else x
    return out.reshape(b * n, d).to(out_dtype), None, None


def _gemm_qkv(A, W, batch, seq_n, heads, dim_head, cos_t, sin_t, q_scale, pos_offset=0, backend=None):
    qkv = (A @ W.t()).view(batch, seq_n, 3, heads, dim_head).permute(2, 0, 3, 1, 4)             # [3, b, h, n, dh]
    c = cos_t[pos_offset:pos_offset + seq_n][None, None, None]
    s = sin_t[pos_offset:pos_offset + seq_n][None, None, None]
    x0, x1 = qkv[..., 0::2], qkv[..., 1::2]
    rot = torch.stack((x0 * c - x1 * s, x1 * c + x0 * s), dim=-1).flatten(-2)
    return (rot[0] * q_scale).contiguous(), rot[1].contiguous(), rot[2].contiguous()


def _attn_fwd(spec, q, k, v, key_mask=None, lay=None, n_k=None):
    b, h, n_q, dh = q.shape
    n_k = k.shape[2] if n_k is None else n_k
    k, v = k[:, :, :n_k], v[:, :, :n_k]
    s = q @ k.transpose(-1, -2)
    i = torch.arange(n_q)[:, None] + (n_k - n_q)
    j = torch.arange(n_k)[None, :]
    ok = torch.ones(n_q, n_k, dtype=torch.bool)
    if spec.causal:
        ok &= j <= i
    if spec.static_mask is not None:
        ok &= spec.static_mask[n_k - n_q:n_k, :n_k].bool()
    s = s.masked_fill(~ok, NEG)
    if key_mask is not None:
        assert key_mask.shape == (b, n_k) and key_mask.dtype == torch.uint8 and key_mask.is_contiguous()
        s = s.masked_fill(~key_mask.bool()[:, None, None, :], NEG)
    p = s.softmax(dim=-1)
    return (p @ v).transpose(1, 2).reshape(b, n_q, h * dh), None


def _gemm_resid(A, W, bias, resid, scale, sign=1.0, keep_y=False, backend=None):
    y = A @ W.t() + bias
    out = sign * y if scale is None else sign * scale * y
    return (out if resid is None else resid + out), (y if keep_y else None)


def _gemm_geglu(A, W1, b1, keep_u=True, backend=None):
    u = A @ W1.t() + b1
    H = u.shape[1] // 2
    return u[:, :H] * F.gelu(u[:, H:]), (u if keep_u else None)


def _decode_shift(h, ring_top, ring_left, pos_t, text_len, fmap, out_dtype):
    slot = (int(pos_t) - text_len) % fmap
    prev = (slot + fmap - 1) % fmap
    q, half = h.shape[1] // 4, h.shape[1] // 2
    y = h.clone()
    y[:, :q] = ring_top[slot]
    y[:, q:half] = ring_left[prev] if slot != 0 else 0.
    ring_top[slot] = h[:, :q]
    ring_left[slot] = h[:, q:half]
    return y.to(out_dtype)


def _decode_kv_append(k_new, v_new, k_cache, v_cache, pos_t):
    k_cache[:, :, int(pos_t)] = k_new[:, :, 0]
    v_cache[:, :, int(pos_t)] = v_new[:, :, 0]


@pytest.fixture
def cpu_kernels(monkeypatch):
    monkeypatch.setattr(ops, 'decode_shift', _decode_shift)
    monkeypatch.setattr(ops, 'decode_kv_append', _decode_kv_append)
    monkeypatch.setattr(ops, 'ln_shift_fwd', _ln_shift_fwd)
    monkeypatch.setattr(ops, 'gemm_qkv', _gemm_qkv)
    monkeypatch.setattr(ops, 'attn_fwd', _attn_fwd)
    monkeypatch.setattr(ops, 'gemm_resid', _gemm_resid)
    monkeypatch.setattr(ops, 'gemm_geglu', _gemm_geglu)
    monkeypatch.setattr(decode, 'WARMUP_STEPS', 10 ** 9)            # never capture: every step runs the device-indexed code eagerly
    with D.compute_dtype_ctx(torch.float32):                         # restores the caller's mode: later tests rely on the fp32 default
        yield


def _model(attn_types=('full',), shift_tokens=True, stable=False, optimize=False, depth=2, sandwich=False):
    torch.manual_seed(0)
    vae = D.TokenVAE(image_size=32, num_layers=3, num_tokens=24)         # fmap 4
    m = D.DALLE(dim=32, vae=vae, num_text_tokens=30, text_seq_len=6, depth=depth, heads=2, dim_head=16, attn_types=attn_types,
                shift_tokens=shift_tokens, stable=stable, optimize_for_inference=optimize, sandwich_norm=sandwich)
    for p in m.parameters():                                             # LayerScale starts at 0.1: make every branch matter
        if p.dim() == 3:
            torch.nn.init.uniform_(p, 0.5, 1.0)
    return m.eval()


@pytest.mark.parametrize('flat,bucket', [(False, 0), (True, 0), (False, 4), (True, 8)])
@pytest.mark.parametrize('name,kw', [
    ('full_shift', dict()),
    ('full_noshift', dict(shift_tokens=False)),
    ('axial_static_masks', dict(attn_types=('axial_row', 'axial_col'), optimize=True, depth=3)),
    ('stable', dict(stable=True)),
    ('sandwich_norm', dict(sandwich=True)),                     # not covered by the flat step: the captured step walks the module nest
])
def test_device_indexed_step_equals_host_indexed_step(cpu_kernels, monkeypatch, name, kw, flat, bucket):
    """flat = GraphedDecoder walks the layers itself (decode kernels + fused LayerScale/residual epilogue) instead of the module
    nest; bucket = attention reads only the first roundup(position + 1, bucket) cache rows."""
    monkeypatch.setattr(decode, 'FLAT_DEFAULT', flat)
    monkeypatch.setattr(decode, 'BUCKET_DEFAULT', bucket)
    m = _model(**kw)
    T, n_img = m.text_seq_len, m.image_seq_len
    g = torch.Generator().manual_seed(1)
    text = torch.randint(1, 30, (2, T), generator=g)
    img = torch.randint(0, 24, (2, n_img), generator=g)
    assert decode._attention_layers(m) is not None
    with torch.no_grad():
        host, dev = {}, {}
        want = [m(text, img[:, :k], cache=host)[:, -1] for k in range(n_img)]            # host-indexed: one forward per position
        got = [m(text, img[:, :0], cache=dev)[:, -1]]
        dec = decode.GraphedDecoder(m, dev)
        assert (dec.plan is not None) == (flat and not kw.get('sandwich', False))
        if kw.get('shift_tokens', True):
            assert any(isinstance(v, decode.ShiftRing) for v in dev.values()) and not any(isinstance(v, deque) for v in dev.values())
        for k in range(1, n_img):
            got.append(dec.step(img[:, k - 1]).clone())
    assert dev['offset'] == host['offset'] == T + n_img and int(dec.pos_t) == T + n_img
    if bucket:
        assert dec.n_k == min(dec.cap, -(-(T + n_img) // bucket) * bucket)               # the last token sees T + n_img keys
    for k, (a, b) in enumerate(zip(want, got)):
        assert a.shape == b.shape
        live = a > NEG / 2
        assert torch.equal(live, b > NEG / 2), (name, k)                                 # same logits mask
        assert torch.allclose(a[live], b[live], rtol=1e-5, atol=1e-6), (name, k, float((a[live] - b[live]).abs().max()))


def test_generate_images_takes_the_device_indexed_path_and_keeps_the_tokens(cpu_kernels, monkeypatch):
    m = _model(attn_types=('axial_row', 'axial_col'), optimize=True)
    real_eligible = decode.eligible
    monkeypatch.setattr(decode, 'eligible', lambda model, text, cond_scale: cond_scale == 1 and decode._attention_layers(model) is not None)
    text = torch.randint(1, 30, (2, m.text_seq_len), generator=torch.Generator().manual_seed(2))
    made = []
    real = decode.GraphedDecoder

    class Spy(real):
        def __init__(self, *a, **k):
            made.append(self)
            super().__init__(*a, **k)
    monkeypatch.setattr(decode, 'GraphedDecoder', Spy)
    toks = {}
    for on in (False, True):
        monkeypatch.setattr(decode, 'GRAPH_DEFAULT', on)
        torch.manual_seed(7)
        toks[on] = m.generate_images(text, use_cache=True, filter_thres=0.8)
    assert len(made) == 1                                                                # only the second call used the decoder
    assert toks[True].shape == (2, m.image_seq_len) and torch.equal(toks[False], toks[True])
    # guidance (cond_scale != 1) and models whose layers re-run the prefix keep the host-indexed loop
    monkeypatch.setattr(decode, 'GRAPH_DEFAULT', True)
    m.generate_images(text, use_cache=True, cond_scale=2.0)
    assert len(made) == 1
    assert decode._attention_layers(_model(attn_types=('axial_row',))) is None           # SparseAxialCausalAttention is NonCached
    assert not real_eligible(m, text, 1.0)                                             # (real check: CPU tensors are not eligible)


def test_allow_table_and_shift_ring_against_brute_force():
    sm = torch.rand(12, 12, generator=torch.Generator().manual_seed(3)) > 0.5
    t = decode.allow_table(sm, 13, 14, 'cpu')
    for p in range(13):
        for j in range(14):
            assert bool(t[p, j]) == (j <= p and p < 12 and j < 12 and bool(sm[p, j]))
    assert torch.equal(decode.allow_table(None, 5, 5, 'cpu').bool(), torch.ones(5, 5).tril().bool())

    class Rec(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.seen = []

        def forward(self, x, cache=None, **kw):
            self.seen.append(x.clone())
            return x

    for fm, T, prime in ((4, 8, 0), (4, 8, 3), (3, 5, 0), (1, 4, 0), (5, 2, 7)):
        seq_len = T + fm * fm
        xs = torch.randn(2, seq_len + 1, 16, generator=torch.Generator().manual_seed(fm))
        fa, fb = Rec(), Rec()
        A, B = PreShiftToken(fa, image_size=fm, seq_len=seq_len), PreShiftToken(fb, image_size=fm, seq_len=seq_len)
        n0 = T + 1 + prime
        ca, cb = {'offset': 0}, {'offset': 0}
        A(xs[:, :n0], cache=ca, cache_key='k')
        B(xs[:, :n0], cache=cb, cache_key='k')
        ca['offset'] = cb['offset'] = n0
        cb['k'] = decode.ShiftRing.from_deque(cb['k'], n0, B.text_len, fm)
        pos_t = torch.tensor([n0])
        cb['pos_t'] = pos_t
        for p in range(n0, seq_len):
            A(xs[:, p:p + 1], cache=ca, cache_key='k')
            ca['offset'] += 1
            cb['shift_idx'] = decode.shift_indices(pos_t, B.text_len, fm)
            B(xs[:, p:p + 1], cache=cb, cache_key='k')
            pos_t.add_(1)
        assert len(fa.seen) == len(fb.seen) == seq_len - n0 + 1
        assert all(torch.equal(u, v) for u, v in zip(fa.seen, fb.seen)), (fm, T, prime)


def test_graphed_decoder_drives_a_patched_reference_model(cpu_kernels):
    """INTEGRATION.md: a reference `DALLE` built after `patch_dalle_pytorch()` keeps the reference's own generate loop, but
    `decode.GraphedDecoder` can take over its cache after the prompt pass -- it only touches attributes both DALLE classes share.
    Device-indexed steps == the reference DALLE's own host-indexed cached forward, position by position."""
    import ref_import
    if not ref_import.reference_available():
        pytest.skip('reference not present')
    ref = ref_import.import_reference()
    undo = D.patch_dalle_pytorch()
    try:
        torch.manual_seed(0)
        vae = ref.DiscreteVAE(image_size=32, num_layers=3, num_tokens=24, codebook_dim=16, hidden_dim=8)       # fmap 4
        m = ref.DALLE(dim=32, vae=vae, num_text_tokens=30, text_seq_len=6, depth=2, heads=2, dim_head=16, attn_types=('axial_row', 'axial_col'),
                      shift_tokens=True, optimize_for_inference=True).eval()
    finally:
        undo()
    assert type(m).__module__.startswith('dalle_pytorch.') and decode._attention_layers(m) is not None and decode._flat_plan(m) is not None
    T, n_img = m.text_seq_len, m.image_seq_len
    g = torch.Generator().manual_seed(4)
    text = torch.randint(1, 30, (2, T), generator=g)
    img = torch.randint(0, 24, (2, n_img), generator=g)
    with torch.no_grad():
        host, dev = {}, {}
        want = [m(text, img[:, :k], cache=host)[:, -1] for k in range(n_img)]
        got = [m(text, img[:, :0], cache=dev)[:, -1]]
        dec = decode.GraphedDecoder(m, dev)
        for k in range(1, n_img):
            got.append(dec.step(img[:, k - 1]).clone())
    for k, (a, b) in enumerate(zip(want, got)):
        live = a > NEG / 2
        assert torch.equal(live, b > NEG / 2), k
        assert torch.allclose(a[live], b[live], rtol=1e-5, atol=1e-6), (k, float((a[live] - b[live]).abs().max()))
