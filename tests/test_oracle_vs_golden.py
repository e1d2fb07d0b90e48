"""Pins oracle/dalle_oracle.py (the CPU restatement) against the golden vectors generated from the
UNMODIFIED reference by oracle/make_golden.py: whole models, and single reference modules (tests/golden/ref_modules.pt).
Tolerance: BASELINE.json north_star — rtol 1e-3 / atol 1e-5 in fp32 (the oracle usually agrees to ~1e-6)."""
import functools

import pytest
import torch

from conftest import load_golden, golden_names
from dalle_oracle import (OracleConfig, make_state_dict, make_inputs, make_attention_inputs, dalle_forward, allowed_mask,
                          attention_core, rotary_angle_table, token_shift)

RTOL, ATOL = 1e-3, 1e-5


def _cfg(rec):
    c = dict(rec['cfg'])
    c['attn_types'] = tuple(c['attn_types'])
    return OracleConfig(**c)


def _oracle_run(rec):
    cfg = _cfg(rec)
    sd = make_state_dict(cfg, seed=rec['seed'])
    for k, v in rec['weight_checksums'].items():
        assert abs(float(sd[k].double().sum()) - v) <= 1e-6 * max(1.0, abs(v)), f'synthetic weight drift in {k}'
    params = {k: v.clone().requires_grad_(k != 'transformer.pos_emb') for k, v in sd.items()}
    loss = dalle_forward(rec['text'].clone(), rec['image'].clone(), params, cfg, return_loss=True)
    loss.backward()
    with torch.no_grad():
        logits = dalle_forward(rec['text'].clone(), rec['image'].clone(), sd, cfg)
    grads = {k: p.grad for k, p in params.items() if p.grad is not None}
    return loss.detach(), logits, grads


# fixtures whose weights are tied (stored with the fixture): the oracle restates the un-tied block stack; these goldens pin
# the product directly (tests/test_parity_gpu.py::test_tied_weight_goldens_fp32)
TIED = {'tiny_shared', 'tiny_tied_emb'}


@pytest.mark.parametrize('name', [n for n in golden_names('tiny_') if n not in TIED])
def test_oracle_matches_reference_tiny(name):
    rec = load_golden(name)
    loss, logits, grads = _oracle_run(rec)
    torch.testing.assert_close(loss, rec['loss'], rtol=RTOL, atol=ATOL)
    masked = rec['logits'] < -1e30
    assert torch.equal(masked, logits < -1e30)
    assert torch.equal(logits[masked], rec['logits'][masked])          # exactly -fp32max (dalle_pytorch.py:651-652)
    torch.testing.assert_close(logits[~masked], rec['logits'][~masked], rtol=RTOL, atol=ATOL)
    assert set(grads) == set(rec['grads'])
    for k, g in rec['grads'].items():
        torch.testing.assert_close(grads[k], g, rtol=RTOL, atol=ATOL, msg=lambda m: f'{k}: {m}')


@pytest.mark.parametrize('name', golden_names('c1_') + ['c3_geom'])
def test_oracle_matches_reference_c1(name):
    rec = load_golden(name)
    loss, logits, grads = _oracle_run(rec)
    torch.testing.assert_close(loss, rec['loss'], rtol=RTOL, atol=ATOL)
    samp = logits[..., ::rec['logits_stride']]
    masked = rec['logits_sample'] < -1e30
    assert torch.equal(samp[masked], rec['logits_sample'][masked])
    torch.testing.assert_close(samp[~masked], rec['logits_sample'][~masked], rtol=RTOL, atol=ATOL)
    torch.testing.assert_close(torch.logsumexp(logits.double(), -1).float(), rec['logits_lse'], rtol=RTOL, atol=1e-4)
    for k, (vals, step) in rec['grad_samples'].items():
        mine = grads[k].reshape(-1)[::step][:vals.numel()]
        torch.testing.assert_close(mine, vals, rtol=RTOL, atol=ATOL, msg=lambda m: f'{k}: {m}')
        assert abs(float(grads[k].double().norm()) - rec['grad_norms'][k]) <= 1e-3 * rec['grad_norms'][k] + 1e-7


@functools.lru_cache(maxsize=None)
def _ref_modules():
    return load_golden('ref_modules')


def _attention_inputs(rec, dim, heads, n, seed):
    w_qkv, w_out, b_out, x = make_attention_inputs(dim, heads, 64, 2, n, seed=seed)
    got = sum(float(t.double().sum()) for t in (w_qkv, w_out, b_out, x))
    assert abs(got - rec['checksum']) <= 1e-6 * max(1.0, abs(rec['checksum'])), 'synthetic weight / input drift'
    return w_qkv, w_out, b_out, x


@pytest.mark.parametrize('kind,axis', [('axial_row', 0), ('axial_col', 1)])
@pytest.mark.parametrize('stable', [False, True])
@pytest.mark.parametrize('n', [24, 19])
def test_oracle_attention_matches_live_reference_axial(kind, axis, stable, n):
    """Module-level pin: SparseAxialCausalAttention (attention.py:225-335) == oracle attention_core with the
    allowed-key predicate, including n < seq_len (padded tail sliced off, attention.py:255-258, 335).  The reference's
    outputs are stored in tests/golden/ref_modules.pt (oracle/make_golden.py:reference_modules)."""
    rec = _ref_modules()['axial'][(kind, stable, n)]
    dim, heads, fmap, text_seq = 64, 2, 4, 8
    seq_len = text_seq + fmap * fmap
    text_len = seq_len - fmap * fmap + 1
    w_qkv, w_out, b_out, x = _attention_inputs(rec, dim, heads, n, seed=n)
    ang = rotary_angle_table(text_len, fmap, 64)
    allow = allowed_mask(kind, n, n, text_len, fmap)
    mine = attention_core(x, w_qkv, w_out, b_out, heads, ang, allow, stable)
    torch.testing.assert_close(mine, rec['out'], rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize('kernel_size,dilation', [(3, 1), (5, 1), (3, 2)])
def test_oracle_attention_matches_live_reference_conv_like(kernel_size, dilation):
    """SparseConvCausalAttention (attention.py:103-221) == oracle attention_core with the conv-like predicate; the reference's
    outputs are stored in tests/golden/ref_modules.pt."""
    rec = _ref_modules()['conv_like'][(kernel_size, dilation)]
    dim, heads, fmap, text_seq = 64, 2, 6, 5
    seq_len = text_seq + fmap * fmap
    text_len = text_seq + 1
    w_qkv, w_out, b_out, x = _attention_inputs(rec, dim, heads, seq_len, seed=kernel_size + 10 * dilation)
    ang = rotary_angle_table(text_len, fmap, 64)
    allow = allowed_mask('conv_like', seq_len, seq_len, text_len, fmap, kernel_size=kernel_size, dilation=dilation)
    mine = attention_core(x, w_qkv, w_out, b_out, heads, ang, allow, False)
    torch.testing.assert_close(mine, rec['out'], rtol=RTOL, atol=ATOL)


def test_oracle_token_shift_matches_live_reference():
    """PreShiftToken (transformer.py) == oracle token_shift, full and shorter sequences; the reference's outputs are stored in
    tests/golden/ref_modules.pt."""
    stored = _ref_modules()['token_shift']
    fmap, text_seq, dim = 4, 8, 32
    seq_len = text_seq + fmap * fmap
    assert sorted(stored) == sorted((seq_len, seq_len - 3, text_seq + 1, 5))
    for n, want in stored.items():
        x = torch.randn(2, n, dim, generator=torch.Generator().manual_seed(n))
        assert torch.equal(want, token_shift(x, text_seq + 1, fmap)), n


def test_static_mask_equals_predicate():
    """The reference's own cross-check (transformer.py:333-350): static axial masks AND causal == predicate; the reference's
    masks are stored in tests/golden/ref_modules.pt."""
    masks = _ref_modules()['static_masks']
    caus = torch.ones(24, 24).tril().bool()
    for kind in ('axial_row', 'axial_col'):
        assert torch.equal(masks[kind] & caus, allowed_mask(kind, 24, 24, 9, 4))
