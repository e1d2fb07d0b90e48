"""Classifier-free guidance on the graph-replayed decoding path (decode.GuidedDecoder) without a GPU.

The guided step decodes the conditional and the unconditional stream as one batch of 2b sequences.  Its host logic is plain torch,
so it is checked on the CPU with the library calls of a cached step replaced by the torch stubs of tests/test_decode_cpu.py: rows
[:b] of every guided step must equal a host-indexed cached pass on the real text, rows [b:] one on zeroed text with a cache of its
own.  The guided logits themselves are pinned against the reference (tests/golden/guided_tiny.pt, tools/make_guided_golden.py)
through the oracle.
"""
import pytest
import torch

from conftest import load_golden
from dalle_oracle import OracleConfig, dalle_forward, make_state_dict
from test_decode_cpu import NEG, _model, cpu_kernels  # noqa: F401  (cpu_kernels is a fixture)

from dalle_pytorch_b200 import decode


@pytest.mark.parametrize('flat,bucket', [(False, 0), (True, 0), (True, 8)])
@pytest.mark.parametrize('name,kw', [
    ('full_shift', dict()),
    ('axial_static_masks', dict(attn_types=('axial_row', 'axial_col'), optimize=True, depth=3)),
    ('sandwich_norm', dict(sandwich=True)),                     # the flat step does not cover it: the guided step walks the module nest
])
def test_guided_step_rows_equal_separate_host_indexed_passes(cpu_kernels, monkeypatch, name, kw, flat, bucket):
    monkeypatch.setattr(decode, 'FLAT_DEFAULT', flat)
    monkeypatch.setattr(decode, 'BUCKET_DEFAULT', bucket)
    m = _model(**kw)
    T, n_img = m.text_seq_len, m.image_seq_len
    g = torch.Generator().manual_seed(5)
    text = torch.randint(1, 30, (2, T), generator=g)
    text[0, -2:] = 0                                                                     # padded tail: the pad-id remap in both streams
    img = torch.randint(0, 24, (2, n_img), generator=g)
    b = text.shape[0]
    with torch.no_grad():
        cond_c, null_c, dev = {}, {}, {}
        want_cond = [m(text, img[:, :k], cache=cond_c)[:, -1] for k in range(n_img)]
        want_null = [m(torch.zeros_like(text), img[:, :k], cache=null_c)[:, -1] for k in range(n_img)]
        got = [decode.guided_prompt(m, text, img[:, :0], dev)]
        dec = decode.GuidedDecoder(m, dev)
        assert dec.batch == 2 * b and (dec.plan is not None) == (flat and name != 'sandwich_norm')
        for k in range(1, n_img):
            got.append(dec.step(img[:, k - 1]).clone())
    assert dev['offset'] == T + n_img and int(dec.pos_t) == T + n_img
    for k in range(n_img):
        assert got[k].shape == (2 * b, m.total_tokens)
        for half, want in ((got[k][:b], want_cond[k]), (got[k][b:], want_null[k])):
            live = want > NEG / 2
            assert torch.equal(live, half > NEG / 2), (name, k)
            assert torch.allclose(half[live], want[live], rtol=1e-5, atol=1e-6), (name, k, float((half[live] - want[live]).abs().max()))
    # the two streams really differ (the text matters), so the comparison above would catch swapped or shared caches
    assert not torch.allclose(got[-1][:b], got[-1][b:])


def test_generate_images_guided_path_keeps_the_uncached_tokens(cpu_kernels, monkeypatch):
    """generate_images(use_cache=True, cond_scale=s) through GuidedDecoder gives, for a seed, the tokens of the uncached guided loop
    (the spec: two independent forwards per token, and the same random draws); DALLE_B200_DECODE_GUIDED=0 keeps the eager cached
    loop."""
    m = _model(attn_types=('full', 'axial_row', 'axial_col'), optimize=True, depth=3)
    monkeypatch.setattr(decode, 'eligible', lambda model, text, cond_scale: decode._attention_layers(model) is not None)
    monkeypatch.setattr(decode, 'GRAPH_DEFAULT', True)
    text = torch.randint(1, 30, (2, m.text_seq_len), generator=torch.Generator().manual_seed(9))
    made = []
    real = decode.GuidedDecoder

    class Spy(real):
        def __init__(self, *a, **k):
            made.append(self)
            super().__init__(*a, **k)
    monkeypatch.setattr(decode, 'GuidedDecoder', Spy)
    # the uncached loop, with every forward over the whole prefix taken through the cached code path on a fresh cache (the
    # stubs cover that path; the same function of the prefix, and the same random draws)
    fwd = m.forward
    m.forward = lambda *a, cache=None, **k: fwd(*a, cache={} if cache is None else cache, **k)
    torch.manual_seed(3)
    want = m.generate_images(text, use_cache=False, cond_scale=3.0, filter_thres=0.8)
    del m.forward
    torch.manual_seed(3)
    got = m.generate_images(text, use_cache=True, cond_scale=3.0, filter_thres=0.8)
    assert len(made) == 1 and made[0].batch == 4
    assert torch.equal(want, got), (want, got)
    monkeypatch.setattr(decode, 'GUIDED_DEFAULT', False)
    m.generate_images(text, use_cache=True, cond_scale=3.0)
    assert len(made) == 1


def test_guided_golden_from_two_oracle_forwards():
    """The reference's uncached forward_with_cond_scale (guided_tiny.pt) == null + (cond - null) * s of two oracle forwards, one on
    the real text and one on zeroed text, at every image position."""
    rec = load_golden('guided_tiny')
    c = dict(rec['cfg'])
    c['attn_types'] = tuple(c['attn_types'])
    cfg = OracleConfig(**c)
    sd, s = make_state_dict(cfg, seed=rec['seed']), rec['cond_scale']
    for key, v in rec['weight_checksums'].items():
        assert abs(float(sd[key].double().sum()) - v) <= 1e-6 * max(1.0, abs(v)), f'synthetic weight drift in {key}'
    text, image = rec['text'], rec['image']
    assert s == 3.0 and rec['logits'].shape == (text.shape[0], cfg.image_seq_len, cfg.total_tokens)
    with torch.no_grad():
        for k in range(cfg.image_seq_len):
            cond = dalle_forward(text, image[:, :k], sd, cfg)[:, -1]
            null = dalle_forward(torch.zeros_like(text), image[:, :k], sd, cfg)[:, -1]
            got, want = null + (cond - null) * s, rec['logits'][:, k]
            masked = want < -1e30
            assert torch.equal(got[masked], want[masked]), k
            assert torch.allclose(got[~masked], want[~masked], rtol=1e-3, atol=1e-5), (k, float((got - want)[~masked].abs().max()))
