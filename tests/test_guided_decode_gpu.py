"""Classifier-free guidance on the graph-replayed decoding path, on the B200: the 32-row small-M GEMM kernel, the guided sampling
kernel, teacher-forced guided logits against the reference (tests/golden/guided_tiny.pt) and generate_images end to end."""
import pytest
import torch

from conftest import load_golden
from util import report
from dalle_oracle import OracleConfig, make_state_dict

pytestmark = pytest.mark.gpu


def ops():
    from dalle_pytorch_b200 import ops as o
    return o


def _mk(shape, dtype, scale=1.0):
    return (torch.randn(shape, device='cuda') * scale).to(dtype)


@pytest.mark.parametrize('M', [17, 24, 32])
@pytest.mark.parametrize('N,K', [(1024, 1024), (3072, 1024), (1024, 4096), (64, 256), (48, 768)])
def test_small_m_gemm_kernel_32_rows(M, N, K):
    """gemm_smallm32_kernel (two A fragments per weight fragment) through the ops entry points under ops.small_m_rows(32): STORE,
    RESID, GEGLU against torch's fp32 product of the same bf16 operands, and every launch on the small-M backend."""
    o = ops()
    torch.manual_seed(171 + M + N)
    A, W = _mk((M, K), torch.bfloat16), _mk((N, K), torch.bfloat16, K ** -0.5)
    bias = _mk((N,), torch.float32)
    acc = A.float() @ W.float().t()
    assert not o._small_m(A, N)                                          # the default rule stays at 16 rows
    o.gemm_timing(True)
    with o.small_m_rows(32):
        got = o.gemm_store(A, W)
        got_b = o.gemm_store(A, W, bias=bias, out_dtype=torch.float32)
        resid, scale = _mk((M, N), torch.float32), _mk((N,), torch.float32)
        out, y = o.gemm_resid(A, W, bias, resid, scale, sign=-1.0, keep_y=True)
        out2, y2 = o.gemm_resid(A, W, bias, None, None, 1.0)
        H = N // 2
        h, u = o.gemm_geglu(A, W, bias, keep_u=True)
        h2, u2 = o.gemm_geglu(A, W, bias, keep_u=False)
    st = o.gemm_timing(False)
    assert st['smallm']['launches'] == 6 and st['tcgen05']['launches'] == 0 and st['simt']['launches'] == 0, st
    report(f'small-M32 store {M}x{N}x{K}', got, acc, 1e-2, 1e-2)
    report(f'small-M32 store+bias fp32 {M}x{N}x{K}', got_b, acc + bias, 1e-4, 1e-4)
    report(f'small-M32 resid {M}x{N}x{K}', out, resid - scale * (acc + bias), 1e-4, 1e-4)
    report(f'small-M32 resid y {M}x{N}x{K}', y, acc + bias, 1e-2, 1e-2)
    report(f'small-M32 plain projection {M}x{N}x{K}', out2, acc + bias, 1e-4, 1e-4)
    assert y2 is None and u2 is None
    ub = acc + bias
    report(f'small-M32 geglu u {M}x{N}x{K}', u, ub, 1e-2, 1e-2)
    report(f'small-M32 geglu h {M}x{N}x{K}', h, ub[:, :H] * torch.nn.functional.gelu(ub[:, H:]), 1e-2, 1e-2)
    assert torch.equal(h, h2)
    # rows 0..15 of the 32-row kernel == the 16-row kernel (the same fixed-order reduction per row)
    assert torch.equal(got_b[:16], o.gemm_store(A[:16].contiguous(), W, bias=bias, out_dtype=torch.float32))


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
@pytest.mark.parametrize('V,thres,s', [(18448, 0.5, 3.0), (18448, 0.9, 1.7), (1000, 0.0, -0.5), (90, 0.99, 3.0)])
def test_guided_sampling_equals_torch_guided_logits(dtype, V, thres, s):
    """dalle_b200_sample_guided_topk_gumbel forms null + (cond - null) * s exactly as torch does, so it gives the tokens of torch's
    guided logits through dalle_b200_sample_topk_gumbel (Philox noise, same seed / offset) and through top_k + Gumbel arg-max with
    explicit noise."""
    o = ops()
    torch.manual_seed(81)
    b = 16
    logits = (torch.randn(2 * b, V, device='cuda') * 3).to(dtype)
    logits[:, : V // 3] = -torch.finfo(dtype).max                        # the logits mask of DALLE.forward, in both streams
    cond, null = logits[:b], logits[b:]
    guided = null + (cond - null) * s
    for seed, off in ((5, 0), (123, 7 * 10 ** 9)):
        for temp in (1.0, 0.7):
            want = o.sample_topk_gumbel(guided.contiguous(), thres, temp, seed=seed, offset=off)
            got = o.sample_guided_topk_gumbel(logits, s, thres, temp, seed=seed, offset=off)
            assert torch.equal(got, want), (seed, temp, got, want)
    noise = -torch.log(-torch.log(torch.rand(b, V, device='cuda').clamp_min(1e-20)))
    k = max(int((1 - thres) * V), 1)
    val, ind = torch.topk(guided.float(), k)
    filt = torch.full_like(guided.float(), float('-inf')).scatter_(1, ind, val)
    for temp in (1.0, 0.7):
        want = (filt / temp + noise).argmax(-1)
        assert torch.equal(o.sample_guided_topk_gumbel(logits, s, thres, temp, gumbel=noise), want)
        assert torch.equal(o.sample_topk_gumbel(guided.contiguous(), thres, temp, gumbel=noise), want)


def _golden_model(rec):
    import dalle_pytorch_b200 as D
    c = dict(rec['cfg'])
    c['attn_types'] = tuple(c['attn_types'])
    cfg = OracleConfig(**c)
    vae = D.TokenVAE(image_size=8 * cfg.fmap, num_layers=3, num_tokens=cfg.num_image_tokens)
    m = D.DALLE(dim=cfg.dim, vae=vae, num_text_tokens=cfg.num_text_tokens, text_seq_len=cfg.text_seq_len, depth=cfg.depth, heads=cfg.heads,
                dim_head=cfg.dim_head, attn_types=cfg.attn_types, shift_tokens=cfg.shift_tokens, optimize_for_inference=rec['optimize_for_inference'])
    m.load_state_dict(make_state_dict(cfg, seed=rec['seed']))
    return m.cuda().eval(), cfg


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
def test_teacher_forced_guided_logits_match_reference(dtype):
    """Guided prompt pass + GuidedDecoder replays, fed the fixture's image tokens: null + (cond - null) * s at every position ==
    the reference's uncached forward_with_cond_scale (fp32: rtol 1e-3 / atol 1e-5; bf16: 6e-2 absolute as test_goldens_bf16_mode)."""
    import dalle_pytorch_b200 as D
    from dalle_pytorch_b200 import decode
    rec = load_golden('guided_tiny')
    m, cfg = _golden_model(rec)
    text, img, s = rec['text'].cuda(), rec['image'].cuda(), rec['cond_scale']
    b = text.shape[0]
    with D.compute_dtype_ctx(dtype), torch.no_grad():
        dev = {}
        steps = [decode.guided_prompt(m, text, img[:, :0], dev).float()]
        dec = decode.GuidedDecoder(m, dev)
        for k in range(1, cfg.image_seq_len):
            steps.append(dec.step(img[:, k - 1]).float().clone())
    assert dec.graph is not None, 'the guided decoder must have captured and replayed its step'
    got = torch.stack([x[b:] + (x[:b] - x[b:]) * s for x in steps], dim=1).cpu()
    want = rec['logits']
    masked = want < -1e30
    assert torch.equal(got[masked], want[masked])
    if dtype == torch.float32:
        report('guided logits fp32', got[~masked], want[~masked], 1e-3, 1e-5)
    else:
        report('guided logits bf16', got[~masked], want[~masked], 0.0, 6e-2)


def test_generate_images_guided_graph_equals_uncached_guidance(monkeypatch):
    """generate_images(use_cache=True, cond_scale=3) takes GuidedDecoder (graphs captured) and gives, for a seed, the tokens of
    generate_images(use_cache=False, cond_scale=3) -- classifier-free guidance by its definition (fp32)."""
    import dalle_pytorch_b200 as D
    from dalle_pytorch_b200 import decode
    rec = load_golden('guided_tiny')
    m, cfg = _golden_model(rec)
    made = []

    class Spy(decode.GuidedDecoder):
        def __init__(self, *a, **k):
            made.append(self)
            super().__init__(*a, **k)
    monkeypatch.setattr(decode, 'GuidedDecoder', Spy)
    text = rec['text'].cuda()
    toks = {}
    with D.compute_dtype_ctx(torch.float32):
        for use_cache in (False, True):
            torch.manual_seed(17)
            toks[use_cache] = m.generate_images(text, use_cache=use_cache, cond_scale=3.0, filter_thres=0.8).cpu()
    assert len(made) == 1 and made[0].graph is not None and made[0].batch == 2 * text.shape[0]
    assert torch.equal(toks[False], toks[True]), (toks[False], toks[True])


def test_guided_step_gemms_run_on_the_small_m_kernel_at_batch_16(monkeypatch):
    """At batch 16 the two streams make M = 32: every GEMM of a guided step (QKV, out-projection, both feed-forward GEMMs of every
    layer) runs on the small-M backend."""
    import dalle_pytorch_b200 as D
    from dalle_pytorch_b200 import decode, ops as o
    torch.manual_seed(31)
    vae = D.TokenVAE(image_size=64, num_layers=3, num_tokens=48)         # fmap 8
    m = D.DALLE(dim=256, vae=vae, num_text_tokens=64, text_seq_len=16, depth=2, heads=4, attn_types=('full', 'axial_row'),
                optimize_for_inference=True).cuda().eval()
    b = 16
    text = torch.randint(1, 64, (b, 16), generator=torch.Generator().manual_seed(32)).cuda()
    img = torch.randint(0, 48, (b, 4), generator=torch.Generator().manual_seed(33)).cuda()
    with D.compute_dtype_ctx(torch.bfloat16), torch.no_grad():
        dev = {}
        decode.guided_prompt(m, text, img[:, :0], dev)
        dec = decode.GuidedDecoder(m, dev)
        assert dec.plan is not None
        o.gemm_timing(True)
        dec.step(img[:, 0])                                               # first step: eager (warm-up), so every launch is seen
        st = o.gemm_timing(False)
        for k in range(1, 4):                                             # and the captured replays run
            dec.step(img[:, k])
    torch.cuda.synchronize()
    assert st['smallm']['launches'] == 4 * 2 and st['tcgen05']['launches'] == 0 and st['simt']['launches'] == 0, st
    assert all(key.split(':')[-1].startswith('32x') for key in st['by_shape']), st['by_shape']
