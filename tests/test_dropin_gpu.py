"""Drop-in test: the UNMODIFIED reference `dalle_pytorch.DALLE` (oracle/_ref, copied there by `build()` through
oracle/build_ref.py) built after `patch_dalle_pytorch()` runs its block stack on libdalle_b200 and reproduces the golden vectors that the
same reference produced on the CPU with its own blocks (rtol 1e-3 / atol 1e-5, fp32 parity mode)."""
import pytest
import torch

from conftest import load_golden
from util import report
from dalle_oracle import OracleConfig, make_state_dict

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-3, 1e-5


@pytest.mark.parametrize('name', ['tiny_full', 'tiny_axial', 'tiny_axial_rev', 'tiny_cycle4', 'tiny_full_sandwich'])
def test_patched_reference_reproduces_goldens(name):
    import ref_import
    if not ref_import.reference_available():
        pytest.skip('reference not built into oracle/_ref')
    import dalle_pytorch_b200 as D
    from dalle_pytorch_b200 import ops
    ref = ref_import.import_reference()
    rec = load_golden(name)
    c = dict(rec['cfg'])
    c['attn_types'] = tuple(c['attn_types'])
    cfg = OracleConfig(**c)
    sd = make_state_dict(cfg, seed=rec['seed'])
    undo = D.patch_dalle_pytorch()
    try:
        vae = ref.DiscreteVAE(image_size=8 * cfg.fmap, num_layers=3, num_tokens=cfg.num_image_tokens, codebook_dim=16, hidden_dim=8)
        m = ref.DALLE(dim=cfg.dim, vae=vae, num_text_tokens=cfg.num_text_tokens, text_seq_len=cfg.text_seq_len, depth=cfg.depth,
                      heads=cfg.heads, dim_head=cfg.dim_head, reversible=cfg.reversible, attn_types=cfg.attn_types, stable=cfg.stable,
                      sandwich_norm=cfg.sandwich_norm, shift_tokens=cfg.shift_tokens, loss_img_weight=cfg.loss_img_weight)
    finally:
        undo()
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith('vae.') for k in missing), (missing, unexpected)
    m = m.cuda().train()
    n0 = ops.launches()
    with D.compute_dtype_ctx(torch.float32):
        loss = m(rec['text'].cuda(), rec['image'].cuda(), return_loss=True)
        loss.backward()
        with torch.no_grad():
            logits = m(rec['text'].cuda(), rec['image'].cuda())
    assert ops.launches() - n0 > 4 * cfg.depth, 'the block stack did not run on libdalle_b200'
    report('loss', loss.detach(), rec['loss'], RTOL, ATOL)
    lg = logits.cpu()
    masked = rec['logits'] < -1e30
    assert torch.equal(lg[masked], rec['logits'][masked])
    report('logits', lg[~masked], rec['logits'][~masked], RTOL, ATOL)
    grads = {k: p.grad for k, p in m.named_parameters() if p.grad is not None and not k.startswith('vae.')}
    assert set(grads) == set(rec['grads']), set(grads) ^ set(rec['grads'])
    for k, g in rec['grads'].items():
        report(f'grad {k}', grads[k], g, RTOL, ATOL)
