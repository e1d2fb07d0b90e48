"""Generate the committed golden fixtures under tests/golden/ from the UNMODIFIED reference.

TEST INFRASTRUCTURE.  Run in the dev container (where /root/reference exists):

    python oracle/make_golden.py

For each variant below it builds the reference `DALLE` (imported by oracle/ref_import.py), loads the
deterministic synthetic weights of `oracle.dalle_oracle.make_state_dict(cfg, seed)`, runs
`loss = dalle(text, image, return_loss=True); loss.backward()` and `logits = dalle(text, image)` on the
CPU in fp32 (reference call-site contract: train_dalle.py:609-616), and stores loss, logits and
parameter gradients.  The tiny variants store everything; the C1 variants (BASELINE.json configs[0])
store a strided sample plus norms so the fixtures stay small.  Weights are NOT stored — they are
regenerated from the seed (a checksum of every tensor is stored to detect RNG drift).
"""
import os
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from dalle_oracle import OracleConfig, make_state_dict, make_inputs   # noqa: E402
from ref_import import import_reference                                # noqa: E402

OUT = os.path.join(HERE, '..', 'tests', 'golden')

TINY = dict(dim=64, depth=2, heads=2, dim_head=64, text_seq_len=8, fmap=4, num_text_tokens=50, num_image_tokens=32)
C1 = dict(dim=256, depth=2, heads=4, dim_head=64, text_seq_len=64, fmap=8, num_text_tokens=10000, num_image_tokens=8192)
# BASELINE.json configs[2..4] geometry (dim 1024, heads 16, text 256, image 32x32, full vocabulary) at depth 2, batch 1
CG = dict(dim=1024, depth=2, heads=16, dim_head=64, text_seq_len=256, fmap=32, num_text_tokens=10000, num_image_tokens=8192)

VARIANTS = {
    # name: (base, overrides, batch, full_store)
    'tiny_full': (TINY, dict(attn_types=('full',)), 2, True),
    'tiny_axial': (TINY, dict(attn_types=('axial_row', 'axial_col')), 2, True),
    'tiny_axial_rev': (TINY, dict(attn_types=('axial_row', 'axial_col'), reversible=True), 2, True),
    'tiny_full_stable': (TINY, dict(attn_types=('full',), stable=True), 2, True),
    'tiny_full_noshift': (TINY, dict(attn_types=('full',), shift_tokens=False), 2, True),
    'tiny_full_sandwich': (TINY, dict(attn_types=('full',), sandwich_norm=True), 2, True),
    'tiny_cycle4': (TINY, dict(depth=4, attn_types=('full', 'axial_row', 'axial_col', 'conv_like')), 2, True),
    'tiny_full_rev': (TINY, dict(attn_types=('full',), reversible=True), 2, True),
    'c1_full': (C1, dict(attn_types=('full',)), 2, False),
    'c1_axial': (C1, dict(attn_types=('axial_row', 'axial_col')), 2, False),
    'c1_axial_rev': (C1, dict(attn_types=('axial_row', 'axial_col'), reversible=True), 2, False),
    'tiny_axial_stable': (TINY, dict(attn_types=('axial_row', 'axial_col'), stable=True), 2, True),
    # weight sharing between layers (transformer.py:261-292) and tied input/output embeddings (dalle_pytorch.py:432-443): the
    # reference's own tied state dict is stored with the fixture ('state')
    'tiny_shared': (TINY, dict(depth=4, attn_types=('full', 'axial_row'), shared_attn_ids=(0, 1, 0, 1), shared_ff_ids=(0, 0, 1, 1)), 2, True),
    'tiny_tied_emb': (TINY, dict(attn_types=('full',), share_input_output_emb=True), 2, True),
    'c3_geom': (CG, dict(attn_types=('axial_row', 'axial_col')), 1, False),
    'c4_geom_rev': (CG, dict(attn_types=('axial_row', 'axial_col'), reversible=True), 1, False),
}
STORE_STATE = {'tiny_shared', 'tiny_tied_emb'}

LOGIT_STRIDE = 127
GRAD_SAMPLE = 2048


def sample_flat(t, k=GRAD_SAMPLE):
    f = t.reshape(-1)
    if f.numel() <= k:
        return f.clone(), 1
    step = f.numel() // k
    return f[::step][:k].clone(), step


def build_reference(R, cfg: OracleConfig, sd, extra=None, tied=False):
    vae = R.DiscreteVAE(image_size=8 * cfg.fmap, num_layers=3, num_tokens=cfg.num_image_tokens,
                        codebook_dim=64, hidden_dim=8)
    model = R.DALLE(dim=cfg.dim, vae=vae, num_text_tokens=cfg.num_text_tokens, text_seq_len=cfg.text_seq_len,
                    depth=cfg.depth, heads=cfg.heads, dim_head=cfg.dim_head, reversible=cfg.reversible,
                    attn_types=cfg.attn_types, stable=cfg.stable, sandwich_norm=cfg.sandwich_norm,
                    shift_tokens=cfg.shift_tokens, rotary_emb=cfg.rotary_emb, loss_img_weight=cfg.loss_img_weight,
                    shared_attn_ids=cfg.shared_attn_ids, shared_ff_ids=cfg.shared_ff_ids, **(extra or {}))
    own = {k: v for k, v in model.state_dict().items() if not k.startswith('vae.')}
    if tied:      # tied weights: the synthetic state dict is loaded where the keys exist (a later layer's copy wins for shared tensors)
        assert torch.equal(own['transformer.pos_emb'], sd['transformer.pos_emb']), 'rotary table mismatch'
        model.load_state_dict({k: v for k, v in sd.items() if k in own and own[k].shape == v.shape}, strict=False)
        return model
    assert set(own.keys()) == set(sd.keys()), (sorted(set(own) ^ set(sd)))
    for k in own:
        assert own[k].shape == sd[k].shape, (k, own[k].shape, sd[k].shape)
    # the oracle's restated rotary table must equal the reference's own buffer (transformer.py:304-328)
    assert torch.equal(own['transformer.pos_emb'], sd['transformer.pos_emb']), 'rotary table mismatch'
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith('vae.') for k in missing)
    return model


def run_variant(R, name, base, over, batch, full_store, seed=0):
    over = dict(over)
    extra = {k: over.pop(k) for k in ('share_input_output_emb',) if k in over}
    cfg = OracleConfig(**{**base, **over})
    sd = make_state_dict(cfg, seed=seed)
    text, image = make_inputs(cfg, batch, seed=seed + 1)
    model = build_reference(R, cfg, sd, extra, tied=name in STORE_STATE)
    model.train()
    t0 = time.time()
    loss = model(text.clone(), image.clone(), return_loss=True)
    loss.backward()
    dt = time.time() - t0
    with torch.no_grad():
        logits = model(text.clone(), image.clone())
    grads = {k: p.grad.detach().clone() for k, p in model.named_parameters() if not k.startswith('vae.') and p.grad is not None}
    rec = dict(name=name, cfg=cfg.__dict__.copy(), seed=seed, batch=batch, loss=loss.detach().clone(),
               text=text, image=image, ref_seconds=dt, torch_version=torch.__version__,
               weight_checksums={k: float(v.double().sum()) for k, v in sd.items()})
    if name in STORE_STATE:
        rec['state'] = {k: v.detach().clone() for k, v in model.state_dict().items() if not k.startswith('vae.')}
        rec['extra'] = extra
    if full_store:
        rec['logits'] = logits.clone()
        rec['grads'] = grads
    else:
        rec['logits_stride'] = LOGIT_STRIDE
        rec['logits_sample'] = logits[..., ::LOGIT_STRIDE].clone()
        live = logits > -1e30
        rec['logits_live_sum'] = torch.where(live, logits, torch.zeros_like(logits)).double().sum(-1).float()
        rec['logits_lse'] = torch.logsumexp(logits.double(), dim=-1).float()
        rec['grad_norms'] = {k: float(g.double().norm()) for k, g in grads.items()}
        rec['grad_samples'] = {k: sample_flat(g) for k, g in grads.items()}
    return rec


def reference_modules(R):
    """Outputs of single reference modules for the module-level pins of tests/test_oracle_vs_golden.py: the axial and
    conv-like sparse attention classes, PreShiftToken, and the static axial masks of the reference Transformer.  Weights
    and inputs come from seeded generators (dalle_oracle.make_attention_inputs, torch.Generator), so only the reference's
    outputs and a checksum of each input are stored."""
    from dalle_oracle import make_attention_inputs, rotary_angle_table
    rec = {'axial': {}, 'conv_like': {}, 'token_shift': {}, 'static_masks': {}, 'torch_version': torch.__version__}

    def attn_record(m, dim, heads, n, text_len, fmap, seed):
        w_qkv, w_out, b_out, x = make_attention_inputs(dim, heads, 64, 2, n, seed=seed)
        with torch.no_grad():
            m.to_qkv.weight.copy_(w_qkv)
            m.to_out[0].weight.copy_(w_out)
            m.to_out[0].bias.copy_(b_out)
            out = m(x, rotary_pos_emb=rotary_angle_table(text_len, fmap, 64)[None])
        return {'out': out, 'checksum': sum(float(t.double().sum()) for t in (w_qkv, w_out, b_out, x))}

    dim, heads, fmap, text_seq = 64, 2, 4, 8
    seq_len = text_seq + fmap * fmap
    for kind, axis in (('axial_row', 0), ('axial_col', 1)):
        for stable in (False, True):
            for n in (24, 19):
                m = R.SparseAxialCausalAttention(dim, seq_len, image_size=fmap, axis=axis, heads=heads, dim_head=64, stable=stable)
                rec['axial'][(kind, stable, n)] = attn_record(m, dim, heads, n, seq_len - fmap * fmap + 1, fmap, seed=n)
    dim, heads, fmap, text_seq = 64, 2, 6, 5
    seq_len = text_seq + fmap * fmap
    for kernel_size, dilation in ((3, 1), (5, 1), (3, 2)):
        m = R.SparseConvCausalAttention(dim, seq_len, image_size=fmap, kernel_size=kernel_size, dilation=dilation, heads=heads, dim_head=64)
        rec['conv_like'][(kernel_size, dilation)] = attn_record(m, dim, heads, seq_len, text_seq + 1, fmap, seed=kernel_size + 10 * dilation)
    fmap, text_seq, dim = 4, 8, 32
    seq_len = text_seq + fmap * fmap
    sh = R.transformer.PreShiftToken(lambda x, **kw: x, image_size=fmap, seq_len=seq_len)
    for n in (seq_len, seq_len - 3, text_seq + 1, 5):
        rec['token_shift'][n] = sh(torch.randn(2, n, dim, generator=torch.Generator().manual_seed(n)))
    t = R.Transformer(dim=64, depth=1, seq_len=24, heads=2, dim_head=64, image_fmap_size=4, attn_types=('full',))
    for kind in ('axial_row', 'axial_col'):
        rec['static_masks'][kind] = t._get_attention_mask(kind).clone()
    return rec


def main():
    torch.manual_seed(0)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    R = import_reference()
    os.makedirs(OUT, exist_ok=True)
    only = sys.argv[1:]
    for name, (base, over, batch, full_store) in VARIANTS.items():
        if only and name not in only:
            continue
        rec = run_variant(R, name, base, over, batch, full_store)
        path = os.path.join(OUT, name + '.pt')
        torch.save(rec, path)
        print(f'{name}: loss={float(rec["loss"]):.6f} ref_time={rec["ref_seconds"]:.3f}s -> {os.path.getsize(path)/1e6:.2f} MB')
    if not only or 'ref_modules' in only:
        path = os.path.join(OUT, 'ref_modules.pt')
        torch.save(reference_modules(R), path)
        print(f'ref_modules -> {os.path.getsize(path) / 1e6:.2f} MB')


if __name__ == '__main__':
    main()
