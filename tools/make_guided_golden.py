"""Generate tests/golden/guided_tiny.pt from the UNMODIFIED reference (needs the reference checkout that oracle/ref_import.py finds):

    python tools/make_guided_golden.py

Classifier-free guidance fixture of tests/test_guided_decode_*.py: a tiny model with full and optimize_for_inference axial layers and
token shift, and the reference's UNCACHED guided logits `forward_with_cond_scale(text.clone(), image[:, :k], cond_scale=s)[:, -1]` at
every image position k.  The clone works around the reference forward's in-place `text *= ~null_mask` (dalle_pytorch.py:590-591),
which zeroes the caller's tensor in the null pass and would make every later call unconditional.  Weights are not stored: they are
regenerated from the seed by oracle.dalle_oracle.make_state_dict (a checksum of every tensor is stored to detect drift); the
reference's optimize_for_inference layers carry the same parameters under the same keys as the sparse ones.
"""
import os
import sys

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
from dalle_oracle import OracleConfig, make_state_dict, make_inputs   # noqa: E402
from make_golden import TINY, build_reference                          # noqa: E402
from ref_import import import_reference                                # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden', 'guided_tiny.pt')


def guided_tiny(R, seed=0, cond_scale=3.0):
    cfg = OracleConfig(**{**TINY, 'depth': 3, 'attn_types': ('full', 'axial_row', 'axial_col')})
    sd = make_state_dict(cfg, seed=seed)
    text, image = make_inputs(cfg, 2, seed=seed + 1)
    model = build_reference(R, cfg, sd, dict(optimize_for_inference=True)).eval()
    with torch.no_grad():
        logits = torch.stack([model.forward_with_cond_scale(text.clone(), image[:, :k], cond_scale=cond_scale)[:, -1]
                              for k in range(cfg.image_seq_len)], dim=1)                        # [b, image_seq_len, total_tokens]
    return dict(name='guided_tiny', cfg=cfg.__dict__.copy(), seed=seed, optimize_for_inference=True, cond_scale=cond_scale,
                weight_checksums={k: float(v.double().sum()) for k, v in sd.items()},
                text=text, image=image, logits=logits, torch_version=torch.__version__)


if __name__ == '__main__':
    torch.manual_seed(0)
    torch.save(guided_tiny(import_reference()), OUT)
    print(f'guided_tiny -> {os.path.getsize(OUT) / 1e3:.1f} kB')
