"""CPU oracle for the DALL-E transformer hot path (TEST INFRASTRUCTURE — never imported by the product).

A functional, loop-and-index restatement of the reference algorithm for the path named by
BASELINE.json `north_star` (SURVEY.md §8a / Appendix A).  It is deliberately written in a different
style from the reference (explicit allowed-key predicates and index arithmetic instead of
einops/einsum reshapes) so that agreement between the two is evidence, not tautology.

Parity status: PINNED against the reference.  `oracle/make_golden.py` imports the unmodified
reference (oracle/ref_import.py, with the dependency shims under oracle/shims) and writes golden
tensors to tests/golden/*.pt: whole models, and single reference modules (ref_modules.pt: sparse
attention classes, token shift, static masks); `tests/test_oracle_vs_golden.py` checks this file
against those fixtures.  One dependency of the
reference, `rotary-embedding-torch`, is un-vendored and unpinned (reference setup.py:29); its two
functions are restated from the published algorithm in oracle/shims/rotary_embedding_torch.py and
here (`rotary_angle_table`, `apply_rotary`), so the rotary part is "pinned to the restated library",
which DESIGN.md states.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module.

All functions are dtype-agnostic: run them on float32 tensors for the reference's own arithmetic or on
float64 tensors for a noise-floor tie-breaker.

Reference citations are relative to /root/reference/dalle_pytorch/.
"""
from dataclasses import dataclass, field
from math import pi
from typing import Optional, Tuple

import torch
import torch.nn.functional as F


# ----------------------------------------------------------------------------------------------
# configuration
# ----------------------------------------------------------------------------------------------
@dataclass
class OracleConfig:
    dim: int
    depth: int
    heads: int
    dim_head: int = 64
    text_seq_len: int = 256
    fmap: int = 32                       # image_fmap_size (dalle_pytorch.py:383)
    num_text_tokens: int = 10000         # BEFORE the +text_seq_len padding ids (dalle_pytorch.py:386)
    num_image_tokens: int = 8192
    attn_types: Tuple[str, ...] = ('full',)
    reversible: bool = False
    stable: bool = False
    sandwich_norm: bool = False
    shift_tokens: bool = True
    rotary_emb: bool = True
    loss_img_weight: float = 7.0
    ff_mult: int = 4
    shared_attn_ids: Optional[Tuple[int, ...]] = None
    shared_ff_ids: Optional[Tuple[int, ...]] = None

    @property
    def image_seq_len(self):
        return self.fmap * self.fmap

    @property
    def seq_len(self):                   # dalle_pytorch.py:397
        return self.text_seq_len + self.image_seq_len

    @property
    def text_len(self):                  # transformer.py:308 ; attention.py:251  (= text_seq_len + 1 for <bos>)
        return self.seq_len - self.image_seq_len + 1

    @property
    def total_text_tokens(self):         # dalle_pytorch.py:386
        return self.num_text_tokens + self.text_seq_len

    @property
    def total_tokens(self):              # dalle_pytorch.py:398
        return self.total_text_tokens + self.num_image_tokens

    def attn_type_of_layer(self, i):     # transformer.py:236-238 (cycle over depth)
        return self.attn_types[i % len(self.attn_types)]


# ----------------------------------------------------------------------------------------------
# rotary embedding (transformer.py:304-328, attention.py:32-35, rotary_embedding_torch restated)
# ----------------------------------------------------------------------------------------------
def rotary_angle_table(text_len: int, fmap: int, dim_head: int, dtype=torch.float32) -> torch.Tensor:
    """Angle table [text_len + fmap^2, 6*(rot_dim//2)] exactly as transformer.py:304-326 builds
    `pos_emb` (float32 arithmetic like the reference; cast at the end)."""
    rot_dim = dim_head // 3
    nf = rot_dim // 2
    f32 = torch.float32
    # RotaryEmbedding(dim=rot_dim) 'lang' freqs
    lang = 1.0 / (10000 ** (torch.arange(0, rot_dim, 2)[:nf].to(f32) / rot_dim))
    # RotaryEmbedding(dim=rot_dim, freqs_for='pixel', max_freq=10)
    pix = torch.linspace(1.0, 10 / 2, nf) * pi
    n_img = fmap * fmap
    n = text_len + n_img
    table = torch.empty(n, 6 * nf, dtype=f32)

    def rep2(v):                                      # '... n -> ... (n r)', r=2
        return v.repeat_interleave(2, dim=-1)

    # text part of the "language" rotary: position p ; image tokens sit at position 8192 (transformer.py:313-315)
    pos_text = torch.arange(text_len).to(f32)
    table[:text_len, 0:2 * nf] = rep2(pos_text[:, None] * lang[None, :])
    table[text_len:, 0:2 * nf] = rep2(torch.full((n_img,), 8192).to(f32)[:, None] * lang[None, :])
    # axial part: text tokens sit at -10 on both axes, image token (r,c) at linspace(-1,1)[r], [c] (transformer.py:317-323)
    lin = torch.linspace(-1, 1, steps=fmap)
    ax = rep2(lin[:, None] * pix[None, :])            # [fmap, 2*nf]
    tx = rep2(torch.full((text_len,), -10.0)[:, None] * pix[None, :])
    table[:text_len, 2 * nf:4 * nf] = tx
    table[:text_len, 4 * nf:6 * nf] = tx
    for r in range(fmap):
        for c in range(fmap):
            p = text_len + r * fmap + c
            table[p, 2 * nf:4 * nf] = ax[r]
            table[p, 4 * nf:6 * nf] = ax[c]
    return table.to(dtype)


def apply_rotary(angles: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
    """t[..., n, dh]; angles[n, R] with R <= dh.  Interleaved-pair rotation of dims [0,R), rest pass
    (rotary_embedding_torch.apply_rotary_emb as called from attention.py:32-35)."""
    R = angles.shape[-1]
    ang = angles.to(t.dtype)
    c, s = ang.cos(), ang.sin()
    x = t[..., :R]
    x_even, x_odd = x[..., 0::2], x[..., 1::2]
    out = torch.empty_like(x)
    out[..., 0::2] = x_even * c[..., 0::2] - x_odd * s[..., 0::2]
    out[..., 1::2] = x_odd * c[..., 1::2] + x_even * s[..., 1::2]
    return torch.cat([out, t[..., R:]], dim=-1)


# ----------------------------------------------------------------------------------------------
# attention patterns as allowed(i, j) predicates
# ----------------------------------------------------------------------------------------------
def allowed_mask(kind: str, n_q: int, n_k: int, text_len: int, fmap: int, causal: bool = True,
                 kernel_size: int = 5, dilation: int = 1) -> torch.Tensor:
    """Boolean [n_q, n_k]: may query i attend key j.
    'full'      : attention.py:84-87   (causal triu(j - i + 1))
    'axial_row' : attention.py:271-314 (text causal; image -> all text + same row, col' <= col)
    'axial_col' : same with axis = 1   (same column, row' <= row)
    'conv_like' : attention.py:103-221 (text causal; image -> all text + causal k x k dilated window)
    The axial definitions equal transformer.py:333-350 `_get_attention_mask` AND causal.
    """
    i = torch.arange(n_q)[:, None] + (n_k - n_q)     # absolute position of query (attention.py:86: triu(j-i+1))
    j = torch.arange(n_k)[None, :]
    caus = (j <= i) if causal else torch.ones(n_q, n_k, dtype=torch.bool)
    if kind == 'full':
        return caus
    is_text_k = j < text_len
    is_img_q = i >= text_len
    qi = (i - text_len).clamp(min=0)
    kj = (j - text_len).clamp(min=0)
    qr, qc = qi // fmap, qi % fmap
    kr, kc = kj // fmap, kj % fmap
    if kind == 'axial_row':
        same = (qr == kr) & (kc <= qc)
    elif kind == 'axial_col':
        same = (qc == kc) & (kr <= qr)
    elif kind == 'conv_like':
        return conv_like_allowed(n_q, n_k, text_len, fmap, kernel_size, dilation)
    else:
        raise ValueError(kind)
    img = is_img_q & (~is_text_k) & same
    text_k = is_text_k & caus                        # text query: causal over text; image query: every text key
    return text_k | img


def conv_like_allowed(n_q, n_k, text_len, fmap, kernel_size, dilation):
    """attention.py:147-207.  Image query q=(r,c) sees every text key plus the image keys of the
    kernel_size x kernel_size (dilation d) window whose BOTTOM-RIGHT corner is (r,c): the reference pads
    the key/value maps with causal_padding = (2*same, 0, 2*same, 0) (left/top only, attention.py:163-168)
    and unfolds, so window element (a,b) is key (r - 2*same + a*d, c - 2*same + b*d); elements that fall
    in the padding are masked (attention.py:181-191).  Every in-range window key precedes or equals the
    query in raster order, so no further causal mask exists in the reference."""
    assert n_q == n_k
    eff = (kernel_size - 1) * dilation + 1
    same = eff // 2
    m = torch.zeros(n_q, n_k, dtype=torch.bool)
    for i in range(n_q):
        if i < text_len:
            m[i, :i + 1] = True
            continue
        m[i, :text_len] = True
        q = i - text_len
        r, c = q // fmap, q % fmap
        for a in range(kernel_size):
            for b in range(kernel_size):
                rr = r - 2 * same + a * dilation
                cc = c - 2 * same + b * dilation
                if 0 <= rr < fmap and 0 <= cc < fmap:
                    m[i, text_len + rr * fmap + cc] = True
    return m


# ----------------------------------------------------------------------------------------------
# sub-layer bodies
# ----------------------------------------------------------------------------------------------
def softmax_rows(scores: torch.Tensor, stable: bool) -> torch.Tensor:
    """attention.py:27-30 (stable_softmax, alpha = 32**2) or plain softmax over the last dim."""
    if stable:
        alpha = 32 ** 2
        t = scores / alpha
        t = t - t.amax(dim=-1, keepdim=True).detach()
        return (t * alpha).softmax(dim=-1)
    return scores.softmax(dim=-1)


def attention_core(x, w_qkv, w_out, b_out, heads, angles, allow, stable, key_mask=None):
    """attention.py:58-99 / 246-335 with the pattern given as a boolean allow[n,n] matrix.
    x [b,n,d]; w_qkv [3*h*dh, d] (no bias, attention.py:52); w_out [d, h*dh], b_out [d]."""
    b, n, d = x.shape
    inner = w_qkv.shape[0] // 3
    dh = inner // heads
    qkv = x @ w_qkv.t()                                         # attention.py:63
    q, k, v = qkv[..., :inner], qkv[..., inner:2 * inner], qkv[..., 2 * inner:]

    def split(t):                                               # 'b n (h d) -> b h n d'
        return t.reshape(b, n, heads, dh).permute(0, 2, 1, 3)

    q, k, v = split(q), split(k), split(v)
    if angles is not None:                                      # rotary on q, k AND v (attention.py:66-67)
        a = angles[:n]
        q, k, v = apply_rotary(a, q), apply_rotary(a, k), apply_rotary(a, v)
    q = q * (dh ** -0.5)                                        # attention.py:69
    scores = q @ k.transpose(-1, -2)
    neg = -torch.finfo(scores.dtype).max                        # attention.py:24-25
    if key_mask is not None:                                    # attention.py:80-83
        scores = scores.masked_fill(~key_mask[:, None, None, :n], neg)
    scores = scores.masked_fill(~allow[None, None, :n, :n], neg)
    p = softmax_rows(scores, stable)
    o = p @ v
    o = o.permute(0, 2, 1, 3).reshape(b, n, inner)              # 'b h n d -> b n (h d)'
    return o @ w_out.t() + b_out                                # attention.py:97 (dropout p=0)


def token_shift(x, text_len, fmap):
    """transformer.py:155-186 (training branch).  x [b,n,d], n >= text_len.
    Restated as a per-position source-index gather (vectorised so the CPU baseline is not slowed by Python loops):
      text token p     : channels [0,d/2)   <- token p-1            (zero at p = 0)            (:171-173)
      image token (r,c): channels [0,d/4)   <- token (r-1,c)        (zero on the first row)    (:177-180)
                         channels [d/4,d/2) <- token (r,c-1)        (zero on the first column)
      remaining channels unchanged."""
    b, n, d = x.shape
    if n < text_len:                                            # transformer.py:160-161
        return x
    half, quarter = d // 2, d // 4
    pos = torch.arange(n)
    is_text = pos < text_len
    q = (pos - text_len).clamp(min=0)
    row, col = q // fmap, q % fmap
    # first quarter: text <- p-1 ; image <- p-fmap
    src_a = torch.where(is_text, pos - 1, pos - fmap)
    ok_a = torch.where(is_text, pos > 0, row > 0)
    # second quarter: text <- p-1 ; image <- p-1 unless first column
    src_b = pos - 1
    ok_b = torch.where(is_text, pos > 0, col > 0)
    part_a = x[:, :, :quarter].index_select(1, src_a.clamp(min=0)) * ok_a.to(x.dtype)[None, :, None]
    part_b = x[:, :, quarter:half].index_select(1, src_b.clamp(min=0)) * ok_b.to(x.dtype)[None, :, None]
    return torch.cat([part_a, part_b, x[:, :, half:]], dim=-1)


def feed_forward(x, w1, b1, w2, b2, drop_mask=None):
    """transformer.py:106-122: Linear(d, 2*mult*d) -> GEGLU (x * gelu_erf(gates)) -> Dropout -> Linear(mult*d, d).
    drop_mask (optional, [b,n,mult*d], entries 0 or 1/(1-p)) is the Dropout of transformer.py:117 with an explicit mask."""
    u = x @ w1.t() + b1
    half = u.shape[-1] // 2
    a, g = u[..., :half], u[..., half:]
    h = a * F.gelu(g)
    if drop_mask is not None:
        h = h * drop_mask
    return h @ w2.t() + b2


def layer_norm(x, w, b):
    return F.layer_norm(x, (x.shape[-1],), w, b, 1e-5)          # nn.LayerNorm default eps (transformer.py:95)


# ----------------------------------------------------------------------------------------------
# state-dict plumbing (SURVEY.md App. A.8)
# ----------------------------------------------------------------------------------------------
def _layer_prefixes(cfg: OracleConfig, i: int):
    if cfg.reversible:
        pa = f'transformer.layers.blocks.{i}.f.net.'
        pf = f'transformer.layers.blocks.{i}.g.net.'
    else:
        pa = f'transformer.layers.layers.{i}.0.'
        pf = f'transformer.layers.layers.{i}.1.'
    return pa, pf


def layer_params(sd, cfg: OracleConfig, i: int, prefix=''):
    """Pull the tensors of layer i out of a reference-format state dict."""
    pa, pf = _layer_prefixes(cfg, i)
    pa, pf = prefix + pa, prefix + pf
    inner_a = 'fn.fn.fn.fn.fn.' if cfg.shift_tokens else 'fn.fn.fn.'
    inner_f = 'fn.fn.fn.fn.' if cfg.shift_tokens else 'fn.fn.'
    P = dict(
        a_scale=sd[pa + 'scale'], a_ln_w=sd[pa + 'fn.norm.weight'], a_ln_b=sd[pa + 'fn.norm.bias'],
        w_qkv=sd[pa + inner_a + 'to_qkv.weight'], w_out=sd[pa + inner_a + 'to_out.0.weight'],
        b_out=sd[pa + inner_a + 'to_out.0.bias'],
        f_scale=sd[pf + 'scale'], f_ln_w=sd[pf + 'fn.norm.weight'], f_ln_b=sd[pf + 'fn.norm.bias'],
        w1=sd[pf + inner_f + 'net.0.weight'], b1=sd[pf + inner_f + 'net.0.bias'],
        w2=sd[pf + inner_f + 'net.3.weight'], b2=sd[pf + inner_f + 'net.3.bias'],
    )
    if cfg.sandwich_norm:
        P.update(a_lno_w=sd[pa + 'fn.norm_out.weight'], a_lno_b=sd[pa + 'fn.norm_out.bias'],
                 f_lno_w=sd[pf + 'fn.norm_out.weight'], f_lno_b=sd[pf + 'fn.norm_out.bias'])
    return P


# ----------------------------------------------------------------------------------------------
# transformer stack (reversible.py:126-157, transformer.py:279-300)
# ----------------------------------------------------------------------------------------------
def attn_sublayer(x, P, cfg: OracleConfig, kind, angles, allow, key_mask=None, drop_mask=None):
    """LayerScale(PreNorm(PreShiftToken(Attention)))   (transformer.py:279-292, 74-102).  drop_mask (optional, [b,n,d], entries 0
    or 1/(1-p)): the Dropout after to_out (attention.py:53-56) with an explicit mask."""
    y = layer_norm(x, P['a_ln_w'], P['a_ln_b'])
    if cfg.shift_tokens:
        y = token_shift(y, cfg.text_len, cfg.fmap)
    y = attention_core(y, P['w_qkv'], P['w_out'], P['b_out'], cfg.heads, angles, allow, cfg.stable, key_mask)
    if drop_mask is not None:
        y = y * drop_mask
    if cfg.sandwich_norm:
        y = layer_norm(y, P['a_lno_w'], P['a_lno_b'])
    return y * P['a_scale']


def ff_sublayer(x, P, cfg: OracleConfig, drop_mask=None):
    y = layer_norm(x, P['f_ln_w'], P['f_ln_b'])
    if cfg.shift_tokens:
        y = token_shift(y, cfg.text_len, cfg.fmap)
    y = feed_forward(y, P['w1'], P['b1'], P['w2'], P['b2'], drop_mask)
    if cfg.sandwich_norm:
        y = layer_norm(y, P['f_lno_w'], P['f_lno_b'])
    return y * P['f_scale']


def transformer_forward(x, sd, cfg: OracleConfig, prefix='', key_mask=None, causal=True, dropout_masks=None):
    """x [b,n,d] -> [b,n,d].  Sequential: reversible.py:134-141.  Reversible: :149-157 + :60-68
    (forward values only; gradients of the reversible executor equal autograd through this forward,
    which is what reversible.py:70-106 reconstructs)."""
    n = x.shape[1]
    angles = None
    if cfg.rotary_emb:
        angles = rotary_angle_table(cfg.text_len, cfg.fmap, cfg.dim_head, dtype=x.dtype)
    allow_cache = {}

    def allow_for(kind):
        if kind not in allow_cache:
            allow_cache[kind] = allowed_mask(kind, n, n, cfg.text_len, cfg.fmap, causal=causal)
        return allow_cache[kind]

    if cfg.reversible:
        x1, x2 = x, x                                            # cat([x, x], -1) then chunk (reversible.py:150, 61)
    for i in range(cfg.depth):
        P = layer_params(sd, cfg, i, prefix)
        kind = cfg.attn_type_of_layer(i)
        allow = allow_for(kind)
        ma, mf = dropout_masks[i] if dropout_masks is not None else (None, None)   # explicit dropout masks (training with p > 0)
        if cfg.reversible:
            x1 = x1 + attn_sublayer(x2, P, cfg, kind, angles, allow, key_mask, ma)   # y1 = x1 + f(x2)
            x2 = x2 + ff_sublayer(x1, P, cfg, mf)                                     # y2 = x2 + g(y1)
        else:
            x = x + attn_sublayer(x, P, cfg, kind, angles, allow, key_mask, ma)
            x = x + ff_sublayer(x, P, cfg, mf)
    if cfg.reversible:
        return (x1 + x2) / 2                                     # stack(chunk).mean(0) (reversible.py:157)
    return x


# ----------------------------------------------------------------------------------------------
# DALLE wrapper (dalle_pytorch.py:576-671)
# ----------------------------------------------------------------------------------------------
def logits_mask(cfg: OracleConfig, seq_len: int) -> torch.Tensor:
    """dalle_pytorch.py:441-455: True where the logit must be filled with -fp32max."""
    pos = torch.arange(cfg.seq_len)[:, None]
    tok = torch.arange(cfg.total_tokens)[None, :]
    m = ((pos >= cfg.text_seq_len) & (tok < cfg.total_text_tokens)) | \
        ((pos < cfg.text_seq_len) & (tok >= cfg.total_text_tokens))
    return m[:seq_len]


def dalle_forward(text, image, sd, cfg: OracleConfig, return_loss=False, dropout_masks=None):
    """text [b,text_seq_len] int64, image [b, <=fmap^2] int64 token ids (or None).
    Returns logits [b,n,total_tokens] or the scalar loss."""
    assert cfg.rotary_emb, 'oracle restates the rotary_emb=True path (DALLE default, dalle_pytorch.py:372)'
    dtype = sd['to_logits.1.weight'].dtype
    b = text.shape[0]
    # unique padding ids (:595-596), <bos> (:600)
    text_range = torch.arange(cfg.text_seq_len) + (cfg.total_text_tokens - cfg.text_seq_len)
    text = torch.where(text == 0, text_range[None, :], text)
    text = F.pad(text, (1, 0), value=0)
    tokens = sd['text_emb.weight'][text]                                        # :602
    if image is not None and image.numel() > 0:
        tokens = torch.cat([tokens, sd['image_emb.weight'][image]], dim=1)      # :617-623
    if tokens.shape[1] > cfg.seq_len:                                           # :629-631
        tokens = tokens[:, :-1]
    n = tokens.shape[1]
    if cfg.stable:                                                              # :633-635
        tokens = tokens * 0.1 + tokens.detach() * 0.9
    out = transformer_forward(tokens, sd, cfg, dropout_masks=dropout_masks)     # :639
    if cfg.stable:                                                              # :641-642, transformer.py:29-36
        out = out / out.amax(dim=-1, keepdim=True).detach()
    out = layer_norm(out, sd['to_logits.0.weight'], sd['to_logits.0.bias'])     # :644
    logits = out @ sd['to_logits.1.weight'].t() + sd['to_logits.1.bias']
    neg = -torch.finfo(logits.dtype).max
    logits = logits.masked_fill(logits_mask(cfg, n)[None], neg)                 # :648-652
    if not return_loss:
        return logits
    labels = torch.cat([text[:, 1:], image + cfg.total_text_tokens], dim=1)     # :662-663
    lg = logits.permute(0, 2, 1)
    T = cfg.text_seq_len
    loss_text = F.cross_entropy(lg[:, :, :T], labels[:, :T])                    # :667
    loss_img = F.cross_entropy(lg[:, :, T:], labels[:, T:])                     # :668
    return (loss_text + cfg.loss_img_weight * loss_img) / (cfg.loss_img_weight + 1)   # :670


# ----------------------------------------------------------------------------------------------
# deterministic synthetic parameters / inputs shared by goldens, tests and bench
# ----------------------------------------------------------------------------------------------
def layerscale_init(layer_index_1based: int) -> float:
    """transformer.py:75-83."""
    if layer_index_1based <= 18:
        return 0.1
    if layer_index_1based <= 24:
        return 1e-5
    return 1e-6


def make_state_dict(cfg: OracleConfig, seed: int = 0, dtype=torch.float32, perturb: bool = True, fast: bool = False):
    """Deterministic synthetic weights in the reference's state-dict format (App. A.8).

    Same distributions as the reference's default init (nn.Linear kaiming-uniform(a=sqrt 5) ->
    U(-1/sqrt(fan_in), 1/sqrt(fan_in)) for weight and bias; nn.Embedding N(0,1); LayerNorm 1/0;
    LayerScale const) drawn from a private torch.Generator so the values do not depend on module
    construction order.  With perturb=True LayerNorm affine and LayerScale get a small random
    perturbation so that their gradients / broadcasting are exercised by the parity tests."""
    g = torch.Generator().manual_seed(seed)
    d, inner = cfg.dim, cfg.heads * cfg.dim_head
    gen_dtype = torch.float32 if fast else torch.float64      # fast: benchmark-sized models (values differ from the fp64 draw)

    def uni(shape, fan_in):
        bound = 1.0 / (fan_in ** 0.5)
        return ((torch.rand(shape, generator=g, dtype=gen_dtype) * 2 - 1) * bound).to(dtype)

    def ln_w():
        w = torch.ones(d, dtype=torch.float64)
        if perturb:
            w = w + 0.1 * torch.randn(d, generator=g, dtype=torch.float64)
        return w.to(dtype)

    def ln_b():
        w = torch.zeros(d, dtype=torch.float64)
        if perturb:
            w = w + 0.1 * torch.randn(d, generator=g, dtype=torch.float64)
        return w.to(dtype)

    sd = {}
    sd['text_emb.weight'] = torch.randn(cfg.total_text_tokens, d, generator=g, dtype=gen_dtype).to(dtype)
    sd['image_emb.weight'] = torch.randn(cfg.num_image_tokens, d, generator=g, dtype=gen_dtype).to(dtype)
    sd['to_logits.0.weight'], sd['to_logits.0.bias'] = ln_w(), ln_b()
    sd['to_logits.1.weight'] = uni((cfg.total_tokens, d), d)
    sd['to_logits.1.bias'] = uni((cfg.total_tokens,), d)
    sd['transformer.pos_emb'] = rotary_angle_table(cfg.text_len, cfg.fmap, cfg.dim_head)[None].to(dtype)
    inner_a = 'fn.fn.fn.fn.fn.' if cfg.shift_tokens else 'fn.fn.fn.'
    inner_f = 'fn.fn.fn.fn.' if cfg.shift_tokens else 'fn.fn.'
    for i in range(cfg.depth):
        pa, pf = _layer_prefixes(cfg, i)
        s0 = layerscale_init(i + 1)
        for p in (pa, pf):
            sc = torch.full((1, 1, d), s0, dtype=torch.float64)
            if perturb:
                sc = sc * (1 + 0.2 * torch.randn(1, 1, d, generator=g, dtype=torch.float64))
            sd[p + 'scale'] = sc.to(dtype)
            sd[p + 'fn.norm.weight'], sd[p + 'fn.norm.bias'] = ln_w(), ln_b()
            if cfg.sandwich_norm:
                sd[p + 'fn.norm_out.weight'], sd[p + 'fn.norm_out.bias'] = ln_w(), ln_b()
        sd[pa + inner_a + 'to_qkv.weight'] = uni((3 * inner, d), d)
        sd[pa + inner_a + 'to_out.0.weight'] = uni((d, inner), inner)
        sd[pa + inner_a + 'to_out.0.bias'] = uni((d,), inner)
        hid = d * cfg.ff_mult
        sd[pf + inner_f + 'net.0.weight'] = uni((2 * hid, d), d)
        sd[pf + inner_f + 'net.0.bias'] = uni((2 * hid,), d)
        sd[pf + inner_f + 'net.3.weight'] = uni((d, hid), hid)
        sd[pf + inner_f + 'net.3.bias'] = uni((d,), hid)
    return sd


def make_inputs(cfg: OracleConfig, batch: int, seed: int = 1, pad_tail: bool = True):
    """Synthetic token ids (SURVEY.md §8d): text in [1, num_text_tokens), a random zero-padded tail on
    half of the samples (exercises the pad-id remap dalle_pytorch.py:595-596); image ids in [0, 8192)."""
    g = torch.Generator().manual_seed(seed)
    text = torch.randint(1, cfg.num_text_tokens, (batch, cfg.text_seq_len), generator=g)
    if pad_tail:
        for bi in range(0, batch, 2):
            k = int(torch.randint(1, max(2, cfg.text_seq_len // 4), (1,), generator=g))
            text[bi, cfg.text_seq_len - k:] = 0
    image = torch.randint(0, cfg.num_image_tokens, (batch, cfg.image_seq_len), generator=g)
    return text, image


def make_attention_inputs(dim: int, heads: int, dim_head: int, batch: int, n: int, seed: int = 0):
    """Deterministic weights of one attention module (to_qkv.weight, to_out.0.weight, to_out.0.bias; the reference's
    default-init distributions) and its input x [batch, n, dim], from a private torch.Generator."""
    g = torch.Generator().manual_seed(seed)
    inner = heads * dim_head

    def uni(shape, fan_in):
        return (torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1).div(fan_in ** 0.5).float()

    w_qkv, w_out, b_out = uni((3 * inner, dim), dim), uni((dim, inner), inner), uni((dim,), inner)
    return w_qkv, w_out, b_out, torch.randn(batch, n, dim, generator=g, dtype=torch.float64).float()
