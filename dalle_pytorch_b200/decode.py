"""Graph-replayed KV-cache decoding: one CUDA-graph replay per generated image token.

`generate_images(use_cache=True)` (dalle_pytorch.py:506-562) walks the module nest once per token: ~110 library launches plus the
torch glue of the token-shift cache, all issued from Python -- 5.2 ms of host time per step for well under 1 ms of GPU work at
batch 16.  The step is the same launch sequence for every token; only the POSITION changes, and the eager path feeds it to the
kernels as host integers (rotary row, KV-cache write offset, number of valid keys, static-mask row, token-shift slot).  Here the
position lives in a device tensor `pos_t` and every use of it is a device-side index operation:

    rotary                 cos/sin row = table.index_select(0, pos_t)            (QKV epilogue called with a 1-row table)
    KV cache               k/v buffers .index_copy_(2, pos_t, new row)            (in-place cache of attention.py::_KVCache)
    valid keys / patterns  attention over the WHOLE buffer, non-causal, with a key mask = row pos_t of a [positions, capacity]
                           uint8 table (causal triangle, AND the layer's static mask): masked keys get weight exp(-max) = 0
                           exactly, so the result equals the causal evaluation over the first pos_t+1 keys bit for bit
    token shift            ring buffers [fmap, b, d/4] indexed by (pos_t - text_len) % fmap instead of the deque of
                           transformer.py:155-186
    logits mask            logits_mask.index_select(1, pos_t)

so the whole step (embedding of the previous sample -> transformer -> logits head -> logits mask) is captured ONCE per
`generate_images` call and replayed; the sampling kernel stays outside the graph because its Philox offset is drawn from torch's
generator per step (exactly like the eager path, so the same seed gives the same tokens).  The first step (the prompt) and two
warm-up steps run eagerly through the same code.

Measured on B200 (C2 weights, batch 16, 1024 image tokens, bf16; tools/decode_probe.py, profiles/r02_decode_matrix.txt), generated
tokens/s of one generate_images call:  host-indexed loop 3 186 (5.02 ms per token step) -> graph replay of the module nest 6 296 ->
flat step (FLAT_DEFAULT) 7 953 -> + 256-key buckets (BUCKET_DEFAULT) 8 896 -> + the single-query attention kernel of
csrc/decode.cu 10 444 -> + the small-M weight-streaming GEMM (csrc/gemm_smallm.cu) 13 781 (1.16 ms per step).  One step of the first graph was 364 kernels / 2.84 ms (profiles/r02_decode_step_launches.txt:
29 % attention over the whole buffer on 128-query tiles, 28 % the four M = 16 GEMMs per layer, 32 % torch index glue).

Classifier-free guidance (cond_scale = s != 1, GuidedDecoder): the conditional and the unconditional stream are decoded as ONE batch of
2b sequences -- rows [:b] on the real text, rows [b:] on zeroed text (what DALLE.forward(null_cond_prob=1.) makes of it), each row with
its own cache -- so every weight byte is read once per token for both streams.  The prompt pass is one eager DALLE.forward over the
prefix repeated twice; every later token is one replay of the same step at batch 2b, fed the sampled token in both halves, its GEMMs on
the small-M kernel up to 32 rows (ops.small_m_rows).  dalle_b200_sample_guided_topk_gumbel forms null + (cond - null) * s from the
[2b, V] logits and samples in one launch.  The result is classifier-free guidance as the uncached forward_with_cond_scale defines it
(two independent forwards over the prefix): the eager cached loop instead hands the null pass a shallow copy of the conditional cache.
tools/guided_probe.py times it against the unguided graph and the eager guided loop.

`DALLE_B200_DECODE_GRAPH=0` restores the host-indexed loop (see GRAPH_DEFAULT), `DALLE_B200_DECODE_GUIDED=0` the eager loop for
cond_scale != 1 only; models the path does not cover (reversible executor, sparse-pattern layers that re-run the prefix) use the eager
loop.
"""
import os
from collections import deque

import torch

GRAPH_DEFAULT = os.environ.get('DALLE_B200_DECODE_GRAPH', '1') != '0'
# flat step: the layers are walked by GraphedDecoder itself with the decode kernels (LayerNorm -> dalle_b200_decode_shift -> QKV ->
# dalle_b200_decode_kv_append -> attention -> out-projection with the LayerScale + residual in its epilogue): 11 launches per layer
# instead of the ~30 of the module nest (whose token-shift cache is seven torch index kernels per sub-layer)
FLAT_DEFAULT = os.environ.get('DALLE_B200_DECODE_FLAT', '1') != '0'
# attention reads only the first n_k = roundup(position + 1, BUCKET) rows of the cache; one graph is captured per bucket (0 = always
# the whole buffer, one graph)
BUCKET_DEFAULT = int(os.environ.get('DALLE_B200_DECODE_BUCKET', '256'))
WARMUP_STEPS = 2
# classifier-free guidance (cond_scale != 1) on the graph-replayed path: GuidedDecoder, both streams as one batch of 2b sequences
GUIDED_DEFAULT = os.environ.get('DALLE_B200_DECODE_GUIDED', '1') != '0'


class ShiftRing:
    """Token-shift history of one PreShiftToken module: slot s holds the (top, left) channel quarters of the last image token
    whose index is congruent to s modulo fmap -- the device-indexed form of the deque of transformer.py:155-170."""
    __slots__ = ('top', 'left')

    def __init__(self, top, left):
        self.top, self.left = top, left

    @staticmethod
    def from_deque(q, next_pos, text_len, fmap):
        """q holds the entries of positions next_pos - fmap .. next_pos - 1 (oldest first)."""
        assert isinstance(q, deque) and len(q) == fmap
        top = torch.stack([e[0] for e in q])
        left = torch.stack([e[1] for e in q])
        slots = torch.tensor([(next_pos - text_len + i) % fmap for i in range(fmap)], device=top.device)
        ring_top, ring_left = torch.empty_like(top), torch.empty_like(left)
        ring_top[slots] = top
        ring_left[slots] = left
        return ShiftRing(ring_top.contiguous(), ring_left.contiguous())


def shift_indices(pos_t, text_len, fmap):
    """(slot of the current token, slot of the previous token, "the token is not the first of its row") as device tensors."""
    slot = torch.remainder(pos_t - text_len, fmap)
    return slot, torch.remainder(slot + (fmap - 1), fmap), slot != 0


def allow_table(static_mask, rows, cap, device):
    """uint8 [rows, cap]: entry (p, j) = may the token at position p attend key j when keys 0..p are in the cache
    (causal triangle, AND the layer's static mask attention.py:89-90 when it has one)."""
    j = torch.arange(cap, device=device)
    allow = j[None, :] <= torch.arange(rows, device=device)[:, None]
    if static_mask is not None:
        sm = torch.zeros(rows, cap, dtype=torch.bool, device=device)
        r, c = min(rows, static_mask.shape[0]), min(cap, static_mask.shape[1])
        sm[:r, :c] = static_mask[:r, :c].to(device=device, dtype=torch.bool)
        allow = allow & sm
    return allow.to(torch.uint8).contiguous()


def _attention_layers(model):
    """[(attention module, its cache key)] of every layer, or None when a layer has no in-place KV cache."""
    from .attention import Attention
    from .transformer import CachedAs, PreShiftToken, PreNorm, LayerScale, FeedForward
    from .reversible import SequentialSequence
    tr = model.transformer
    if not isinstance(tr.layers, SequentialSequence) or tr.pos_emb is None:
        return None
    found = []
    for pair in tr.layers.layers:
        for ls in pair:
            if not isinstance(ls, LayerScale) or not isinstance(ls.fn, PreNorm):
                return None
            inner = ls.fn.fn
            if isinstance(inner, CachedAs) and isinstance(inner.fn, PreShiftToken):
                inner = inner.fn.fn
            if isinstance(inner, FeedForward):
                continue
            if not (isinstance(inner, CachedAs) and type(inner.fn) is Attention):
                return None
            found.append((inner.fn, inner.cache_key))
    return found


class _FlatSub:
    __slots__ = ('kind', 'ln', 'shift_key', 'mod', 'scale', 'attn_key')


def _flat_plan(model):
    """The sub-layers of the stack resolved to (LayerNorm, token-shift cache key, Attention | FeedForward, LayerScale vector), or
    None when the flat step does not cover the model (sandwich norm, channel count not a multiple of 4)."""
    from .attention import Attention
    from .transformer import CachedAs, PreShiftToken, FeedForward
    if _attention_layers(model) is None:
        return None
    plan = []
    for pair in model.transformer.layers.layers:
        for ls in pair:
            pre = ls.fn
            if pre.sandwich or pre.norm.weight.shape[0] % 4:
                return None
            r = _FlatSub()
            r.ln, r.scale, r.shift_key, r.attn_key = pre.norm, ls.scale, None, None
            inner = pre.fn
            if isinstance(inner, CachedAs) and isinstance(inner.fn, PreShiftToken):
                r.shift_key = inner.cache_key
                inner = inner.fn.fn
            if isinstance(inner, FeedForward):
                r.kind, r.mod = 'ff', inner
            else:
                assert isinstance(inner, CachedAs) and type(inner.fn) is Attention
                r.kind, r.mod, r.attn_key = 'attn', inner.fn, inner.cache_key
            plan.append(r)
    return plan


def eligible(model, text, cond_scale):
    """May generate_images(use_cache=True, cond_scale=cond_scale) decode through GraphedDecoder (cond_scale == 1) or GuidedDecoder?"""
    return bool(text.is_cuda and _attention_layers(model) is not None)


class GraphedDecoder:
    """Takes over the cache of an eager `DALLE.forward(..., cache=cache)` prompt pass and produces the logits of every following
    position with one graph replay per token:  logits = dec.step(previous_sample)  ([b] int64 image-token ids -> [b, total_tokens])."""

    def __init__(self, model, cache):
        from .attention import rotary_tables, _KVCache
        from .transformer import PreShiftToken
        self.model, self.cache = model, cache
        attn = _attention_layers(model)
        assert attn is not None and cache.get('offset'), 'GraphedDecoder: run the prompt through DALLE.forward(cache=cache) first'
        dev = model.logits_mask.device
        pos = int(cache['offset'])
        self.pos_t = torch.tensor([pos], device=dev, dtype=torch.int64)
        ent0 = cache[attn[0][1]]
        assert isinstance(ent0, _KVCache)
        self.batch, cap = ent0.k.shape[0], ent0.k.shape[2]
        self.cos, self.sin = rotary_tables(model.transformer.pos_emb, attn[0][0].dim_head)
        rows = min(self.cos.shape[0], cap)
        # one allowed-key table per distinct static mask (None = plain causal)
        self.allow, self.allow_key, masks = {}, {}, []
        for mod, key in attn:
            ent = cache[key]
            assert isinstance(ent, _KVCache) and ent.k.shape[2] == cap and mod.dim_head == attn[0][0].dim_head
            sm = mod.static_mask
            tkey = None
            if sm is not None:           # layers of the same pattern carry equal masks: one table per distinct mask
                tkey = next((t for t, s in masks if s.shape == sm.shape and torch.equal(s, sm)), None)
                if tkey is None:
                    tkey = len(masks)
                    masks.append((tkey, sm))
            if tkey not in self.allow:
                self.allow[tkey] = allow_table(sm, rows, cap, dev)
            self.allow_key[key] = tkey
        # token-shift deques -> rings
        self.shift = None
        for mod in model.transformer.modules():
            if isinstance(mod, PreShiftToken):
                self.shift = (mod.text_len, mod.image_size)
                break
        if self.shift is not None:
            for key in [k for k, v in cache.items() if isinstance(v, deque)]:
                cache[key] = ShiftRing.from_deque(cache[key], pos, *self.shift)
        self.tok = torch.zeros(self.batch, device=dev, dtype=torch.int64)
        self.logits = None
        self.graph, self.graphs = None, {}
        self.warm = 0
        self.cap, self.n_k, self.bucket = cap, None, BUCKET_DEFAULT
        self.plan = _flat_plan(model) if FLAT_DEFAULT else None
        cache['pos_t'] = self.pos_t          # marks the cache as device-indexed for PreShiftToken / Attention

    def _step(self):
        m, cache, pos = self.model, self.cache, self.pos_t
        if self.shift is not None:
            cache['shift_idx'] = shift_indices(pos, *self.shift)
        cache['rot_row'] = (self.cos.index_select(0, pos), self.sin.index_select(0, pos))
        nk = self.cap if self.n_k is None else self.n_k
        km = {tkey: tab.index_select(0, pos)[:, :nk].expand(self.batch, -1).contiguous() for tkey, tab in self.allow.items()}
        cache['key_mask'] = {key: km[tkey] for key, tkey in self.allow_key.items()}
        cache['n_k'] = self.n_k
        tokens = m.image_emb(self.tok[:, None])
        if m.stable:
            alpha = 0.1
            tokens = tokens * alpha + tokens.detach() * (1 - alpha)
        out = self._flat_layers(tokens) if self.plan is not None else m.transformer(tokens, cache=cache)
        if m.stable:
            out = m.norm_by_max(out)
        logits = m.to_logits(out)
        logits = logits.masked_fill(m.logits_mask.index_select(1, pos), -torch.finfo(logits.dtype).max)[:, -1]
        if self.logits is None:
            self.logits = torch.empty_like(logits)
        self.logits.copy_(logits)
        pos.add_(1)

    def _flat_layers(self, tokens):
        """The transformer stack for one token per sequence, sub-layer by sub-layer on the library kernels (see FLAT_DEFAULT)."""
        from . import ops, config
        from .functional import _w
        from ._lib import ATTN_FULL
        cache, b = self.cache, self.batch
        dtype = config.compute_dtype()
        x = tokens.reshape(b, -1).float().contiguous()
        d = x.shape[1]
        cos_r, sin_r = cache['rot_row']
        for r in self.plan:
            ln = r.ln
            if r.shift_key is not None:
                h, _, _ = ops.ln_shift_fwd(x.view(1, b, d), ln.weight, ln.bias, torch.float32, 0, 1, do_ln=True, do_shift=False, eps=ln.eps)
                ring = cache[r.shift_key]
                a = ops.decode_shift(h, ring.top, ring.left, self.pos_t, self.shift[0], self.shift[1], dtype)
            else:
                a, _, _ = ops.ln_shift_fwd(x.view(1, b, d), ln.weight, ln.bias, dtype, 0, 1, do_ln=True, do_shift=False, eps=ln.eps)
            sc = r.scale.detach().reshape(-1).contiguous()
            if r.kind == 'attn':
                m = r.mod
                ent = cache[r.attn_key]
                q, k, v = ops.gemm_qkv(a, _w(m.to_qkv.weight, dtype), b, 1, m.heads, m.dim_head, cos_r, sin_r, m.scale, pos_offset=0)
                ops.decode_kv_append(k, v, ent.k, ent.v, self.pos_t)
                o, _ = ops.attn_fwd(ops.AttnSpec(ATTN_FULL, causal=False, stable=m.stable), q, ent.k, ent.v, cache['key_mask'][r.attn_key],
                                    n_k=self.n_k)
                x, _ = ops.gemm_resid(o.view(b, -1), _w(m.to_out[0].weight, dtype), m.to_out[0].bias.detach(), x, sc, 1.0)
            else:
                f = r.mod
                hh, _ = ops.gemm_geglu(a, _w(f.net[0].weight, dtype), f.net[0].bias.detach(), keep_u=False)
                x, _ = ops.gemm_resid(hh, _w(f.net[3].weight, dtype), f.net[3].bias.detach(), x, sc, 1.0)
        return x.view(b, 1, d)

    def step(self, sample):
        """sample: [b] image-token ids of the position just generated -> logits [b, total_tokens] of the next position."""
        self.tok.copy_(sample)
        if self.bucket > 0:                                  # keys this token can see, rounded up to the bucket
            nk = min(self.cap, -(-(int(self.cache['offset']) + 1) // self.bucket) * self.bucket)
            if nk != self.n_k:
                self.n_k, self.graph = nk, self.graphs.get(nk)
        if self.graph is None and self.warm < WARMUP_STEPS:
            self._step()                                     # eager: allocator, weight-copy and autocast caches, cuBLAS handles
            self.warm += 1
        else:
            if self.graph is None:
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._step()
                self.graph = self.graphs[self.n_k] = g
            self.graph.replay()
        self.cache['offset'] += 1
        return self.logits


def guided_prompt(model, text, image, cache):
    """Prompt pass of guided decoding: one DALLE.forward of the prefix for 2b sequences (rows [:b] with the text, rows [b:] with zeroed
    text, the image prefix in both) that fills `cache` for all of them -> [2b, V] logits of the last position."""
    return model(torch.cat((text, torch.zeros_like(text))), torch.cat((image, image)), cache=cache)[:, -1]


class GuidedDecoder(GraphedDecoder):
    """GraphedDecoder over the 2b-sequence cache of guided_prompt: step(sample) feeds the [b] sampled tokens to both halves and returns
    the [2b, V] logits (conditional rows first).  The step's GEMMs of up to 32 rows run on the small-M kernel."""

    def step(self, sample):
        from . import ops
        with ops.small_m_rows(32):
            return super().step(sample.repeat(2))


def sample_guided(logits, cond_scale, filter_thres, temperature):
    """[2b, V] logits (conditional rows, then unconditional) -> [b] tokens of null + (cond - null) * cond_scale, consuming the random
    numbers of the eager loop: the draw of DALLE.forward(null_cond_prob=1.) (prob_mask_like), then the sampling draw -- so a seed gives
    the tokens of generate_images(use_cache=False, cond_scale=cond_scale)."""
    from . import ops
    from .dalle import prob_mask_like, top_k, gumbel_sample
    from .functional import DropoutRNG
    b, V = logits.shape[0] // 2, logits.shape[1]
    prob_mask_like((b,), 1., device=logits.device)
    if logits.is_cuda and V * 4 <= 200 * 1024:
        seed, off = DropoutRNG.draw(b * V)
        return ops.sample_guided_topk_gumbel(logits.contiguous(), cond_scale, filter_thres, temperature, seed, off)
    null = logits[b:]
    guided = null + (logits[:b] - null) * cond_scale
    return gumbel_sample(top_k(guided, thres=filter_thres), temperature=temperature, dim=-1)
