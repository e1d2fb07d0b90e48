"""DALLE wrapper with the reference's constructor / forward / generate_images signatures and state-dict keys
(reference dalle_pytorch/dalle_pytorch.py:353-671).  Embedding lookup, the logits head and the weighted
cross-entropy are thin PyTorch glue around the transformer stack, which is the hot path (SURVEY.md §8a a10, §8f-1).
"""
import torch
from torch import nn
import torch.nn.functional as F

from .transformer import Transformer, DivideMax
from . import ops, decode
from .functional import DropoutRNG


def exists(val):
    return val is not None


def default(val, d):
    return val if exists(val) else d


def is_empty(t):
    return t.nelement() == 0


def prob_mask_like(shape, prob, device):
    return torch.zeros(shape, device=device).float().uniform_(0, 1) < prob


def set_requires_grad(model, value):
    for param in model.parameters():
        param.requires_grad = value


def eval_decorator(fn):
    def inner(model, *args, **kwargs):
        was_training = model.training
        model.eval()
        out = fn(model, *args, **kwargs)
        model.train(was_training)
        return out
    return inner


def top_k(logits, thres=0.5):
    """dalle_pytorch.py:63-69"""
    num_logits = logits.shape[-1]
    k = max(int((1 - thres) * num_logits), 1)
    val, ind = torch.topk(logits, k)
    probs = torch.full_like(logits, float('-inf'))
    probs.scatter_(1, ind, val)
    return probs


def gumbel_sample(t, temperature=1., dim=-1):
    """dalle_pytorch.py:53-61"""
    noise = torch.zeros_like(t).uniform_(0, 1)
    g = -torch.log((-torch.log(noise.clamp(min=1e-20))).clamp(min=1e-20))
    return ((t / temperature) + g).argmax(dim=dim)


class always:
    def __init__(self, val):
        self.val = val

    def __call__(self, x, *args, **kwargs):
        return self.val


class TokenVAE(nn.Module):
    """Metadata carrier standing in for the reference's DiscreteVAE / OpenAIDiscreteVAE / VQGanVAE when images are
    supplied as token ids (dalle_pytorch.py:608-615 bypasses the VAE in that case; the conv VAEs are out of scope,
    SURVEY.md §2 rows 5 and 7).  Any object exposing image_size / num_layers / num_tokens is accepted by DALLE."""

    def __init__(self, image_size=256, num_layers=3, num_tokens=8192, channels=3):
        super().__init__()
        self.image_size, self.num_layers, self.num_tokens, self.channels = image_size, num_layers, num_tokens, channels

    def get_codebook_indices(self, images):
        raise NotImplementedError('TokenVAE carries geometry only; pass image token ids or plug a real VAE')

    def decode(self, img_seq):
        raise NotImplementedError('TokenVAE carries geometry only; pass a real VAE to decode image tokens')


class SharedEmbedding(nn.Embedding):
    """dalle_pytorch.py:71-83"""

    def __init__(self, linear, start_index, end_index, **kwargs):
        super().__init__(end_index - start_index, linear.weight.shape[1], **kwargs)
        del self.weight
        self.linear = linear
        self.start_index = start_index
        self.end_index = end_index

    def forward(self, input):
        return F.embedding(input, self.linear.weight[self.start_index:self.end_index], self.padding_idx, self.max_norm,
                           self.norm_type, self.scale_grad_by_freq, self.sparse)


class DALLE(nn.Module):
    def __init__(self, *, dim, vae, num_text_tokens=10000, text_seq_len=256, depth, heads=8, dim_head=64, reversible=False,
                 attn_dropout=0., ff_dropout=0, sparse_attn=False, attn_types=None, loss_img_weight=7, stable=False,
                 sandwich_norm=False, shift_tokens=True, rotary_emb=True, shared_attn_ids=None, shared_ff_ids=None,
                 share_input_output_emb=False, optimize_for_inference=False):
        super().__init__()
        for attr in ('image_size', 'num_layers', 'num_tokens'):
            assert hasattr(vae, attr), f'vae must expose `{attr}` (DiscreteVAE-like object)'
        num_image_tokens = vae.num_tokens
        image_fmap_size = vae.image_size // (2 ** vae.num_layers)
        image_seq_len = image_fmap_size ** 2
        num_text_tokens = num_text_tokens + text_seq_len         # unique padding token per position

        if not rotary_emb:
            raise NotImplementedError('rotary_emb=False needs the un-vendored axial_positional_embedding package; the DALLE '
                                      'default (rotary_emb=True, dalle_pytorch.py:372) is the supported path')
        self.text_pos_emb = always(0)
        self.image_pos_emb = always(0)

        self.num_text_tokens = num_text_tokens
        self.num_image_tokens = num_image_tokens
        self.text_seq_len = text_seq_len
        self.image_seq_len = image_seq_len
        seq_len = text_seq_len + image_seq_len
        total_tokens = num_text_tokens + num_image_tokens
        self.total_tokens = total_tokens
        self.total_seq_len = seq_len

        self.vae = vae
        if isinstance(vae, nn.Module):
            set_requires_grad(self.vae, False)

        self.transformer = Transformer(dim=dim, causal=True, seq_len=seq_len, depth=depth, heads=heads, dim_head=dim_head,
                                       reversible=reversible, attn_dropout=attn_dropout, ff_dropout=ff_dropout, attn_types=attn_types,
                                       image_fmap_size=image_fmap_size, sparse_attn=sparse_attn, stable=stable,
                                       sandwich_norm=sandwich_norm, shift_tokens=shift_tokens, rotary_emb=rotary_emb,
                                       shared_attn_ids=shared_attn_ids, shared_ff_ids=shared_ff_ids,
                                       optimize_for_inference=optimize_for_inference)
        self.stable = stable
        if stable:
            self.norm_by_max = DivideMax(dim=-1)

        self.to_logits = nn.Sequential(nn.LayerNorm(dim), nn.Linear(dim, self.total_tokens))

        if share_input_output_emb:
            self.text_emb = SharedEmbedding(self.to_logits[1], 0, num_text_tokens)
            self.image_emb = SharedEmbedding(self.to_logits[1], num_text_tokens, total_tokens)
        else:
            self.text_emb = nn.Embedding(num_text_tokens, dim)
            self.image_emb = nn.Embedding(num_image_tokens, dim)

        seq_range = torch.arange(seq_len)[None, :, None]
        logits_range = torch.arange(total_tokens)[None, None, :]
        logits_mask = (((seq_range >= text_seq_len) & (logits_range < num_text_tokens)) |
                       ((seq_range < text_seq_len) & (logits_range >= num_text_tokens)))
        self.register_buffer('logits_mask', logits_mask, persistent=False)
        self.loss_img_weight = loss_img_weight

    # ---- sampling (dalle_pytorch.py:506-574) -----------------------------------------------------------
    @torch.no_grad()
    @eval_decorator
    def generate_images(self, text, *, clip=None, filter_thres=0.5, temperature=1., img=None, num_init_img_tokens=None,
                        cond_scale=1., use_cache=False):
        vae, text_seq_len, image_seq_len, num_text_tokens = self.vae, self.text_seq_len, self.image_seq_len, self.num_text_tokens
        total_len = text_seq_len + image_seq_len
        text = text[:, :text_seq_len]
        out = text
        if exists(img):
            image_size = vae.image_size
            assert img.shape[1] == 3 and img.shape[2] == image_size and img.shape[3] == image_size, \
                f'input image must have the correct image size {image_size}'
            indices = vae.get_codebook_indices(img)
            num_img_tokens = default(num_init_img_tokens, int(0.4375 * image_seq_len))
            assert num_img_tokens < image_seq_len, 'number of initial image tokens for priming must be less than the total image token sequence length'
            out = torch.cat((out, indices[:, :num_img_tokens]), dim=-1)

        cache = {} if use_cache else None
        # graph-replayed steps (decode.py): after the prompt pass every image token is one CUDA-graph replay + the sampling launch
        graph_ok = use_cache and decode.GRAPH_DEFAULT and decode.eligible(self, text, cond_scale)
        # classifier-free guidance on that path: the conditional and the unconditional stream as one batch of 2b sequences
        guided = graph_ok and cond_scale != 1
        if guided and not decode.GUIDED_DEFAULT:
            graph_ok = guided = False
        stepper, sample = None, None
        for cur_len in range(out.shape[1], total_len):
            is_image = cur_len >= text_seq_len
            if graph_ok and stepper is None and cur_len > text_seq_len and cache.get('offset') == cur_len:
                stepper = decode.GuidedDecoder(self, cache) if guided else decode.GraphedDecoder(self, cache)
            if stepper is not None:
                logits = stepper.step(sample)
            elif guided:
                logits = decode.guided_prompt(self, out[:, :text_seq_len], out[:, text_seq_len:], cache)
            else:
                text, image = out[:, :text_seq_len], out[:, text_seq_len:]
                logits = self.forward_with_cond_scale(text, image, cond_scale=cond_scale, cache=cache)
                logits = logits[:, -1, :]
            if guided:
                sample = decode.sample_guided(logits, cond_scale, filter_thres, temperature)
            elif logits.is_cuda and logits.shape[-1] * 4 <= 200 * 1024:
                # top_k + gumbel_sample (dalle_pytorch.py:533-539) as one library launch; the Philox pair follows torch's generator
                seed, off = DropoutRNG.draw(logits.numel())
                sample = ops.sample_topk_gumbel(logits.contiguous(), filter_thres, temperature, seed, off)
            else:
                filtered_logits = top_k(logits, thres=filter_thres)
                sample = gumbel_sample(filtered_logits, temperature=temperature, dim=-1)
            sample -= (num_text_tokens if is_image else 0)
            out = torch.cat((out, sample[:, None]), dim=-1)

        text_seq = out[:, :text_seq_len]
        img_seq = out[:, -image_seq_len:]
        self.last_image_tokens = img_seq
        images = vae.decode(img_seq) if not isinstance(vae, TokenVAE) else img_seq
        if exists(clip):
            scores = clip(text_seq, images, return_loss=False)
            return images, scores
        return images

    def forward_with_cond_scale(self, *args, cond_scale=1, cache=None, **kwargs):
        if cond_scale == 1:
            return self(*args, cache=cache, **kwargs)
        prev_cache = cache.copy() if exists(cache) else None
        logits = self(*args, cache=cache, **kwargs)
        null_cond_logits = self(*args, null_cond_prob=1., cache=prev_cache, **kwargs)
        return null_cond_logits + (logits - null_cond_logits) * cond_scale

    # ---- training / scoring forward (dalle_pytorch.py:576-671) -----------------------------------------
    def forward(self, text, image=None, return_loss=False, null_cond_prob=0., cache=None):
        assert text.shape[-1] == self.text_seq_len, \
            f'the length {text.shape[-1]} of the text tokens you passed in does not have the correct length ({self.text_seq_len})'
        batch, device, total_seq_len = text.shape[0], text.device, self.total_seq_len

        if null_cond_prob > 0:
            null_mask = prob_mask_like((batch,), null_cond_prob, device=device)
            text = text * (~null_mask)[:, None]

        text_range = torch.arange(self.text_seq_len, device=device) + (self.num_text_tokens - self.text_seq_len)
        text = torch.where(text == 0, text_range, text)
        text = F.pad(text, (1, 0), value=0)                      # <bos>

        # library path (plain nn.Embedding tables on the GPU): both lookups and the concatenation are one gather each into the
        # [b, n, d] token buffer, and the table gradients are atomic scatter-adds (functional.EmbedTokensFn)
        fused_embed = (text.is_cuda and type(self.text_emb) is nn.Embedding and type(self.image_emb) is nn.Embedding
                       and self.text_emb.weight.dtype == torch.float32 and self.text_emb.weight.shape[1] % 4 == 0
                       and self.text_emb.padding_idx is None and self.text_emb.max_norm is None)
        img_ids = None
        image_len = 0
        if exists(image) and not is_empty(image):
            if len(image.shape) == 4:
                image_size = self.vae.image_size
                channels = self.vae.channels
                assert tuple(image.shape[1:]) == (channels, image_size, image_size), \
                    f'invalid image of dimensions {image.shape} passed in during training'
                image = self.vae.get_codebook_indices(image)
            image_len = image.shape[1]
            # dalle_pytorch.py:627-630 embeds every image token and then drops the last position when the sequence is one too
            # long; embedding only the tokens that survive gives the same tensor without a strided slice + 84 MB copy
            drop = 1 if text.shape[1] + image_len > total_seq_len else 0
            img_ids = image[:, :image_len - drop] if drop else image
            image_len -= drop
        if fused_embed:
            from .functional import EmbedTokensFn
            # (ids are not range-checked on the host -- that would be a device sync per step; the kernels never index outside
            #  the tables: an out-of-range id reads row 0 and receives no gradient)
            tokens = EmbedTokensFn.apply(text.contiguous(), None if img_ids is None else img_ids.contiguous(),
                                         self.text_emb.weight, self.image_emb.weight)
        else:
            tokens = self.text_emb(text)
            if img_ids is not None:
                tokens = torch.cat((tokens, self.image_emb(img_ids)), dim=1)
        seq_len = text.shape[1] + image_len

        if tokens.shape[1] > total_seq_len:
            seq_len -= 1
            tokens = tokens[:, :-1]

        if self.stable:
            alpha = 0.1
            tokens = tokens * alpha + tokens.detach() * (1 - alpha)

        if exists(cache) and cache.get('offset'):
            tokens = tokens[:, -1:]
        out = self.transformer(tokens, cache=cache)

        if self.stable:
            out = self.norm_by_max(out)

        if return_loss:
            assert exists(image), 'when training, image must be supplied'
            return self._loss_head(out, text, image, seq_len)

        logits = self.to_logits(out)

        logits_mask = self.logits_mask[:, :seq_len]
        if exists(cache) and cache.get('offset'):
            logits_mask = logits_mask[:, -1:]
        max_neg_value = -torch.finfo(logits.dtype).max
        logits = logits.masked_fill(logits_mask, max_neg_value)

        if exists(cache):
            cache['offset'] = cache.get('offset', 0) + logits.shape[1]
        return logits

    def _loss_head(self, out, text, image, seq_len):
        """Logits head + weighted cross-entropy of dalle_pytorch.py:644-671 without materialising the masked
        [b, n, total_tokens] logits: the logits mask (dalle_pytorch.py:441-455) fills every image-vocabulary logit of a text
        position (and vice versa) with -fp32max, whose softmax weight is exactly 0, so the text loss only needs the
        text-vocabulary columns at the text positions and the image loss only the image-vocabulary columns at the image
        positions — the same numbers with 2.1x fewer head FLOPs and no [b, c, n] transposed softmax."""
        ln, lin = self.to_logits[0], self.to_logits[1]
        T, ntt = self.text_seq_len, self.num_text_tokens
        n_img_ = seq_len - T
        if out.is_cuda and ntt % 8 == 0 and self.num_image_tokens % 8 == 0 and out.shape[-1] % 8 == 0:
            # library path: LayerNorm + both vocabulary GEMMs + cross-entropy as kernels (functional.HeadLossFn)
            from .functional import HeadLossFn
            from . import config
            d_ = out.shape[-1]
            x2 = torch.cat((out[:, :T].reshape(-1, d_), out[:, T:seq_len].reshape(-1, d_)), dim=0).float()
            return HeadLossFn.apply(x2, ln.weight, ln.bias, lin.weight, lin.bias, text[:, 1:T + 1].reshape(-1).contiguous(),
                                    image[:, :n_img_].reshape(-1).contiguous(), ntt, float(self.loss_img_weight),
                                    config.compute_dtype(), ln.eps)
        h = ln(out)
        labels_text = text[:, 1:]                                  # text already carries <bos> at index 0
        d = h.shape[-1]
        h_text = h[:, :T].reshape(-1, d)
        logits_text = F.linear(h_text, lin.weight[:ntt], lin.bias[:ntt])
        loss_text = F.cross_entropy(logits_text.float(), labels_text[:, :T].reshape(-1))
        n_img = seq_len - T
        h_img = h[:, T:seq_len].reshape(-1, d)
        logits_img = F.linear(h_img, lin.weight[ntt:], lin.bias[ntt:])
        loss_img = F.cross_entropy(logits_img.float(), image[:, :n_img].reshape(-1))
        return (loss_text + self.loss_img_weight * loss_img) / (self.loss_img_weight + 1)
