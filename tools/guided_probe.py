"""Classifier-free guidance in generate_images(use_cache=True) at the C2 weights (depth 12, dim 1024, 1024 image tokens, bf16) on one
GPU: generated image tokens/s of ONE generate_images call for
    unguided graph replay (cond_scale = 1),
    guided graph replay   (cond_scale = 3, decode.GuidedDecoder: both streams as one batch of 2b),
    guided eager loop     (cond_scale = 3, DALLE_B200_DECODE_GUIDED=0),
at batch 8 and 16; the per-launch time of the small-M GEMM at M = 16 vs M = 32 for the four C2 GEMM shapes of a layer; and a
torch.profiler kernel summary of guided replays at batch 16 (a separate, later pass: profiling slows the host).

    python tools/guided_probe.py --out DIR [--batches 8,16] [--no-eager]

Each timed call is preceded by an untimed call at batch 2 (allocator, weight caches, library modules).  Writes DIR/guided_probe.json.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
import torch

COND_SCALE = 3.0


def gpu_info():
    info = {'device': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = q.stdout.strip()
    except Exception as ex:                                             # the numbers stay valid; the field says why it is missing
        info['power_limit_and_max_sm_clock'] = f'unavailable: {type(ex).__name__}'
    return info


def build_model():
    import bench
    import dalle_pytorch_b200 as D
    c = bench.CONFIGS['c2']
    torch.manual_seed(0)
    vae = D.TokenVAE(image_size=8 * c['fmap'], num_layers=3, num_tokens=bench.NUM_IMAGE_TOKENS)
    m = D.DALLE(dim=c['dim'], vae=vae, num_text_tokens=bench.NUM_TEXT_TOKENS, text_seq_len=c['text_seq_len'], depth=c['depth'],
                heads=c['heads'], dim_head=64, attn_types=c['attn_types']).cuda().eval()
    return m, c, bench.NUM_TEXT_TOKENS, bench.NUM_IMAGE_TOKENS


def time_generate(m, text, cond_scale, guided_graph):
    """(ms of one generate_images call, tokens) with decode.GUIDED_DEFAULT = guided_graph."""
    from dalle_pytorch_b200 import decode
    was = decode.GUIDED_DEFAULT
    decode.GUIDED_DEFAULT = guided_graph
    try:
        with torch.no_grad():
            m.generate_images(text[:2], use_cache=True, cond_scale=cond_scale)
            torch.cuda.synchronize()
            torch.manual_seed(1)
            t0 = time.perf_counter()
            img = m.generate_images(text, use_cache=True, cond_scale=cond_scale)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3
    finally:
        decode.GUIDED_DEFAULT = was
    return ms, img


def small_m_launch_times(reps=20):
    """Per-launch time (us) of the small-M kernel for the C2 GEMMs of a layer at M = 16 and 32.  Twelve distinct weight sets (one per
    C2 layer, 300 MB of bf16 > the 126 MB L2) are swept in turn, so the weights stream from HBM as in a decoding step."""
    from dalle_pytorch_b200 import ops
    d, hid, layers = 1024, 4096, 12
    W = [dict(qkv=torch.randn(3 * d, d, device='cuda').bfloat16(), out=torch.randn(d, d, device='cuda').bfloat16(),
              ff1=torch.randn(2 * hid, d, device='cuda').bfloat16(), ff2=torch.randn(d, hid, device='cuda').bfloat16()) for _ in range(layers)]
    bias_d, bias_h = torch.zeros(d, device='cuda'), torch.zeros(2 * hid, device='cuda')
    res = {}
    for M in (16, 32):
        a = torch.randn(M, d, device='cuda').bfloat16()
        h = torch.randn(M, hid, device='cuda').bfloat16()
        x = torch.randn(M, d, device='cuda')
        scale = torch.ones(d, device='cuda')
        calls = {'qkv store 3072x1024': lambda w: ops.gemm_store(a, w['qkv']),
                 'out-proj resid 1024x1024': lambda w: ops.gemm_resid(a, w['out'], bias_d, x, scale),
                 'ff1 geglu 8192x1024': lambda w: ops.gemm_geglu(a, w['ff1'], bias_h, keep_u=False),
                 'ff2 resid 1024x4096': lambda w: ops.gemm_resid(h, w['ff2'], bias_d, x, scale)}
        res[f'M={M}'] = {}
        with ops.small_m_rows(32):
            for name, fn in calls.items():
                for w in W:                                               # warm-up
                    fn(w)
                ops.gemm_timing(True)
                for _ in range(reps):
                    for w in W:
                        fn(w)
                st = ops.gemm_timing(False)
                assert st['smallm']['launches'] == reps * layers and st['tcgen05']['launches'] == 0, st
                res[f'M={M}'][name] = {'us_per_launch': 1e3 * st['smallm']['ms'] / st['smallm']['launches'],
                                       'weight_GB_per_s': 2 * w_numel(W[0], name) / (1e-3 * st['smallm']['ms'] / st['smallm']['launches']) / 1e9}
    return res


def w_numel(w, name):
    return w[name.split()[0].replace('out-proj', 'out')].numel()


def guided_kernel_summary(m, text, steps=24):
    """torch.profiler over `steps` guided replays at text's batch: device time per kernel name, sorted."""
    from torch.profiler import profile, ProfilerActivity
    from dalle_pytorch_b200 import decode, ops
    with torch.no_grad():
        dev = {}
        logits = decode.guided_prompt(m, text, text[:, :0], dev)
        dec = decode.GuidedDecoder(m, dev)
        ntt = m.num_text_tokens                                          # sampled ids index [text vocab | image vocab]
        tok = ops.sample_guided_topk_gumbel(logits, COND_SCALE, 0.5, 1.0, 0, 0) - ntt
        assert 0 <= int(tok.min()) and int(tok.max()) < m.num_image_tokens
        for i in range(4):                                                # warm-up steps + capture
            logits = dec.step(tok)
            tok = ops.sample_guided_topk_gumbel(logits, COND_SCALE, 0.5, 1.0, 0, i) - ntt
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(steps):
                logits = dec.step(tok)
                tok = ops.sample_guided_topk_gumbel(logits, COND_SCALE, 0.5, 1.0, 0, 100 + i) - ntt
            torch.cuda.synchronize()
    rows = {}
    for e in prof.key_averages():
        t = getattr(e, 'device_time_total', None) or getattr(e, 'cuda_time_total', 0)
        if t > 0 and e.count > 0:
            rows[e.key] = {'launches_per_step': e.count / steps, 'us_per_step': t / steps}
    rows = dict(sorted(rows.items(), key=lambda kv: -kv[1]['us_per_step']))
    return {'steps': steps, 'batch': text.shape[0], 'device_us_per_step': sum(r['us_per_step'] for r in rows.values()), 'kernels': rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True, help='directory for guided_probe.json')
    ap.add_argument('--batches', default='8,16')
    ap.add_argument('--no-eager', action='store_true')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'guided_probe measures on a GPU'
    import dalle_pytorch_b200 as D
    D.set_compute_dtype(torch.bfloat16)
    m, c, ntt, nit = build_model()
    n_img = c['fmap'] ** 2
    out = {'workload': f'c2 weights (depth {c["depth"]}, dim {c["dim"]}), generate_images(use_cache=True): {n_img} image tokens after '
                       f'{c["text_seq_len"]} text tokens, filter_thres 0.5, temperature 1, bf16; cond_scale {COND_SCALE} for the guided legs',
           'unit': 'generated image tokens/s (one generate_images call, host clock around the call ending in a device synchronise)',
           'gpu': gpu_info(), 'batches': {}}
    for b in [int(x) for x in args.batches.split(',')]:
        text = torch.randint(1, ntt, (b, c['text_seq_len']), generator=torch.Generator().manual_seed(5)).cuda()
        legs = {}
        for name, scale, graph in (('unguided_graph', 1.0, True), ('guided_graph', COND_SCALE, True), ('guided_eager_loop', COND_SCALE, False)):
            if name == 'guided_eager_loop' and args.no_eager:
                continue
            ms, img = time_generate(m, text, scale, graph)
            assert img.shape == (b, n_img) and int(img.min()) >= 0 and int(img.max()) < nit
            legs[name] = {'tokens_per_s': b * n_img / (ms / 1e3), 'ms_per_token_step': ms / n_img, 'total_ms': ms}
            print(f'batch {b} {name}: {legs[name]["tokens_per_s"]:.0f} tok/s ({legs[name]["ms_per_token_step"]:.3f} ms/step)', flush=True)
        g = legs['guided_graph']['tokens_per_s']
        legs['guided_graph_over_unguided_graph'] = g / legs['unguided_graph']['tokens_per_s']
        if 'guided_eager_loop' in legs:
            legs['guided_graph_over_guided_eager_loop'] = g / legs['guided_eager_loop']['tokens_per_s']
        out['batches'][str(b)] = legs
    out['small_m_gemm_per_launch'] = small_m_launch_times()
    text = torch.randint(1, ntt, (16, c['text_seq_len']), generator=torch.Generator().manual_seed(5)).cuda()
    out['guided_step_kernels_batch16'] = guided_kernel_summary(m, text)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'guided_probe.json'), 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != 'guided_step_kernels_batch16'}, indent=1))


if __name__ == '__main__':
    main()
