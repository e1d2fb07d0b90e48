"""bench.py — DALL-E fwd+bwd tokens/sec (BASELINE.json metric) on N x B200, and the reference arm on the host CPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2|c3|c4|c1] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = `loss = dalle(text, image_ids, return_loss=True); loss.backward()` on one synthetic batch (reference
call-site contract train_dalle.py:609-616), gradients zeroed every step, for N>1 followed by the flat NCCL gradient
all-reduce (dalle_pytorch_b200.distributed).  Prints ONE JSON line (rank 0).

  value   tokens/s with the token-id inputs already resident in HBM
  e2e     tokens/s through the public module API with HOST (pinned) token buffers: H2D copy of the ids and a D2H read of
          the loss inside every timed step
  roofline  the tcgen05 GEMM family (dominant kernel): algorithmic FLOPs of every launch / CUDA-event time of those
          launches inside the timed region, against MEASURED_PEAKS.json bf16_tflops_sustained
  cpu_baseline  the UNMODIFIED reference (oracle/_ref, its own DALLE(...) API) on the host cores, on a bounded sample (batch 1
          of the same configuration, best of a few thread counts); the oracle port only if the reference cannot be imported
  gpu_eager_baseline  the same unmodified reference module on cuda:0 with torch's eager kernels under bf16 autocast, same batch --
          the practical GPU baseline
  extra_configs  BASELINE.json configs[2], [3] (one GPU) / configs[4] (eight GPUs) timed in the same run
`--impl reference` times the unmodified reference on the host CPU for K steps of a batch-1 sample of the configuration.
`--dump-outputs DIR` writes what the headline step returned in its last timed step (see output_snapshot) so that two builds can be
compared output for output: weights and token ids come from fixed seeds, so the inputs are the same on every run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # BASELINE.json configs[1..3]; c1 = configs[0] (the reference's CPU-runnable case)
    'c1': dict(dim=256, depth=2, heads=4, text_seq_len=64, fmap=8, batch=2, attn_types=('full',), reversible=False, dtype='fp32'),
    'c2': dict(dim=1024, depth=12, heads=16, text_seq_len=256, fmap=32, batch=16, attn_types=('full',), reversible=False, dtype='bf16'),
    'c3': dict(dim=1024, depth=12, heads=16, text_seq_len=256, fmap=32, batch=16, attn_types=('axial_row', 'axial_col'), reversible=False, dtype='bf16'),
    'c4': dict(dim=1024, depth=12, heads=16, text_seq_len=256, fmap=32, batch=64, attn_types=('axial_row', 'axial_col'), reversible=True, dtype='bf16'),
    'c5': dict(dim=1024, depth=64, heads=16, text_seq_len=256, fmap=32, batch=32, attn_types=('axial_row', 'axial_col'), reversible=False, dtype='bf16'),
}
NUM_TEXT_TOKENS, NUM_IMAGE_TOKENS = 10000, 8192
# measured with ncu on B200 (profiles/r01_gemm_ncu_summary.txt): mean dram__bytes_read+write of 20 consecutive tcgen05 GEMM launches
# of a C2 step (algorithmic operand+result bytes of the same launches: 226 MB per launch)
GEMM_DRAM_BYTES_PER_LAUNCH = 229e6
METRIC = 'DALL-E fwd+bwd tokens/sec at seq=1280, dim=1024'
DUMP_BYTES = 60 * 2 ** 20      # gradient samples of --dump-outputs; with the .npy headers and the loss the files stay below 64 MB


def log(msg):
    print(f'[bench {time.strftime("%H:%M:%S")}] {msg}', file=sys.stderr, flush=True)


def usable_cores():
    """Host threads this process may actually use: the affinity mask capped by the cgroup CPU quota (a container that sees
    200 cores but is limited to 8 must not spawn 200 threads)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
        if quota != 'max':
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
            per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                n = max(1, min(n, int(q / per + 0.5)))
        except Exception:
            pass
    return n


def workload_name(name, c):
    return (f"{name}: depth={c['depth']} dim={c['dim']} heads={c['heads']} text_seq={c['text_seq_len']} image={c['fmap']}x{c['fmap']} "
            f"attn={'+'.join(c['attn_types'])}{' reversible' if c['reversible'] else ''} batch/GPU={c['batch']}")


# ------------------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region.  NVML (nvidia_ml_py) polled every 10 ms from a thread -- the
    timed region of a default run is a few hundred ms, too short for `nvidia-smi -lms` to deliver a sample reliably (its start-up
    alone can take longer on an 8-GPU box); nvidia-smi is the fallback when NVML cannot be loaded."""
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
    REASONS = ((0x8, 'hw_slowdown'), (0x40, 'hw_thermal_slowdown'), (0x20, 'sw_thermal_slowdown'), (0x4, 'sw_power_cap'))

    def __init__(self, gpu_index=0):
        self.proc, self.lines, self.gpu_index = None, [], gpu_index
        self.nvml, self.samples, self.stop_flag, self.t = None, [], False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.gpu_index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '200',
                                          '-i', str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1e3
                try:
                    rs = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((float(sm), float(pw), int(rs)))
            except Exception:
                pass
            time.sleep(0.01)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=2)
            if not self.samples:
                return {'sm_mhz': None, 'sm_max_mhz': float(self.max_sm), 'reasons': ['no samples']}
            sm = sorted(x[0] for x in self.samples)
            bits = 0
            for x in self.samples:
                bits |= x[2]
            return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(self.max_sm), 'power_w_max': max(x[1] for x in self.samples),
                    'samples': len(sm), 'source': 'nvml, 10 ms period', 'reasons': sorted(name for bit, name in self.REASONS if bits & bit)}
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(',')]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': max(mx), 'power_w_max': max(pw), 'samples': len(sm), 'source': 'nvidia-smi -lms 200',
                'reasons': sorted(reasons)}


# ------------------------------------------------------------------------------------------------------------
# Reference legs: the UNMODIFIED reference (oracle/_ref, built by oracle/build_ref.py; imported through oracle/ref_import.py with
# the dependency shims under oracle/shims) driven through its own public API -- DALLE(...)(text, image, return_loss=True);
# loss.backward() (train_dalle.py:609-616).  If the reference cannot be imported the oracle port is timed instead and the
# line says kind = "port".
# ------------------------------------------------------------------------------------------------------------
def _thread_candidates():
    cores = usable_cores()
    return sorted({c for c in (16, 32, cores) if 1 <= c <= cores} or {cores})


def ref_step_fn(cfg_name, sample_batch, device='cpu', autocast=False):
    """-> (step() -> loss float, tokens per step, kind).  kind = 'reference' (stock DALLE) or 'port' (oracle restatement)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    c = CONFIGS[cfg_name]
    seq = c['text_seq_len'] + c['fmap'] ** 2
    g = torch.Generator().manual_seed(1)
    text = torch.randint(1, NUM_TEXT_TOKENS, (sample_batch, c['text_seq_len']), generator=g).to(device)
    image = torch.randint(0, NUM_IMAGE_TOKENS, (sample_batch, c['fmap'] ** 2), generator=g).to(device)
    try:
        import ref_import
        ref = ref_import.import_reference()
        torch.manual_seed(0)
        vae = ref.DiscreteVAE(image_size=8 * c['fmap'], num_layers=3, num_tokens=NUM_IMAGE_TOKENS, codebook_dim=64, hidden_dim=8)
        model = ref.DALLE(dim=c['dim'], vae=vae, num_text_tokens=NUM_TEXT_TOKENS, text_seq_len=c['text_seq_len'], depth=c['depth'],
                          heads=c['heads'], dim_head=64, attn_types=c['attn_types'], reversible=c['reversible']).to(device).train()

        def step():
            for p in model.parameters():
                p.grad = None
            with torch.autocast(device_type='cuda' if device != 'cpu' else 'cpu', dtype=torch.bfloat16, enabled=autocast):
                loss = model(text, image, return_loss=True)
            loss.backward()
            return loss

        return step, sample_batch * seq, 'reference'
    except Exception as ex:
        if device != 'cpu':
            raise
        log(f'reference import failed ({type(ex).__name__}: {ex}); timing the oracle port instead')
    from dalle_oracle import OracleConfig, make_state_dict, dalle_forward
    cfg = OracleConfig(dim=c['dim'], depth=c['depth'], heads=c['heads'], text_seq_len=c['text_seq_len'], fmap=c['fmap'],
                       num_text_tokens=NUM_TEXT_TOKENS, num_image_tokens=NUM_IMAGE_TOKENS, attn_types=c['attn_types'],
                       reversible=c['reversible'])
    sd = make_state_dict(cfg, seed=0, perturb=False, fast=True)
    params = {k: v.requires_grad_(k != 'transformer.pos_emb') for k, v in sd.items()}

    def step():
        for p in params.values():
            p.grad = None
        loss = dalle_forward(text, image, params, cfg, return_loss=True)
        loss.backward()
        return loss

    return step, sample_batch * seq, 'port'


def pick_threads(step):
    """One untimed + one timed step per candidate thread count; returns (best count, {count: seconds}).  All visible cores is
    often NOT the fastest (r01: 96 threads were slower than 16 on the 8-GPU box)."""
    import torch
    seen = {}
    for t in _thread_candidates():
        torch.set_num_threads(t)
        if not seen:
            step()                      # first-touch / allocator warm-up
        t0 = time.perf_counter()
        step()
        seen[t] = time.perf_counter() - t0
    best = min(seen, key=seen.get)
    torch.set_num_threads(best)
    return best, seen


def run_cpu_sample(args):
    """`--cpu-sample`: a bounded CPU sample (batch 1 of the configuration, best thread count, up to 3 timed steps or ~25 s) of
    the reference; prints {"value", "cores", "seconds", "kind", ...} (called as a subprocess with a hard timeout by the GPU arm
    so that a slow host can never stall the bench)."""
    step, tokens, kind = ref_step_fn(args.config, 1)
    best, seen = pick_threads(step)
    n, t0 = 0, time.perf_counter()
    while n < 3 and (n == 0 or time.perf_counter() - t0 < 25.0):
        step()
        n += 1
    dt = (time.perf_counter() - t0) / n
    print(json.dumps({'value': tokens / dt, 'cores': best, 'seconds': dt, 'tokens': tokens, 'kind': kind, 'steps': n,
                      'threads_tried': {str(k): round(v, 3) for k, v in seen.items()}}))


def run_gpu_eager_sample(args):
    """`--gpu-eager-sample`: the unmodified reference module on cuda:0, torch eager kernels, bf16 autocast, the configuration's
    own batch (halved on out-of-memory) -- the practical GPU baseline SURVEY.md §8(d) asks for."""
    import torch
    c = CONFIGS[args.config]
    batch = args.batch or c['batch']
    while True:
        try:
            step, tokens, kind = ref_step_fn(args.config, batch, device='cuda', autocast=True)
            for _ in range(2):
                step()
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n = 5
            s.record()
            for _ in range(n):
                step()
            e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e) / n
            print(json.dumps({'value': tokens / (ms * 1e-3), 'unit': 'tokens/s', 'ms_per_step': ms, 'batch': batch, 'steps': n,
                              'peak_mem_gb': torch.cuda.max_memory_allocated() / 2 ** 30,
                              'impl': 'unmodified reference DALLE on cuda:0 (torch eager, bf16 autocast, fp32 master weights)'}))
            return
        except torch.OutOfMemoryError:
            step = None
            torch.cuda.empty_cache()
            if batch == 1:
                raise
            batch //= 2


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    c = CONFIGS[args.config]
    step, tokens, kind = ref_step_fn(args.config, 1)
    cores, seen = pick_threads(step)
    for _ in range(max(0, args.warmup - 2)):          # pick_threads already ran >= 2 steps
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = tokens * args.steps / dt
    what = ('unmodified reference DALLE (oracle/_ref) through its public API' if kind == 'reference'
            else 'oracle port of the reference (oracle/dalle_oracle.py)')
    sample = (f'{what}: each step = fwd+bwd on a bounded sample, batch 1 of the configuration\'s {c["batch"]} ({tokens} tokens), full '
              f'depth, fp32, torch CPU with {cores} threads (best of {sorted(seen)})')
    wl = workload_name(args.config, c).replace(f"batch/GPU={c['batch']}", f"batch={c['batch']} (CPU arm timed on a batch-1 sample)")
    out = {'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'tokens/s', 'n_gpus': args.gpus, 'steps': args.steps,
           'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
           'dtype': 'f32', 'data': 'synthetic', 'config': {'workload': wl, 'sample_batch': 1, 'seq_len': tokens},
           'cpu_baseline': {'value': val, 'unit': 'tokens/s', 'cores': cores, 'kind': kind, 'sample': sample},
           'e2e': {'value': val, 'unit': 'tokens/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------
def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        j = json.load(open(p))
        return j.get('bf16_tflops_sustained', 1405.9), j.get('hbm_gbs', 6567.4), 'measured (MEASURED_PEAKS.json, sustained)'
    return 1400.0, 6650.0, 'fallback (B200_PROFILING.md)'


def model_flops_per_token(c):
    """SURVEY.md §8(d) model FLOPs per token (fwd+bwd = 3x fwd; masked pairs and recompute not counted; the head counts only the
    live half of the vocabulary each position class can predict -- the masked half is never computed)."""
    d = c['dim']
    pairs = {'full': 819840, 'axial_row': 312928, 'axial_col': 312928}
    attn_flops = sum(4096.0 * pairs.get(t, 819840) / 1280 * (c['heads'] / 16) for t in c['attn_types']) / len(c['attn_types'])
    seq = c['text_seq_len'] + c['fmap'] ** 2
    n_text_pos, n_img_pos = c['text_seq_len'], c['fmap'] ** 2
    head = 2.0 * d * (n_text_pos * (NUM_TEXT_TOKENS + c['text_seq_len']) + n_img_pos * NUM_IMAGE_TOKENS) / seq
    return 3 * (c['depth'] * (32.0 * d * d + attn_flops) + head)


def named_grads(model):
    return [(k, p.grad) for k, p in model.named_parameters() if p.grad is not None]


def output_snapshot(loss, grads):
    """What a caller of one fwd+bwd step receives, on the host: the loss (float64) and every parameter gradient (float32).  A
    gradient larger than its share of DUMP_BYTES is a sample at fixed flat indices (seeded by the parameter name, sorted)."""
    import zlib
    import torch
    cap = DUMP_BYTES // 4 // max(1, len(grads))
    out = {'loss': loss.detach().double().cpu().numpy()}
    for k, g in grads:
        f = g.detach().reshape(-1)
        if f.numel() > cap:
            idx = torch.randperm(f.numel(), generator=torch.Generator().manual_seed(zlib.crc32(k.encode())))[:cap].sort().values
            f = f[idx.to(f.device)]
        out['grad.' + k] = f.float().cpu().numpy()
    return out


def dump_outputs(out_dir, arrays):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)
    log(f'dumped {len(arrays)} arrays ({sum(a.nbytes for a in arrays.values()) / 2 ** 20:.1f} MB) to {out_dir}')


def measure_config(cfg_name, args, ctx, steps, want_e2e=True, want_clocks=True, batch=None, dtype_name=None):
    """Builds the configuration's model, warms up, times `steps` fwd+bwd steps device-resident (per-GEMM CUDA events on) and,
    optionally, end to end from host token buffers.  Returns a dict of raw measurements; the model is freed before returning."""
    import gc
    import torch
    import torch.distributed as dist
    import dalle_pytorch_b200 as D
    from dalle_pytorch_b200 import ops
    world, rank, dev, backend = ctx['world'], ctx['rank'], ctx['dev'], ctx['backend']
    c = CONFIGS[cfg_name]
    batch = batch or c['batch']
    dtype = {'fp32': torch.float32, 'bf16': torch.bfloat16}[dtype_name or c['dtype']]
    D.set_compute_dtype(dtype)
    torch.manual_seed(0)
    vae = D.TokenVAE(image_size=8 * c['fmap'], num_layers=3, num_tokens=NUM_IMAGE_TOKENS)
    kw = dict(dim=c['dim'], vae=vae, num_text_tokens=NUM_TEXT_TOKENS, text_seq_len=c['text_seq_len'], depth=c['depth'],
              heads=c['heads'], dim_head=64, attn_types=c['attn_types'], reversible=c['reversible'])
    try:
        with torch.device(dev):      # parameters are created on the GPU (depth 64 = 1.1 B parameters)
            model = D.DALLE(**kw)
    except Exception as ex:
        log(f'{cfg_name}: construction under torch.device({dev}) failed ({type(ex).__name__}); building on the CPU')
        model = D.DALLE(**kw)
    model = model.to(dev).train()
    reducer = None
    if backend is not None and os.environ.get('DALLE_B200_BENCH_NO_ALLREDUCE') != '1':      # (=1: N independent replicas, diagnosis only)
        backend.distribute(model=model)
        reducer = model.grad_reducer
    seq = c['text_seq_len'] + c['fmap'] ** 2
    g = torch.Generator().manual_seed(1 + rank)
    text_h = torch.randint(1, NUM_TEXT_TOKENS, (batch, c['text_seq_len']), generator=g).pin_memory()
    image_h = torch.randint(0, NUM_IMAGE_TOKENS, (batch, c['fmap'] ** 2), generator=g).pin_memory()
    text_d, image_d = text_h.to(dev), image_h.to(dev)
    head_autocast = dtype == torch.bfloat16
    dump = args.dump_outputs is not None and cfg_name == args.config and rank == 0
    graph_leg = world == 1 and not args.no_graph
    last = {}

    def zero():
        if reducer is not None:
            reducer.zero_grad()
        else:
            for p in model.parameters():
                p.grad = None

    def fwd_bwd(text, image):
        zero()
        with torch.autocast('cuda', dtype=torch.bfloat16, enabled=head_autocast):
            loss = model(text, image, return_loss=True)
        loss.backward()
        if reducer is not None:
            reducer.finish()
        if dump:
            last['loss'] = loss.detach()      # detached: a kept autograd graph would break the CUDA-graph capture that follows
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(n):
            fn()
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    log(f'{cfg_name}: model built ({sum(p.numel() for p in model.parameters()) / 1e6:.1f} M params); warm-up')
    for i in range(max(args.warmup, 3)):
        t0 = time.perf_counter()
        fwd_bwd(text_d, image_d)
        torch.cuda.synchronize()
        log(f'{cfg_name}: warm-up step {i}: {1e3 * (time.perf_counter() - t0):.1f} ms')

    sampler = ClockSampler(ctx['local_rank'])
    if rank == 0 and want_clocks:
        sampler.start()
    ops.gemm_timing(True)
    n0 = ops.launches()
    ms_dev = timed(lambda: fwd_bwd(text_d, image_d), steps)
    launches = ops.launches() - n0
    gemm_stats = ops.gemm_timing(False)
    clocks = sampler.stop() if (rank == 0 and want_clocks) else None
    outputs = None
    if dump:
        # only the path that becomes the headline is copied out: the eager step when no graph leg follows (now, before later steps
        # reuse the data-parallel gradient buffers), otherwise the references are kept until the graph leg is timed.  They stay the
        # eager step's values because GraphedStep._zero and the e2e steps' zero() set p.grad = None (fresh tensors afterwards)
        # instead of zeroing the old ones in place; a change to in-place zeroing there must snapshot here instead.
        eager_out = (last['loss'], named_grads(model))
        if not graph_leg:
            outputs = output_snapshot(*eager_out)
    log(f'{cfg_name}: device-resident {ms_dev / steps:.2f} ms/step')
    res = {'cfg': cfg_name, 'c': c, 'batch': batch, 'seq': seq, 'dtype': dtype, 'ms_dev': ms_dev, 'steps': steps, 'launches': launches,
           'gemm_stats': gemm_stats, 'clocks': clocks, 'peak_mem_gb': torch.cuda.max_memory_allocated() / 2 ** 30,
           'h2d': int(text_h.numel() * 8 + image_h.numel() * 8), 'outputs': outputs}
    if dtype == torch.bfloat16 and gemm_stats['simt']['launches'] != 0:
        raise RuntimeError(f"{cfg_name}: {gemm_stats['simt']['launches']} GEMM launches fell back to the fp32 CUDA-core kernel in bf16 mode "
                           '(mis-aligned operand?) -- the measured step is not the tcgen05 path')
    if want_e2e:
        def e2e_step():
            t = text_h.to(dev, non_blocking=True)
            i = image_h.to(dev, non_blocking=True)
            return fwd_bwd(t, i).item()

        e2e_step()
        res['ms_e2e'] = timed(e2e_step, steps)
        log(f"{cfg_name}: e2e {res['ms_e2e'] / steps:.2f} ms/step")
    # ---- the same step captured into ONE CUDA graph and replayed (single process): no Python / ctypes between the kernels ----
    if graph_leg:
        try:
            step = D.GraphedStep(model, text_d, image_d, autocast_bf16=head_autocast)
            for _ in range(2):
                step()
            ms_g = timed(lambda: step(), steps)
            if dump and ms_g <= ms_dev:                     # run_gpu_arm's headline rule: the replay when it is not slower
                res['outputs'] = output_snapshot(step.loss, named_grads(model))
            g = {'ms_dev': ms_g, 'kernels_per_step': step.kernels_per_step}
            if want_e2e:
                def e2e_graph():
                    return step(text_h, image_h).item()          # H2D copies of the ids into the static buffers, replay, D2H of the loss

                e2e_graph()
                g['ms_e2e'] = timed(e2e_graph, steps)
            res['graph'] = g
            log(f"{cfg_name}: CUDA-graph replay {ms_g / steps:.2f} ms/step ({step.kernels_per_step} library kernels per step)"
                + (f", e2e {g['ms_e2e'] / steps:.2f}" if 'ms_e2e' in g else ''))
            del step
        except Exception as ex:
            log(f'{cfg_name}: CUDA-graph capture failed ({type(ex).__name__}: {str(ex)[:200]}); eager numbers stand')
            res['graph'] = {'error': f'{type(ex).__name__}: {str(ex)[:200]}'}
            torch.cuda.synchronize()
    if dump and res['outputs'] is None:                     # the eager step is the headline
        res['outputs'] = output_snapshot(*eager_out)
    if args.with_optimizer and cfg_name == args.config:
        # full training step of the reference trainer (train_dalle.py:609-619): fwd + bwd + clip_grad_norm_(0.5) + Adam
        opt = D.FusedAdam(model.parameters(), lr=3e-4, max_grad_norm=0.5, reducer=reducer)

        def train_step():
            with torch.autocast('cuda', dtype=torch.bfloat16, enabled=head_autocast):
                loss = model(text_d, image_d, return_loss=True)
            loss.backward()
            opt.step()

        for _ in range(3):
            train_step()
        res['ms_train'] = timed(train_step, steps)
        log(f"{cfg_name}: train step (fwd+bwd+clip+Adam) {res['ms_train'] / steps:.2f} ms/step")
        del opt
    if reducer is not None:
        reducer.remove()
    del model, reducer
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    return res


def measure_decode(args, ctx, cfg_name='c2', batch=16, host_indexed=True):
    """Autoregressive image generation with the KV cache (generate_images(use_cache=True), dalle_pytorch.py:506-562): image tokens
    per second on one GPU -- cached attention over the in-place KV cache, library sampling kernel, one token per step."""
    import gc
    import torch
    import dalle_pytorch_b200 as D
    from dalle_pytorch_b200 import ops
    dev = ctx['dev']
    c = CONFIGS[cfg_name]
    D.set_compute_dtype(torch.bfloat16)
    torch.manual_seed(0)
    vae = D.TokenVAE(image_size=8 * c['fmap'], num_layers=3, num_tokens=NUM_IMAGE_TOKENS)
    model = D.DALLE(dim=c['dim'], vae=vae, num_text_tokens=NUM_TEXT_TOKENS, text_seq_len=c['text_seq_len'], depth=c['depth'], heads=c['heads'],
                    dim_head=64, attn_types=c['attn_types']).to(dev).eval()
    g = torch.Generator().manual_seed(5)
    text = torch.randint(1, NUM_TEXT_TOKENS, (batch, c['text_seq_len']), generator=g).to(dev)
    n_img = c['fmap'] ** 2
    from dalle_pytorch_b200 import decode

    def timed(graph):
        """One full generate_images call: (ms, library launches per token step)."""
        was, decode.GRAPH_DEFAULT = decode.GRAPH_DEFAULT, graph
        try:
            with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16):
                model.generate_images(text[:2], use_cache=True)          # warm-up (allocator, caches)
                torch.cuda.synchronize()
                n0 = ops.launches()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                img = model.generate_images(text, use_cache=True)
                e.record()
                torch.cuda.synchronize()
        finally:
            decode.GRAPH_DEFAULT = was
        assert img.shape == (batch, n_img) and int(img.min()) >= 0 and int(img.max()) < NUM_IMAGE_TOKENS
        return s.elapsed_time(e), (ops.launches() - n0) / n_img

    legs, ms_host = {}, float('inf')
    if host_indexed:
        ms_host, k_host = timed(False)
        legs['host_indexed'] = {'value': batch * n_img / (ms_host / 1e3), 'ms_per_token_step': ms_host / n_img,
                                'library_launches_per_token_step': k_host}
    ms = ms_host
    try:      # decode.py: one CUDA-graph replay per token (position on the device); includes the capture of the call's graph
        ms_graph, k_graph = timed(True)
        legs['graph_replay'] = {'value': batch * n_img / (ms_graph / 1e3), 'ms_per_token_step': ms_graph / n_img,
                                'library_launches_issued_from_python_per_token_step': k_graph}
        ms = min(ms_host, ms_graph)
    except Exception as ex:                                              # keep the leg: the host-indexed loop is the fallback path
        legs['graph_replay'] = {'error': f'{type(ex).__name__}: {ex}'[:300]}
        if not host_indexed:
            raise
    out = {'workload': f'{cfg_name} weights, generate_images(use_cache=True): {n_img} image tokens after {c["text_seq_len"]} text tokens, batch {batch}, '
                       'filter_thres 0.5, temperature 1, bf16',
           'value': batch * n_img / (ms / 1e3), 'unit': 'generated image tokens/s', 'ms_per_token_step': ms / n_img, 'total_ms': ms,
           'paths': legs, 'default_path': 'graph_replay' if decode.GRAPH_DEFAULT else 'host_indexed', 'n_gpus': 1,
           'graph_step': {'flat_layers': decode.FLAT_DEFAULT, 'key_bucket': decode.BUCKET_DEFAULT,
                          'single_query_attention_kernel': os.environ.get('DALLE_B200_DECODE_ATTN', 'default')}}
    log(f"decode: {out['value']:.0f} image tokens/s ({out['ms_per_token_step']:.3f} ms per step of {batch} sequences; "
        + ', '.join(f"{k} {v['value']:.0f}" if 'value' in v else f'{k} FAILED' for k, v in legs.items()) + ')')
    del model
    gc.collect()
    torch.cuda.empty_cache()
    return out


def leg_summary(res, world, peak_tf):
    """Compact per-configuration entry for `extra_configs`."""
    c = res['c']
    tokens = res['batch'] * res['seq'] * world * res['steps']
    graphed = 'ms_dev' in res.get('graph', {}) and res['graph']['ms_dev'] <= res['ms_dev']     # the faster of the two execution paths
    value = tokens / ((res['graph']['ms_dev'] if graphed else res['ms_dev']) / 1e3)
    fam = res['gemm_stats']['tcgen05']
    flops_tok = model_flops_per_token(c)
    out = {'workload': workload_name(res['cfg'], c), 'value': value, 'unit': 'tokens/s',
           'ms_per_step': (res['graph']['ms_dev'] if graphed else res['ms_dev']) / res['steps'],
           'execution': 'one CUDA-graph replay per step' if graphed else 'eager launches',
           'eager_ms_per_step': res['ms_dev'] / res['steps'],
           'graph_ms_per_step': (res['graph']['ms_dev'] / res['steps']) if 'ms_dev' in res.get('graph', {}) else None,
           'steps': res['steps'], 'n_gpus': world, 'gpu_launches': res['launches'], 'peak_mem_gb': res['peak_mem_gb'],
           'mfu_vs_sustained_peak': value / world * flops_tok / 1e12 / peak_tf,
           'gemm_roofline_frac': (fam['flops'] / (fam['ms'] * 1e-3) / 1e12 / peak_tf) if fam['ms'] > 0 else None,
           'simt_gemm_launches': res['gemm_stats']['simt']['launches']}
    if 'ms_e2e' in res:
        out['e2e'] = {'value': tokens / (res['ms_e2e'] / 1e3), 'unit': 'tokens/s', 'h2d_bytes_per_step': res['h2d'] * world, 'd2h_bytes_per_step': 4 * world}
    if c['reversible']:
        out['note'] = 'reversible: the backward recomputes every block (4/3 of the block FLOPs); MFU counts model FLOPs only'
    return out


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from dalle_pytorch_b200.distributed import NCCLBackend

    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    assert world == args.gpus or world == 1, f'--gpus {args.gpus} but WORLD_SIZE={world}'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    backend = None
    if world > 1:
        backend = NCCLBackend()
        backend.initialize()
    ctx = {'world': world, 'rank': rank, 'local_rank': local_rank, 'dev': dev, 'backend': backend}

    main_res = measure_config(args.config, args, ctx, args.steps, want_e2e=True, batch=args.batch, dtype_name=args.dtype)
    # the other BASELINE.json configurations as extra legs of the same run (configs[2], [3] on one GPU; configs[4] -- the one the
    # multi-GPU metric is written for, depth 64, 32 samples per GPU -- when all 8 GPUs are present)
    extras = []
    if args.extra is not None:
        extras = [e for e in args.extra.split(',') if e]
    elif args.config == 'c2' and not args.batch and not args.dtype:
        extras = ['c3', 'c4'] if world == 1 else (['c5'] if world == 8 else [])
    extra_res = []
    for name in extras:
        try:
            extra_res.append(measure_config(name, args, ctx, min(args.steps, 5), want_e2e=False, want_clocks=False))
        except Exception as ex:          # an extra leg must never cost the headline line
            log(f'extra leg {name} failed: {type(ex).__name__}: {ex}')
            extra_res.append({'cfg': name, 'error': f'{type(ex).__name__}: {ex}'})
            torch.cuda.empty_cache()

    decode = None
    if world == 1 and args.extra is None and args.config == 'c2' and not args.batch and not args.dtype:
        try:
            decode = measure_decode(args, ctx)
        except Exception as ex:
            log(f'decode leg failed: {type(ex).__name__}: {ex}')
            decode = {'error': f'{type(ex).__name__}: {str(ex)[:200]}'}
            torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
        if rank != 0:
            dist.destroy_process_group()
    if rank != 0:
        return

    c, batch, seq, dtype = main_res['c'], main_res['batch'], main_res['seq'], main_res['dtype']
    ms_eager, ms_e2e_eager, gemm_stats = main_res['ms_dev'], main_res['ms_e2e'], main_res['gemm_stats']
    gr = main_res.get('graph', {})
    graphed = 'ms_dev' in gr and gr['ms_dev'] <= ms_eager
    # headline = the product's execution path: the captured step when the capture succeeded and is not slower, eager otherwise
    ms_dev = gr['ms_dev'] if graphed else ms_eager
    ms_e2e = gr.get('ms_e2e', ms_e2e_eager) if graphed else ms_e2e_eager
    if args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, main_res['outputs'])
    tokens_per_step = batch * seq * world
    value = tokens_per_step * args.steps / (ms_dev / 1e3)
    e2e_value = tokens_per_step * args.steps / (ms_e2e / 1e3)
    peak_tf, peak_bw, peak_src = peaks()
    fam = gemm_stats.get('tcgen05', {'flops': 0.0, 'ms': 0.0, 'launches': 0})
    if fam['ms'] > 0:
        ach = fam['flops'] / (fam['ms'] * 1e-3) / 1e12
        roof = {'bound': 'tensor', 'kernel': 'gemm_tcgen05_kernel (all fwd/dgrad/wgrad GEMMs of the block stack)', 'achieved': ach,
                'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': ach / peak_tf, 'traffic': GEMM_DRAM_BYTES_PER_LAUNCH if args.config == 'c2' else None,
                'traffic_note': 'dram__bytes_read+write per launch, mean of the 20 consecutive GEMM launches (last forward layer, head, first backward layer) of the ncu --set full capture summarised in profiles/r01_gemm_ncu_summary.txt; algorithmic bytes of the same 20 launches average 226 MB',
                'peak_source': peak_src,
                'launches_per_step': fam['launches'] / args.steps, 'share_of_step': fam['ms'] / ms_eager,
                'timing_note': 'per-GEMM CUDA events are taken in the eager pass of the same run (events cannot be read back from inside a graph replay); share_of_step is relative to the eager step',
                'simt_gemm_launches': gemm_stats['simt']['launches'],
                'by_shape': gemm_stats.get('by_shape', {})}
    else:
        fam = gemm_stats.get('simt', {'flops': 0.0, 'ms': 0.0, 'launches': 0})
        ach = fam['flops'] / (fam['ms'] * 1e-3) / 1e12 if fam['ms'] > 0 else 0.0
        roof = {'bound': 'tensor', 'kernel': 'gemm_simt_kernel (fp32 FFMA path)', 'achieved': ach, 'peak': peak_tf, 'unit': 'TFLOP/s',
                'frac': ach / peak_tf, 'traffic': None, 'peak_source': peak_src, 'share_of_step': fam['ms'] / ms_eager if ms_eager else None}

    def sub(flag, limit, extra_args=()):
        r = subprocess.run([sys.executable, os.path.abspath(__file__), flag, '--config', args.config, *extra_args], capture_output=True,
                           text=True, timeout=limit, env={**os.environ, **({'CUDA_VISIBLE_DEVICES': ''} if flag == '--cpu-sample' else {})})
        try:
            return json.loads(r.stdout.strip().splitlines()[-1])
        except Exception:
            raise RuntimeError((r.stderr or r.stdout or 'no output')[-300:])

    cpu = eager = None
    if world == 1 and not args.no_cpu_baseline:
        log('gpu_eager_baseline: the unmodified reference module on cuda:0 (subprocess, 300 s limit)')
        try:
            eager = sub('--gpu-eager-sample', 300, ('--batch', str(batch)))
            eager['speedup_of_this_repo'] = value / eager['value']
        except Exception as ex:
            eager = {'value': None, 'unit': 'tokens/s', 'error': f'{type(ex).__name__}: {str(ex)[-200:]}'}
        log('cpu_baseline: the reference on the host cores (subprocess, 420 s limit)')
        what = f'batch 1 of {batch} ({seq} tokens), full depth, fwd+bwd, fp32'
        try:
            j = sub('--cpu-sample', 420)
            src = 'unmodified reference DALLE (oracle/_ref)' if j['kind'] == 'reference' else 'oracle/dalle_oracle.py (port)'
            cpu = {'value': j['value'], 'unit': 'tokens/s', 'cores': j['cores'], 'kind': j['kind'],
                   'sample': f"{j['steps']} step(s) on {what}, {src} on {j['cores']} torch threads ({j['seconds']:.1f} s/step; tried {j['threads_tried']})"}
        except Exception as ex:   # timeout / parse failure: report the failure, keep the GPU numbers
            cpu = {'value': None, 'unit': 'tokens/s', 'cores': usable_cores(), 'kind': 'reference', 'sample': what + f' — not completed: {type(ex).__name__}'}

    flops_tok = model_flops_per_token(c)
    out = {'metric': METRIC, 'value': value, 'unit': 'tokens/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
           'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
           'dtype': 'bf16' if dtype == torch.bfloat16 else 'f32', 'data': 'synthetic',
           'config': {'workload': workload_name(args.config, c), 'global_batch': batch * world, 'seq_len': seq,
                      'parallelism': f'dp{world}', 'l2': 'activations and weights per step (GBs) exceed the 126 MB L2; no flush needed',
                      'head': 'token embedding gather/scatter, block stack, logits head GEMMs and cross-entropy all run in libdalle_b200'},
           'e2e': {'value': e2e_value, 'unit': 'tokens/s', 'ms_per_step': ms_e2e / args.steps,
                   'h2d_bytes_per_step': main_res['h2d'] * world, 'd2h_bytes_per_step': 4 * world},
           'gpu_launches': (gr['kernels_per_step'] * args.steps) if graphed else main_res['launches'],
           'execution': ({'mode': 'cuda_graph', 'host_launches_per_step': 1, 'library_kernels_per_step': gr['kernels_per_step'],
                          'eager_ms_per_step': ms_eager / args.steps, 'eager_e2e_ms_per_step': ms_e2e_eager / args.steps}
                         if graphed else {'mode': 'eager', 'library_kernels_per_step': main_res['launches'] / args.steps,
                                          **({'graph_error': gr['error']} if 'error' in gr else {}),
                                          **({'graph_ms_per_step': gr['ms_dev'] / args.steps} if 'ms_dev' in gr else {})}),
           'model_tflops_per_gpu': value / world * flops_tok / 1e12,
           'mfu_vs_sustained_peak': value / world * flops_tok / 1e12 / peak_tf,
           'clocks': main_res['clocks'], 'roofline': roof}
    if cpu is not None:
        out['cpu_baseline'] = cpu
    if eager is not None:
        out['gpu_eager_baseline'] = eager
    if extra_res:
        out['extra_configs'] = {r['cfg']: (leg_summary(r, world, peak_tf) if 'error' not in r else r) for r in extra_res}
    if decode is not None:
        out.setdefault('extra_configs', {})['decode_c2'] = decode
    if 'ms_train' in main_res:
        out['train_step'] = {'ms_per_step': main_res['ms_train'] / args.steps, 'tokens_per_s': tokens_per_step * args.steps / (main_res['ms_train'] / 1e3),
                             'optimizer': 'FusedAdam lr=3e-4 betas=(0.9,0.999) clip_grad_norm 0.5 (2 launches over flat fp32 buffers)'}
    print(json.dumps(out))
    sys.stdout.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='c2', choices=sorted(CONFIGS))
    ap.add_argument('--batch', type=int, default=None)
    ap.add_argument('--dtype', default=None, choices=['fp32', 'bf16'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='time the eager step only (no CUDA-graph capture)')
    ap.add_argument('--with-optimizer', action='store_true',
                    help='also time fwd+bwd+FusedAdam(clip 0.5) steps and report them under "train_step" (headline metric unchanged)')
    ap.add_argument('--extra', default=None,
                    help='comma-separated extra configurations timed in the same run and reported under "extra_configs" '
                         "(default: c3,c4 on one GPU, c5 on eight; '' = none)")
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the loss and (sampled) parameter gradients of the last step of the headline '
                         'path as DIR/<name>.npy (float64 loss, float32 gradients, < 64 MB in all)')
    ap.add_argument('--cpu-sample', action='store_true', help=argparse.SUPPRESS)
    ap.add_argument('--gpu-eager-sample', action='store_true', help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.cpu_sample:
        run_cpu_sample(args)
    elif args.gpu_eager_sample:
        run_gpu_eager_sample(args)
    elif args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_gpu_arm(args)
        try:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()
        except Exception:
            pass


if __name__ == '__main__':
    main()
