"""bench.py -- captions/sec of the GIT captioning hot path (BASELINE.json metric).

A "step" is ONE `model(batch)` call of the reference surface on synthetic pixels with random-init weights of the named size:
CLIP-ViT encoder -> visual projection -> image-row prefill of the 6 decoder layers -> KV-cached decode steps (max_len 40) ->
search, i.e. the reference's `CaptioningModel.forward` in eval mode (reference layers/decoder.py:838-877, 977-1011).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|3|4|5] [--impl reference] [--dump-outputs DIR]

--config names the BASELINE.json configuration (default 2 = the one the metric is quoted on):
  2  GIT_BASE,        64 images per call,            greedy   (BASELINE.json configs[1])
  3  GIT_LARGE,       32 images per call,            beam 4   (configs[2]; 128 decoder rows, image K/V shared by the beams)
  4  GIT_BASE_VATEX,  16 videos x 6 frames per call, greedy   (configs[3]; 1182 image tokens per video)
  5  GIT_LARGE,       a 1024-image shard per GPU (8192 images on 8 GPUs) in micro-batches of 64, greedy (configs[4]);
                      one step = one pass over the rank's shard, ending with ONE all_gather of the finished captions.

Numbers of a run (all with every call's full work inside the timed region):
  value   : captions/s of K back-to-back `model(batch)` calls, pixels resident in HBM -- the metric as SURVEY.md section 8d
            defines it (one call at a time, the reference's calling pattern); `median_ms_per_step` is the median call.
  e2e     : the same calls with pinned HOST pixels in and token ids / logprobs read back to the host in every step.
  serving : (configs 2-4) the engine's asynchronous form `model.submit(batch, depth, coalesce)`: `coalesce` submitted batches
            share one engine launch, `depth` launches are in flight (dynamic batching: a serving technique, reported
            beside the per-call metric, never in place of it).  It times K steps too: with K below depth * coalesce (8 for
            configs 2 and 4 at the defaults) the pipeline never fills, so serving figures compare only at the same K.
Multi-GPU (torchrun, one rank per GPU): every rank captions its own batches (weak scaling, image-wise sharding, reference
inference.py:165-169); the timed region ends with ONE fused NCCL all_gather of all finished token ids + logprobs.
`--dump-outputs DIR` writes what the last timed `value` step returned on rank 0 (its own shard, not the gathered
captions) -- the token ids (float64, EOS-padded to 40 columns) and logprobs (float32) of its model(batch) calls -- as
DIR/predictions.npy and DIR/logprobs.npy.  With `--impl reference` it writes the last timed CPU step instead: its
`cpu_sample` images only, token ids not padded.  Weights and pixels are seeded, so two builds run with the same
arguments can be compared output for output; the two arms' dumps are not the same images.
`--impl reference` times the reference's own CPU algorithm (the as-shipped, no-KV-cache restatement in
oracle/git_oracle.py -- the Python reference itself cannot travel to the GPU box) on the host cores.
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

UNIT = 'captions/s'
MAX_STEPS = 40
LARGE = {'visual_feature_size': 1024, 'image_encoder_type': 'CLIPViT_L_14'}
CONFIGS = {
    2: dict(metric='captions/sec (greedy, max_len=40) GIT_BASE batch64', model='GIT_BASE', param={}, batch=64, frames=0,
            search='greedy', cpu_sample=4, enc=dict(g=14, p=16, d=768, layers=12, L=197)),
    3: dict(metric='captions/sec (beam=4, max_len=40) GIT_LARGE batch32', model='GIT_LARGE', param=LARGE, batch=32, frames=0,
            search='beam', cpu_sample=1, enc=dict(g=16, p=14, d=1024, layers=24, L=257)),
    4: dict(metric='captions/sec (greedy, max_len=40) GIT_BASE_VATEX 6 frames batch16', model='GIT_BASE_VATEX',
            param={'num_image_with_embedding': 6}, batch=16, frames=6, search='greedy', cpu_sample=1,
            enc=dict(g=14, p=16, d=768, layers=12, L=197)),
    5: dict(metric='captions/sec (greedy, max_len=40) GIT_LARGE 8192-image shard, 1024 images per GPU', model='GIT_LARGE',
            param=LARGE, batch=64, shard=1024, frames=0, search='greedy', cpu_sample=2,
            enc=dict(g=16, p=14, d=1024, layers=24, L=257)),
}
# threads of the CPU arm: measured on the pool's host (128 hardware threads, profiles/cpu_threads_probe_r02.txt): 8 threads
# 0.79 s, 16 threads 0.53 s, 32 threads 1.11 s, 64 threads 2.41 s, 128 threads 112 s for the same B=2 / 9-step job --
# intra-op parallelism of these small fp32 ops stops scaling at 16 threads and collapses beyond
CPU_THREADS_CAP = 16


class Tok:
    cls_token_id, sep_token_id = 101, 102


def env_int(name, default):
    return int(os.environ.get(name, default))


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d['hbm_gbs'], bf16_tflops=d['bf16_tflops'], bf16_sustained=d.get('bf16_tflops_sustained'),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source='fallback (B200_PROFILING.md)')


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` captures
    (profiles/roofline_traffic.json names the .ncu-rep extract each figure comes from)."""
    p = os.path.join(ROOT, 'profiles', 'roofline_traffic.json')
    if os.path.exists(p):
        return json.load(open(p)).get(kernel, {}).get('dram_bytes_per_launch')
    return None


def algorithmic_work(cfg):
    """SURVEY.md section 8d formulas: (FLOP per caption, HBM bytes the decode steps stream per call)."""
    e = cfg['enc']
    g, p, d, layers, L = e['g'], e['p'], e['d'], e['layers'], e['L']
    D, F, V, nl = 768, 3072, 30522, 6
    frames = max(1, cfg['frames'])
    beam = 4 if cfg['search'] == 'beam' else 1
    B = cfg['batch']
    M = frames * L
    enc = frames * (g * g * 3 * p * p * d * 2 + layers * (2 * L * d * 3 * d + 4 * L * L * d + 2 * L * d * d + 16 * L * d * d))
    vproj = 2 * M * d * D
    prefill = nl * (6 * M * D * D + 4 * M * M * D + 2 * M * D * D + 4 * M * D * F)
    steps = MAX_STEPS - 1
    decode = sum(beam * (nl * (8 * D * D + 4 * (M + t + 1) * D + 4 * D * F) + 2 * D * V) for t in range(steps))
    wbytes = 2 * (nl * (4 * D * D + 2 * D * F) + V * D)
    dbytes = sum(wbytes + B * nl * 2 * M * D * 2 + B * beam * nl * 2 * t * D * 2 for t in range(steps))
    return dict(flop_per_caption=enc + vproj + prefill + decode, flop_tensor_part=enc + vproj + prefill, decode_bytes=dbytes)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line), streamed with
    `-lms` so that even a sub-second region gets several samples."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.proc = None
        self.stop_flag = False

    def run(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                          '--format=csv,noheader,nounits', '-lms', '20'], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                f = [x.strip() for x in line.strip().split(',')]
                if len(f) < 6:
                    continue
                try:
                    self.samples.append(float(f[0]))
                    self.max_mhz = float(f[1])
                except ValueError:
                    continue
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith('active'):
                        self.reasons.add(n)
                if self.stop_flag:
                    break
        except Exception:
            pass

    def stop(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self):
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2] if s else None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(s)}


def dump_outputs(dirname, predictions, logprobs):
    """--dump-outputs: the arrays one timed step returned, token ids as float64 (exact) and logprobs as float32."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, 'predictions.npy'), predictions.cpu().numpy().astype(np.float64))
    np.save(os.path.join(dirname, 'logprobs.npy'), logprobs.cpu().numpy().reshape(-1).astype(np.float32))


def cpu_reference_runs(cfg, sample, steps, warmup):
    """The reference's CPU path as shipped (full [image || text] recompute every step), fp32: `warmup` untimed then `steps`
    timed `model(batch)`-equivalents on `sample` images each.  Returns (captions/s, mean seconds per step, threads, the last
    step's outputs)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import git_oracle
    from generativeimage2text_b200.synthetic import synthetic_state_dict, synthetic_images
    threads = min(os.cpu_count(), CPU_THREADS_CAP)
    torch.set_num_threads(threads)
    sd = synthetic_state_dict(cfg['param'], 0, 'init')
    img = synthetic_images(sample, cfg['frames'], 1234)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = git_oracle.generate(sd, cfg['param'], {'image': img}, cfg['search'], MAX_STEPS, cached=False)
        dt = time.perf_counter() - t0
        assert out['predictions'].shape[0] == sample
        if i >= warmup:
            times.append(dt)
    mean = sum(times) / len(times)
    return sample / mean, mean, threads, out


def cpu_sample_text(cfg, sample, sec=None):
    return ('oracle/git_oracle.py as-shipped mode (no KV cache, fp32 torch CPU ops) on %d %s per step instead of %d '
            '(same per-caption work: CPU throughput is batch-insensitive here)%s' % (
                sample, 'videos' if cfg['frames'] else 'images', cfg['batch'], '' if sec is None else ', %.1f s per step' % sec))


def run_reference_arm(args, cfg, rank):
    if rank != 0:
        return
    sample = cfg['cpu_sample']
    value, sec, threads, out = cpu_reference_runs(cfg, sample, args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out['predictions'], out['logprobs'])
    line = {
        'impl': 'reference', 'metric': cfg['metric'], 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': '%s %s max_len=40, synthetic 224x224, random-init weights; CPU arm: %d captions per step '
                               '(bounded sample of the %d-caption call, throughput extrapolates linearly)' % (
                                   cfg['model'], cfg['search'], sample, cfg['batch']),
                   'global_batch': sample, 'bench_config': args.config},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': threads, 'kind': 'port',
                         'host_cpus': os.cpu_count(),
                         'threads_note': 'capped at %d: see profiles/cpu_threads_probe_r02.txt' % CPU_THREADS_CAP,
                         'sample': cpu_sample_text(cfg, sample, sec)},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


def main():
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get('GITB200_BENCH_WATCHDOG_S', '900')), exit=True)   # a hung run reports where
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='gitb200')
    ap.add_argument('--config', type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-micro', action='store_true')
    ap.add_argument('--no-serving', action='store_true')
    ap.add_argument('--pipeline', type=int, default=2, choices=[1, 2, 3, 4],
                    help='serving leg: engine launches in flight (the encoder of launch i+1 overlaps the decode loop of launch i)')
    ap.add_argument('--coalesce', type=int, default=4, choices=[1, 2, 3, 4],
                    help='serving leg: this many submitted batches share one engine launch (at most 256 decoder rows)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step as DIR/predictions.npy and DIR/logprobs.npy')
    ap.add_argument('--ncu-range', action='store_true',
                    help='bracket the timed region of `value` with cudaProfilerStart/Stop (use with ncu --profile-from-start off)')
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    if args.steps is None:
        args.steps = 4 if args.config == 5 else 16
    rank, world, local = env_int('RANK', 0), env_int('WORLD_SIZE', 1), env_int('LOCAL_RANK', 0)
    if args.impl == 'reference':
        run_reference_arm(args, cfg, rank)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import __graft_entry__
    __graft_entry__.build()
    from generativeimage2text_b200 import _lib
    from generativeimage2text_b200.model import get_git_model, AutoRegressiveBeamSearch, GeneratorWithBeamSearch
    from generativeimage2text_b200.sharding import gather_captions
    from generativeimage2text_b200.synthetic import synthetic_state_dict, synthetic_images

    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
    B = cfg['batch']
    beam = 4 if cfg['search'] == 'beam' else 1
    shard = cfg.get('shard', B)                 # captions per rank and step
    n_micro = shard // B
    os.environ.setdefault('GITB200_SLOTS', str(max(4, args.pipeline)))
    model = get_git_model(Tok(), cfg['param'])
    model.load_state_dict(synthetic_state_dict(cfg['param'], 0, 'init'), strict=True)
    model = model.to(dev).eval()
    if cfg['search'] == 'greedy':
        model.decoder = AutoRegressiveBeamSearch(102, max_steps=MAX_STEPS, beam_size=1, per_node_beam_size=1,
                                                 fix_missing_prefix=True)
    else:
        model.decoder = GeneratorWithBeamSearch(102, max_steps=MAX_STEPS, beam_size=4, length_penalty=0.6)

    def to_list(x):
        return x if isinstance(x, (list, tuple)) else [x]

    # this rank's pixels for one step: `n_micro` micro-batches (all configs but 5: one), host-pinned and device-resident
    host_batches, dev_batches = [], []
    for i in range(n_micro):
        im = synthetic_images(B, cfg['frames'], 1234 + 1000 * rank + i)
        hb = [t.contiguous().pin_memory() for t in to_list(im)]
        host_batches.append(hb if cfg['frames'] else hb[0])
        db = [t.to(dev) for t in hb]
        dev_batches.append(db if cfg['frames'] else db[0])
    h2d_bytes = sum(t.numel() * 4 for hb in host_batches for t in to_list(hb))
    stream = torch.cuda.Stream(device=dev)
    n_total = shard * world

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def one_step(batches, to_host, depth, coalesce):
        """All micro-batches of one step -> (tokens [shard, 40], logprobs [shard]) on the device."""
        toks, lps = [], []

        def keep(out):
            t, l = out['predictions'], out['logprobs'].reshape(-1)
            if to_host:                      # the caller reads the result: D2H inside the timed region
                t, l = t.cpu(), l.cpu()
                if world > 1:
                    t, l = t.to(dev), l.to(dev)
            if t.shape[1] < MAX_STEPS:       # (never with random weights: EOS does not fire)
                t = torch.nn.functional.pad(t, (0, MAX_STEPS - t.shape[1]), value=102)
            toks.append(t)
            lps.append(l)
        if depth == 1:
            for x in batches:
                keep(model({'image': x}))    # the reference call, one at a time, on the caller's stream
        else:
            pend = []
            for x in batches:
                pend.append(model.submit({'image': x}, depth=depth, coalesce=coalesce))
                if len(pend) >= depth * coalesce:
                    keep(pend.pop(0).result())
            while pend:
                keep(pend.pop(0).result())
        return toks, lps

    last_step = {}

    def run(k, to_host=False, depth=1, coalesce=1, steps_per_call=1):
        """k steps; returns the per-step host-side completion times are not needed: events bracket the whole region."""
        src = host_batches if to_host else dev_batches
        all_t, all_l = [], []
        if depth == 1:
            for _ in range(k):
                t, l = one_step(src, to_host, 1, 1)
                all_t += t
                all_l += l
            last_step['outputs'] = (t, l)    # the tensors the step's calls returned (fresh per call: no copy needed)
        else:
            # serving leg: the k steps' batches are submitted back to back so that launches stay in flight across steps
            t, l = one_step(src * k, to_host, depth, coalesce)
            all_t, all_l = t, l
        toks, lps = torch.cat(all_t, dim=0), torch.cat(all_l, dim=0)
        if world > 1:                        # ONE collective for everything this rank finished in the region
            toks, lps = gather_captions(toks.to(dev), lps.to(dev), toks.shape[0] * world)
        return toks

    def timed(k, **kw):
        barrier()
        launches0 = model.launch_count()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        evs[0].record(stream)
        toks = run(k, **kw)
        torch.cuda.current_stream().wait_stream(stream)
        for sl in model._slots:          # the pipelined engines run on their own streams: join them before the end event
            if sl['stream'] is not None:
                stream.wait_stream(sl['stream'])
        evs[1].record(stream)
        barrier()
        ms = evs[0].elapsed_time(evs[1])
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        assert toks.shape[0] == n_total * k and toks.shape[1] == MAX_STEPS, tuple(toks.shape)
        return t.item(), model.launch_count() - launches0

    sampler = ClockSampler(local)
    with torch.cuda.stream(stream):
        # ---------------- `value`: K model(batch) calls, pixels resident in HBM ----------------
        run(args.warmup)
        # per-call durations (median): one event pair per step, outside the max-over-ranks region
        per = []
        for _ in range(min(args.steps, 10)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            one_step(dev_batches, False, 1, 1)
            e1.record(stream)
            e1.synchronize()
            per.append(e0.elapsed_time(e1))
        per.sort()
        if rank == 0:
            sampler.start()
        if args.ncu_range:
            torch.cuda.profiler.start()
        ms, launches = timed(args.steps)
        if args.ncu_range:
            torch.cuda.profiler.stop()
        value_outputs = last_step['outputs']
        value = n_total * args.steps / (ms / 1e3)
        # ---------------- `e2e`: the same calls with HOST pixels in, tokens + logprobs back ----------------
        run(2, to_host=True)
        ms_e2e, _ = timed(args.steps, to_host=True)
        e2e_value = n_total * args.steps / (ms_e2e / 1e3)
        if rank == 0:
            sampler.stop()
            sampler.join(timeout=2)
        # ---------------- serving leg: dynamic batching + launches in flight ----------------
        serving = None
        if not args.no_serving and args.config != 5:
            co = max(1, min(args.coalesce, 256 // (B * beam)))
            depth = args.pipeline
            k_serv = args.steps
            run(2 * depth * co, depth=depth, coalesce=co)
            ms_s, _ = timed(k_serv, depth=depth, coalesce=co)
            run(2 * depth * co, to_host=True, depth=depth, coalesce=co)
            ms_se, _ = timed(k_serv, to_host=True, depth=depth, coalesce=co)
            serving = {'value': n_total * k_serv / (ms_s / 1e3), 'e2e_value': n_total * k_serv / (ms_se / 1e3), 'unit': UNIT,
                       'steps': k_serv, 'launches_in_flight': depth, 'batches_per_launch': co,
                       'api': 'model.submit(batch, depth=%d, coalesce=%d) -> handle.result(): %d submitted batches of %d share one '
                              'engine launch (one encoder pass, one decode chain over all their rows), %d launches in flight' % (
                                  depth, co, co, B, depth)}

    # ---------------- roofline of the dominant kernel, measured live ----------------
    peaks = measured_peaks()
    lib = _lib.load()
    roofline = None
    roofline_gemm = None
    work = algorithmic_work(cfg)
    if rank == 0 and cfg['search'] == 'greedy':
        # dominant kernel of a greedy call = decode_mega_kernel, one launch per decode step (profiles/launches_r02_*: ~2/3 of
        # a config-2 call).  HBM bound: algorithmic bytes per launch = the bf16 decoder weights + LM head, the image K/V of
        # every sequence and the text K/V so far (SURVEY.md 8d 'step bytes', averaged over the call's steps); duration =
        # CUDA events on the engine's stream around the call's decode loop / its step launches (gitb200_last_decode_ms).
        with torch.cuda.stream(stream):
            one_step(dev_batches, False, 1, 1)          # no collective here: this leg runs on rank 0 only
            ms_loop, n_launch, one_kernel = model.last_decode_timing()
        if one_kernel:
            bytes_per_launch = work['decode_bytes'] / (MAX_STEPS - 1)
            avg_ms = ms_loop / n_launch
            achieved = bytes_per_launch / (avg_ms / 1e3) / 1e9
            roofline = {'kernel': 'decode_mega_kernel (one persistent 148-CTA launch per decode step: 6 decoder layers + LM head + '
                                  'argmax / log-softmax + next embedding for %d sequences)' % B,
                        'bound': 'hbm', 'achieved': achieved, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                        'frac': achieved / peaks['hbm_gbs'], 'traffic': ncu_traffic('decode_mega_kernel') if args.config == 2 else None,
                        'avg_launch_ms': avg_ms, 'launches_timed': n_launch,
                        'algorithmic_bytes_per_launch': bytes_per_launch,
                        'peak_source': peaks['source'] + ', HBM copy bandwidth; the launches run back to back inside a call, '
                                       'so the figure includes the ~2 us between two graph launches'}
    if rank == 0 and not args.no_micro:
        # dominant kernel = the tcgen05 GEMM family (profiles/: > 1/2 of a call); its largest instance is the ViT MLP c_fc
        # GEMM [images * L, d] x [d, 4d] (+bias +QuickGELU, bf16 out): algorithmic FLOPs = 2*M*N*K.
        e = cfg['enc']
        M, N, K = B * max(1, cfg['frames']) * e['L'], 4 * e['d'], e['d']
        a = (torch.randn(M, K, device=dev) * 1.0).to(torch.bfloat16)
        w = (torch.randn(N, K, device=dev) * 0.03).to(torch.bfloat16)
        bias = torch.randn(N, device=dev)
        out = torch.empty(M, N, dtype=torch.bfloat16, device=dev)
        flush = torch.empty(160 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
        with torch.cuda.stream(stream):
            def gemm():
                rc = lib.gitb200_op_gemm(a.data_ptr(), w.data_ptr(), bias.data_ptr(), None, out.data_ptr(), M, N, K, 1, 1, 0, 1,
                                         0, stream.cuda_stream)
                assert rc == 0, _lib.last_error(None)
            for _ in range(3):
                gemm()
            durs = []
            for _ in range(10):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                gemm()
                e1.record(stream)
                e1.synchronize()
                durs.append(e0.elapsed_time(e1))
        avg_ms = sum(durs) / len(durs)
        flops = 2.0 * M * N * K
        achieved = flops / (avg_ms / 1e3) / 1e12
        roofline_gemm = {'kernel': 'gemm2_bf16_tcgen05<256> (ViT mlp.c_fc shape %dx%dx%d, bias+QuickGELU epilogue)' % (M, N, K),
                    'bound': 'tensor', 'achieved': achieved, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s',
                    'frac': achieved / peaks['bf16_tflops'], 'traffic': ncu_traffic('gemm2_bf16_tcgen05') if args.config == 2 else None,
                    'avg_launch_ms': avg_ms,
                    'peak_source': peaks['source'] + ', burst bf16 figure (kernel timed alone, L2 flushed between launches)'}
    # whole-call roofline (SURVEY.md section 8d): tensor part at the sustained GEMM peak + decode bytes at the HBM peak
    t_floor = work['flop_tensor_part'] * B / (peaks['bf16_sustained'] * 1e12) + work['decode_bytes'] / (peaks['hbm_gbs'] * 1e9)
    whole = {'algorithmic_gflop_per_caption': work['flop_per_caption'] / 1e9,
             'decode_bytes_per_call_gb': work['decode_bytes'] / 1e9,
             'roofline_ms_per_call': t_floor * 1e3,
             'roofline_captions_per_s_per_gpu': B / t_floor,
             'frac_of_roofline': (value / world) / (B / t_floor),
             'achieved_tflops': work['flop_per_caption'] * (value / world) / 1e12}

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        sample = {2: 12, 3: 3, 4: 2, 5: 6}[args.config]
        v, sec, threads, _ = cpu_reference_runs(cfg, sample, 1, 0)
        cpu = {'value': v, 'unit': UNIT, 'cores': threads, 'host_cpus': os.cpu_count(), 'kind': 'port',
               'sample': 'one call, ' + cpu_sample_text(cfg, sample, sec)}

    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, *(torch.cat(x, dim=0) for x in value_outputs))

    if rank == 0:
        steps_desc = ('one pass over the rank\'s %d-image shard in %d micro-batches of %d' % (shard, n_micro, B)) if n_micro > 1 \
            else 'one model(batch) call of %d %s' % (B, 'videos x %d frames' % cfg['frames'] if cfg['frames'] else 'images')
        line = {
            'metric': cfg['metric'], 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms / args.steps, 'median_ms_per_step': per[len(per) // 2], 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
            'config': {'workload': '%s %s max_len=40, synthetic 224x224 pixels, random-init weights; step = %s' % (
                           cfg['model'], 'beam 4 (length_penalty 0.6)' if beam > 1 else 'greedy', steps_desc),
                       'bench_config': args.config, 'global_batch': n_total, 'per_gpu_batch': shard,
                       'parallelism': 'image-parallel x%d, ONE fused all_gather of the finished captions per timed region' % world,
                       'l2': 'inputs larger than L2: every call streams the bf16 weights (%.2f GB) + the image K/V cache per step '
                             '(>> 126 MB); no flush needed between steps' % (0.31 if cfg['model'] != 'GIT_LARGE' else 0.74),
                       'compute': 'bf16 operands, fp32 accumulate, fp32 residual stream',
                       'calls': 'one model(batch) at a time (SURVEY.md 8d); the dynamic-batching form is under "serving"'},
            'e2e': {'value': e2e_value, 'unit': UNIT, 'ms_per_step': ms_e2e / args.steps, 'h2d_bytes_per_step': h2d_bytes,
                    'd2h_bytes_per_step': shard * MAX_STEPS * 8 + shard * 4,
                    'api': "model({'image': pinned host tensor(s)}) -> predictions.cpu(), logprobs.cpu()"},
            'gpu_launches': int(launches),
            'clocks': sampler.summary(),
            'roofline': roofline if roofline is not None else roofline_gemm,
            'roofline_encoder_gemm': roofline_gemm if roofline is not None else None,
            'whole_call': whole,
            'serving': serving,
            'cpu_baseline': cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
