"""bench.py — tokens/sec of one ProGen training step (BASELINE.json configs[1]) on N B200s of one node.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...      # the CPU arm: the oracle port timed on the host cores
    python bench.py ... --dump-outputs DIR    # also write what the last timed step computed, as DIR/<name>.npy

A "step" is one pass of the hot path over one synthetic batch: forward + loss + backward + (DDP gradient all-reduce) +
clip/AdamW/apply_every, i.e. one iteration of the reference's inner loop (train.py:186-190).  Prints ONE JSON line.
Inputs and parameters are seeded, so two builds run with the same arguments can be compared dump for dump.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (no __pycache__ for the project's modules)

CONFIGS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on
    'cfg2': dict(kwargs=dict(num_tokens=256, dim=512, seq_len=1024, depth=12, heads=8, dim_head=64, window_size=256,
                             global_mlp_depth=2, ff_glu=True), batch=64,
                 name='ProGen dim=512 depth=12 heads=8 seq_len=1024 window=256 gmlp=2 bf16 - training step, synthetic batch=64/GPU (BASELINE configs[1])'),
    'cfg3': dict(kwargs=dict(num_tokens=256, dim=1024, seq_len=2048, depth=24, heads=16, dim_head=64, window_size=512,
                             global_mlp_depth=2, ff_glu=True), batch=8,
                 name='ProGen dim=1024 depth=24 heads=16 seq_len=2048 window=512 gmlp=2 bf16 - training step (BASELINE configs[2])'),
    # BASELINE.json configs[3]: HBM-bandwidth stress (heads unspecified => constructor default 8 x 64, so inner 512 != dim)
    'cfg4': dict(kwargs=dict(num_tokens=256, dim=1536, seq_len=4096, depth=36, heads=8, dim_head=64, window_size=256,
                             global_mlp_depth=2, ff_glu=True), batch=4,
                 name='ProGen dim=1536 depth=36 seq_len=4096 window=256 ff_glu bf16 - training step (BASELINE configs[3])'),
    # BASELINE.json configs[4]: sample.py decode, seq_len 1024, prime '[Tax=Mammalia] #', on the configs[1] model
    'cfg5': dict(kwargs=dict(num_tokens=256, dim=512, seq_len=1024, depth=12, heads=8, dim_head=64, window_size=256,
                             global_mlp_depth=2, ff_glu=True), batch=1, decode=True,
                 name="sample.py autoregressive decode seq_len=1024, prime='[Tax=Mammalia] #', top_k=25, add_bos - ProGen dim=512 "
                      "depth=12 heads=8 window=256 gmlp=2, bf16 weights, KV-cached persistent kernel (BASELINE configs[4])"),
    'tiny': dict(kwargs=dict(num_tokens=256, dim=128, seq_len=128, depth=2, heads=2, dim_head=64, window_size=64,
                             global_mlp_depth=1, ff_glu=True), batch=4, name='tiny smoke configuration (not a bench line)'),
}


def fwd_flops_per_token(kw):
    """SURVEY.md §8(d): causal-algorithmic forward FLOPs per token (LN / softmax / GELU / rotary excluded)."""
    d, n, w = kw['dim'], kw['seq_len'], kw['window_size']
    I = kw['heads'] * kw['dim_head']
    V = kw['num_tokens']
    total = 2 * d * V
    for i in range(kw['depth']):
        attn = 6 * d * I + 2 * I * d + 4 * I * (w + (w + 1) / 2)
        gmlp = (kw['depth'] - i) <= kw['global_mlp_depth']
        ff = (20 * d * d + 2 * (n + 1) * d) if gmlp else (24 * d * d if kw['ff_glu'] else 16 * d * d)
        total += attn + ff
    return total


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(burst=j['bf16_tflops'], sustained=j.get('bf16_tflops_sustained', j['bf16_tflops']), hbm=j['hbm_gbs'],
                    source='measured (MEASURED_PEAKS.json)')
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            f = [x.strip() for x in r.split(',')]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except Exception:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def synthetic_batches(count, B, n, seed):
    """uniform-random [0,256) rows of n+1 tokens (BASELINE north_star), int32, pinned when a GPU is present"""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        t = torch.from_numpy(rng.integers(0, 256, (B, n + 1)).astype(np.int32))
        out.append(t.pin_memory() if torch.cuda.is_available() else t)
    return out


DUMP_SAMPLE = 1 << 21    # elements kept of a larger output: three 8 MB float32 samples stay well inside 64 MB per dump


def dump_sample(x, seed):
    """x flattened to float32; above DUMP_SAMPLE elements, a fixed subset whose indices depend only on `seed` and x.size"""
    x = np.asarray(x, np.float32).ravel()
    if x.size <= DUMP_SAMPLE:
        return x
    return x[np.sort(np.random.default_rng(seed).integers(0, x.size, DUMP_SAMPLE))]


def dump_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), a)


def train_step_outputs(eng, loss):
    """What the last timed training step computed: its loss, its logits, the parameter gradient and the parameters after
    the optimizer update.  Trees are flattened in sorted (module, name) order, so the sample does not depend on the
    engine's internal buffer layout."""
    flat = lambda tree: np.concatenate([tree[m][k].ravel() for m in sorted(tree) for k in sorted(tree[m])])
    return dict(loss=np.array([loss], np.float32), logits=dump_sample(eng.logits.cpu().numpy(), 1),
                grads=dump_sample(flat(eng.export_grads()), 2), params=dump_sample(flat(eng.export_params()), 3))


CPU_THREAD_CAP = 32      # the box reports 128 logical CPUs shared with other tenants; 128 torch threads thrash (6-52 tok/s)


def cpu_threads():
    return max(1, min(len(os.sched_getaffinity(0)), CPU_THREAD_CAP))


def cpu_port_tokens_per_sec(kw, steps, warmup, rows=1, seed=123, budget_s=60.0):
    """The reference's Jax path is not installable (no jax wheels, no network), so the timed CPU implementation is the
    oracle's torch port of the same algorithm: fp32, host cores through torch intra-op threads, fwd + bwd.
    Bounded: stops as soon as `budget_s` of timed work has accumulated (a slow warm-up step counts as the sample)."""
    from oracle import progen_ref as O
    from oracle import progen_torch as T
    torch.set_num_threads(cpu_threads())
    cfg = O.make_config(**kw)
    params = O.init_params(cfg, 0)
    prm = T.to_torch(params, torch.float32, requires_grad=True)
    rng = np.random.default_rng(seed)
    n = cfg['seq_len']
    times, first = [], None
    for i in range(warmup + steps):
        data = torch.as_tensor(rng.integers(0, 256, (rows, n + 1)).astype(np.int64))
        t0 = time.perf_counter()
        loss = T.batch_loss(prm, data, cfg)
        loss.backward()
        for d in prm.values():
            for v in d.values():
                v.grad = None
        dt = time.perf_counter() - t0
        first = dt if first is None else first
        if i >= warmup:
            times.append(dt)
        if sum(times) + (first if not times else 0.0) > budget_s:
            break
    if not times:
        times = [first]
    sec = sum(times) / len(times)
    return rows * n / sec, sec, rows, len(times)


def decode_bytes_per_token(kw, wbytes):
    """algorithmic HBM bytes one decoded position must move: every weight once (`wbytes` per element; the embedding row and
    the SGU spatial row are negligible), the visible K / V rows of every layer (fp32 cache, on average w + w/2 keys), the
    gate history of the gMLP layers (on average n/2 rows)"""
    d, n, w, L = kw['dim'], kw['seq_len'], kw['window_size'], kw['depth']
    I = kw['heads'] * kw['dim_head']
    hid = 4 * d
    nsgu = min(L, kw['global_mlp_depth'])
    per_glu = d * 3 * I + I * d + d * 2 * hid + hid * d
    per_sgu = d * 3 * I + I * d + d * hid + (hid // 2) ** 2 + (hid // 2) * d
    weights = ((L - nsgu) * per_glu + nsgu * per_sgu + d * kw['num_tokens']) * wbytes
    kv = L * 2 * (w + w / 2) * I * 4
    hist = nsgu * (n / 2) * (hid // 2) * 4
    return weights, kv + hist


def cpu_decode_tokens_per_sec(kw, prime, tokens=4):
    """the reference's sampler on the host: one FULL forward of the padded sequence per generated token (utils.py:115-117),
    oracle NumPy/torch port, fp32, bounded to a few tokens"""
    from oracle import progen_ref as O
    from oracle import progen_torch as T
    torch.set_num_threads(cpu_threads())
    cfg = O.make_config(**kw)
    prm = T.to_torch(O.init_params(cfg, 0), torch.float32)
    n = cfg['seq_len']
    seq = torch.zeros(1, n, dtype=torch.int64)
    seq[0, 1:1 + len(prime)] = torch.as_tensor(np.asarray(prime).astype(np.int64))
    times = []
    with torch.no_grad():
        for i in range(tokens + 1):
            t0 = time.perf_counter()
            logits = T.forward(prm, seq, cfg)[0, len(prime) + i]
            seq[0, len(prime) + 1 + i] = int(torch.argmax(logits))
            if i > 0:
                times.append(time.perf_counter() - t0)
    return 1.0 / (sum(times) / len(times)), len(times)


def run_decode_bench(args, cfgd):
    """BASELINE configs[4]: tokens/s of the KV-cached sampler.  A "step" = one whole generation (seq_len - prime tokens) of
    one sequence per GPU; `value` = generated tokens / device time with the prime already on the device; `e2e` = the
    public call with the prime on the host and the ids read back.  Beside it: B = 64 primes decoded in lock step."""
    import torch.distributed as dist
    from progen_b200 import ProGen, lib as L
    from progen_b200.decode import BatchDecoder
    from progen_b200.data import encode_tokens
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get('NCCL_DEBUG', '').upper() in ('', 'VERSION'):
            os.environ['NCCL_DEBUG'] = 'WARN'
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    L.require_device()
    kw = cfgd['kwargs']
    n = kw['seq_len']
    model = ProGen(**kw)
    params = model.init(1234)
    prime = np.array(encode_tokens('[Tax=Mammalia] #'), dtype=np.int64)
    wdt = torch.float32 if args.fp32 else torch.bfloat16
    dec = BatchDecoder(model.config, params, batch=1, weights_dtype=wdt)
    c0 = L.load().progen_launch_count()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        dec.sample(prime, top_k=25, add_bos=True, greedy=False, seed=rank)
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    dev_s, gen_tokens = 0.0, 0
    t0 = time.perf_counter()
    for i in range(args.steps):
        ids, gen, secs = dec.sample(prime, top_k=25, add_bos=True, greedy=False, seed=100 + i)
        dev_s += secs
        gen_tokens += gen
    barrier()
    wall_s = time.perf_counter() - t0
    clocks = sampler.stop() if sampler else None
    launches = L.load().progen_launch_count() - c0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(ids=np.asarray(ids, np.float64)))     # the last generation's token ids
    t = torch.tensor([dev_s, wall_s], device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_s, wall_s = float(t[0]), float(t[1])
    tps = gen_tokens * world / dev_s
    tps_e2e = gen_tokens * world / wall_s
    # batched: 64 primes in lock step
    Bb = 64
    decb = BatchDecoder(model.config, params, batch=Bb, weights_dtype=wdt)
    decb.sample([prime] * Bb, top_k=25, add_bos=True, greedy=False, seed=7)
    _, genb, secb = decb.sample([prime] * Bb, top_k=25, add_bos=True, greedy=False, seed=8)
    if rank == 0:
        peaks = measured_peaks()
        wb, rest = decode_bytes_per_token(kw, 4 if args.fp32 else 2)
        per_tok_s = dev_s / gen_tokens
        achieved = (wb + rest) / per_tok_s / 1e9
        per_step_b = secb / (genb / Bb)
        achieved_b = (wb + Bb * rest) / per_step_b / 1e9
        try:
            dk = json.load(open(os.path.join(ROOT, 'profiles', 'r02_decode_kernel.json')))
            traffic, traffic_b = dk['single']['dram_bytes_per_token'], dk['batched']['dram_bytes_per_step']
        except Exception:
            traffic = traffic_b = None
        roofline = dict(bound='hbm', achieved=achieved, peak=peaks['hbm'], unit='GB/s', frac=achieved / peaks['hbm'], traffic=traffic,
                        traffic_unit='DRAM bytes per token (ncu --set full of one 8-position launch, profiles/r02_ncu_decode_persistent.txt)',
                        kernel='decode_persistent_kernel<1, bf16> (one cooperative kernel for the whole generation)',
                        algorithmic_bytes_per_token=wb + rest, us_per_token=per_tok_s * 1e6, peak_source=peaks['source'],
                        batched=dict(batch=Bb, tokens_per_sec=genb / secb, us_per_step=per_step_b * 1e6, achieved=achieved_b, traffic=traffic_b,
                                     frac=achieved_b / peaks['hbm'], algorithmic_bytes_per_step=wb + Bb * rest))
        line = dict(metric='decode_tokens_per_sec', value=tps, unit='tokens/s', n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=dev_s / args.steps * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None,
                    dtype='f32' if args.fp32 else 'bf16', data='synthetic',
                    config=dict(workload=cfgd['name'], global_batch=world, seq_len=n, parallelism=f'replicas x{world}',
                                l2='103 MB of bf16 weights + K/V do not stay in the 126 MB L2 between positions: ncu measures 125 MB of DRAM reads per token, the algorithmic 122 MB',
                                step='one generation of %d tokens' % (gen_tokens // args.steps)),
                    e2e=dict(value=tps_e2e, unit='tokens/s', h2d_bytes_per_step=int(n * 4 + 4), d2h_bytes_per_step=int(n * 4),
                             ms_per_step=wall_s / args.steps * 1e3),
                    gpu_launches=int(launches), clocks=clocks, roofline=roofline)
        if not args.no_cpu_baseline and world == 1:
            v, timed = cpu_decode_tokens_per_sec(kw, prime)
            line['cpu_baseline'] = dict(value=v, unit='tokens/s', cores=cpu_threads(), kind='port',
                                        sample=f'{timed} generated tokens, one full {n}-token forward each (reference sampler), fp32')
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_reference_arm(args, cfgd):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    kw = cfgd['kwargs']
    if cfgd.get('decode'):
        from progen_b200.data import encode_tokens
        prime = np.array(encode_tokens('[Tax=Mammalia] #'), dtype=np.int64)
        v, timed = cpu_decode_tokens_per_sec(kw, prime, tokens=max(2, min(args.steps, 8)))
        line = dict(impl='reference', metric='decode_tokens_per_sec', value=v, unit='tokens/s', n_gpus=args.gpus, steps=args.steps,
                    warmup=args.warmup, ms_per_step=1e3 / v, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32',
                    data='synthetic', config=dict(workload=cfgd['name']),
                    cpu_baseline=dict(value=v, unit='tokens/s', cores=cpu_threads(), kind='port',
                                      sample=f'{timed} generated tokens, one full forward each'),
                    e2e=dict(value=v, unit='tokens/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                    note='oracle torch port of the reference sampler (full re-forward per token) on the host cores')
        print(json.dumps(line), flush=True)
        return
    cores = cpu_threads()
    # bounded sample: one sequence per step; the loop stops once ~60 s of timed work has accumulated (a step takes
    # 0.6 s on an idle box and up to 40 s on a loaded one), so the whole arm ends within a few minutes either way
    steps, warmup = max(1, min(args.steps, 50)), max(1, min(args.warmup, 2))
    tps, sec, rows, timed = cpu_port_tokens_per_sec(kw, steps, warmup, rows=1)
    sample = f"{rows} sequence x {kw['seq_len']} tokens per step (fwd+bwd, fp32), {timed} timed steps (of --steps {args.steps})"
    line = dict(impl='reference', metric='tokens_per_sec', value=tps, unit='tokens/s', n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=sec * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None,
                dtype='f32', data='synthetic', config=dict(workload=cfgd['name']),
                cpu_baseline=dict(value=tps, unit='tokens/s', cores=cores, kind='port', sample=sample),
                e2e=dict(value=tps, unit='tokens/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                note='reference Jax/Haiku is not installable here (no jax/jaxlib/haiku wheels, no network); this is the '
                     'oracle torch port of the same algorithm on the host cores')
    print(json.dumps(line), flush=True)


def _time_launch(launch, iters):
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        launch()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def attn_fwd_flops_per_token(kw):
    """SURVEY 8(d): 4 I (w + (w + 1) / 2) per token per layer — the causal keys actually visible, two contractions"""
    return 4.0 * kw['heads'] * kw['dim_head'] * (kw['window_size'] + (kw['window_size'] + 1) / 2)


def time_step_kernels(eng, kw, iters=20):
    """The kernels that carry the step, each timed ALONE with CUDA events on the launching stream (same buffers and shapes
    as inside the step), with the number of launches of that shape per step and its algorithmic FLOPs (SURVEY 8(d): no
    recompute credit — the attention backward is charged 2x the forward's FLOPs although its two kernels execute 3.5x).
    The caller picks the largest share of the step as the `roofline` kernel and lists the rest beside it."""
    from progen_b200 import lib as L
    from progen_b200.engine import P
    out = []
    T, d, I, hid = eng.T, eng.d, eng.I, eng.hid
    nl = len(eng.kinds)
    s0 = eng.lay[0]
    if eng.attn_tc:
        fa = attn_fwd_flops_per_token(kw) * T
        ms = _time_launch(lambda: eng.attn_fwd(s0['qkv'], s0['att'], s0['lse']), iters)
        out.append(dict(key='attn_fwd', kernel='sliding-window attention forward (tcgen05, P and O in TMEM)', per_step=nl, ms=ms,
                        flops=fa, shape=[eng.B, eng.h, eng.n, eng.w]))
        ms = _time_launch(lambda: eng.attn_bwd(s0['qkv'], s0['att'], eng.datt, s0['lse'], eng.dqkv), iters)
        out.append(dict(key='attn_bwd', kernel='sliding-window attention backward (dQ kernel + dK/dV kernel, tcgen05)', per_step=nl,
                        ms=ms, flops=2.0 * fa, shape=[eng.B, eng.h, eng.n, eng.w]))
    i = next((j for j, k in enumerate(eng.kinds) if k == 'glu'), None)
    if i is not None:
        s = eng.lay[i]
        f = P + f'ff{i}/~/'
        n_glu = sum(1 for k in eng.kinds if k == 'glu')
        ms = _time_launch(lambda: eng.wgrad_gemm(s['y2'], d, eng.du, 2 * hid, eng.G(f + 'linear', 'w')), iters)
        out.append(dict(key='wgrad_ffin', kernel='gemm_tc2_kernel<MN-major A, MN-major B, EPI_ACCUM, fp32> (CTA-pair tcgen05, FF proj_in '
                                                 'weight gradient, split-K + TMA reduce-add)', per_step=n_glu, ms=ms,
                        flops=2.0 * T * d * 2 * hid, shape=[d, 2 * hid, T]))
        ms = _time_launch(lambda: eng.fwd_gemm(s['y2'], d, eng.W(f + 'linear', 'w'), 2 * hid, s['hact'], epi=L.EPI_GLU, ldo=hid,
                                               out2=s['u'], ldo2=2 * hid, bias=eng.Pf(f + 'linear', 'b')), iters)
        out.append(dict(key='ffin_glu', kernel='gemm_tc2_kernel<K-major A, MN-major B, EPI_GLU, bf16> (CTA-pair tcgen05, FF proj_in fwd)',
                        per_step=n_glu, ms=ms, flops=2.0 * T * d * 2 * hid, shape=[T, 2 * hid, d]))
        ms = _time_launch(lambda: eng.dgrad_gemm(eng.dres_lp, d, eng.W(f + 'linear_1', 'w'), hid, eng.du, epi=L.EPI_GLU_BWD,
                                                 ldo=2 * hid, aux=s['u'], ldaux=2 * hid), iters)
        out.append(dict(key='ffout_dgrad_glu_bwd', kernel='gemm_tc2_kernel<K-major, K-major, EPI_GLU_BWD, bf16> (FF proj_out dgrad + GLU backward)',
                        per_step=n_glu, ms=ms, flops=2.0 * T * d * hid, shape=[T, hid, d]))
    for o in out:
        o['tflops'] = o['flops'] / o['ms'] / 1e9
        o['step_ms'] = o['ms'] * o['per_step']
    return out


def dominant_kernel_traffic(config, batch, key):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of kernel `key`, from the committed `ncu --set full`
    captures (profiles/r02_dominant_kernel.json, else round 1's file); null for any other shape."""
    for name in ('r02_dominant_kernel.json', 'r01_dominant_kernel.json'):
        try:
            j = json.load(open(os.path.join(ROOT, 'profiles', name)))
            if j.get('config') == config and j.get('batch') == batch and key in j['kernels']:
                return j['kernels'][key]['dram_bytes_per_launch']
        except Exception:
            pass
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='cfg2', choices=sorted(CONFIGS))
    ap.add_argument('--batch', type=int, default=None, help='per-GPU batch override')
    ap.add_argument('--fp32', action='store_true', help='fp32 engine (parity path) instead of bf16')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed to DIR/<name>.npy (float32 / float64, seeded samples of large arrays)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of the b200 implementation')
    args.warmup = max(3, args.warmup) if args.impl == 'b200' else args.warmup
    cfgd = CONFIGS[args.config]
    kw = cfgd['kwargs']
    if args.impl == 'reference':
        run_reference_arm(args, cfgd)
        return
    if cfgd.get('decode'):
        run_decode_bench(args, cfgd)
        return

    import torch.distributed as dist
    from progen_b200 import ProGen, lib as L
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get('NCCL_DEBUG', '').upper() in ('', 'VERSION'):
            os.environ['NCCL_DEBUG'] = 'WARN'             # the version banner goes to stdout; keep it to the single JSON line
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    assert world == args.gpus, f'--gpus {args.gpus} but WORLD_SIZE={world}'
    L.require_device()
    B = args.batch or cfgd['batch']
    n = kw['seq_len']
    model = ProGen(**kw, mixed_precision=not args.fp32)
    params = model.init(1234)                      # same seed on every rank: identical replicas
    tr = model.trainer(params)                     # reference optimizer chain, grad_accum_every=4
    eng = model.engine
    total = args.warmup + args.steps
    batches = synthetic_batches(total, B, n, 42 + rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident leg: inputs already in HBM when the timed region starts
    dev_batches = [b.cuda() for b in batches]
    for i in range(args.warmup):
        eng.ensure_batch(B)
        eng.tok.copy_(dev_batches[i][:, :-1].reshape(-1)); eng.labels.copy_(dev_batches[i][:, 1:].reshape(-1))
        tr.step_resident(global_batch=B * world)
    # single GPU: the whole step (forward, loss, backward, norm, AdamW) is captured ONCE into a CUDA graph after the eager
    # warm-up and replayed by the same Trainer.step / step_resident calls (PROGEN_BENCH_GRAPH=0 keeps eager launches)
    # The whole step (forward, loss, backward, gradient all-reduce, norm, AdamW) is captured ONCE into a CUDA graph after the
    # eager warm-up and replayed by the same Trainer.step / step_resident calls — at N > 1 the NCCL all-reduce is part of the
    # graph (PROGEN_BENCH_GRAPH=0 keeps eager launches; PROGEN_DDP_OVERLAP=1 is the round-1 bucketed overlap, eager only)
    graph_nodes = 0
    graph_ok = torch.ones(1, device='cuda')
    if os.environ.get('PROGEN_BENCH_GRAPH', '1') != '0' and not tr.overlap:
        c0 = L.load().progen_launch_count()
        try:
            tr.capture_graph(B, B * world)
            graph_nodes = int(L.load().progen_launch_count() - c0)     # kernels of ours recorded per step
        except Exception as e:                                          # same kernels, launched eagerly instead
            print(f'[bench] rank {rank}: CUDA-graph capture failed ({type(e).__name__}: {e}); continuing with eager launches', file=sys.stderr)
            tr._graph = None
            graph_ok.zero_()
            torch.cuda.synchronize()
        if world > 1:
            dist.all_reduce(graph_ok, op=dist.ReduceOp.MIN)             # all ranks replay, or none does (the collectives must pair up)
            if graph_ok.item() == 0:
                tr._graph, graph_nodes = None, 0
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    launches0 = L.load().progen_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    prof_range = os.environ.get('PROGEN_PROFILE_RANGE') == '1'    # ncu --profile-from-start off: only the timed steps
    if prof_range:
        torch.cuda.profiler.start()
    e0.record()
    for i in range(args.warmup, total):
        eng.tok.copy_(dev_batches[i][:, :-1].reshape(-1)); eng.labels.copy_(dev_batches[i][:, 1:].reshape(-1))
        tr.step_resident(global_batch=B * world)
    e1.record()
    barrier()
    if prof_range:
        torch.cuda.profiler.stop()
    launches = L.load().progen_launch_count() - launches0
    if graph_nodes:
        launches = graph_nodes * args.steps            # replayed graph: the host-side counter only sees the capture
    ms = torch.tensor([e0.elapsed_time(e1)], device='cuda')
    per_rank_ms = [float(ms.item()) / args.steps]
    if world > 1:
        gathered = [torch.zeros_like(ms) for _ in range(world)]
        dist.all_gather(gathered, ms)
        per_rank_ms = [float(g.item()) / args.steps for g in gathered]
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    clocks = sampler.stop() if sampler else None
    loss_t = eng.loss.clone()
    if world > 1:
        dist.all_reduce(loss_t)                        # per-rank losses are pre-scaled by 1/global_batch: the sum is the mean
    final_loss = float(loss_t.item())
    if args.dump_outputs and rank == 0:                # before the legs below train further
        dump_outputs(args.dump_outputs, train_step_outputs(eng, final_loss))

    # ---------------- end-to-end leg: public API with HOST (pinned) buffers, H2D + loss D2H inside the timed region.
    # Two readers of the per-step loss: (a) a training loop that keeps the GPU fed — `Trainer.step(host_batch)` returns the
    # device scalar and the loop copies it to pinned host memory with a non-blocking copy (every step's loss IS read back
    # inside the timed region; the host only waits at the end); (b) the reference's `print(loss)` style, `.item()` after
    # every step, which leaves the GPU idle while the host launches the next step's graph.  (a) is `e2e.value`.
    for i in range(min(2, args.warmup)):
        float(tr.step(batches[i]).item())
    host_losses = torch.empty(args.steps, dtype=torch.float32).pin_memory()
    barrier()
    e0.record()
    for j, i in enumerate(range(args.warmup, total)):
        loss = tr.step(batches[i])
        host_losses[j:j + 1].copy_(loss.reshape(1), non_blocking=True)
    e1.record()
    barrier()
    assert bool(torch.isfinite(host_losses).all()) and float(host_losses.abs().min()) > 0.0, host_losses
    ms2 = torch.tensor([e0.elapsed_time(e1)], device='cuda')
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    ms_e2e = float(ms2.item())
    barrier()
    e0.record()
    for i in range(args.warmup, total):
        float(tr.step(batches[i]).item())
    e1.record()
    barrier()
    ms3 = torch.tensor([e0.elapsed_time(e1)], device='cuda')
    if world > 1:
        dist.all_reduce(ms3, op=dist.ReduceOp.MAX)
    ms_e2e_blocking = float(ms3.item())

    # ---------------- exposed communication: the same K steps with the gradient exchange removed (same launch mode, same box);
    # the ranks no longer agree afterwards, so this runs last and nothing is reported from its state
    comm = None
    if world > 1:
        tr.skip_allreduce = True
        try:
            if tr._graph is not None:
                tr._graph = None
                tr.capture_graph(B, B * world)
            for i in range(2):
                tr.step_resident(global_batch=B * world)
            barrier()
            e0.record()
            for i in range(args.warmup, total):
                eng.tok.copy_(dev_batches[i][:, :-1].reshape(-1)); eng.labels.copy_(dev_batches[i][:, 1:].reshape(-1))
                tr.step_resident(global_batch=B * world)
            e1.record()
            barrier()
            ms3 = torch.tensor([e0.elapsed_time(e1)], device='cuda')
            dist.all_reduce(ms3, op=dist.ReduceOp.MAX)
            comm = dict(step_ms_without_exchange=float(ms3.item()) / args.steps,
                        comm_exposed_ms=ms_total / args.steps - float(ms3.item()) / args.steps,
                        grad_bytes=int(eng.n_params_padded) * 4, mode='bucketed overlap (eager)' if tr.overlap else
                        'one fp32 SUM all-reduce after backward, inside the step graph' if graph_nodes else 'one fp32 SUM all-reduce after backward (eager)')
        except Exception as e:
            print(f'[bench] rank {rank}: comm_exposed measurement failed ({type(e).__name__}: {e})', file=sys.stderr)
        tr.skip_allreduce = False

    tokens_per_step = B * n * world
    tps = tokens_per_step * args.steps / (ms_total / 1e3)
    tps_e2e = tokens_per_step * args.steps / (ms_e2e / 1e3)
    if rank == 0:
        peaks = measured_peaks()
        train_flops = 3.0 * fwd_flops_per_token(kw)
        achieved = tps * train_flops / 1e12 / world
        kernels = time_step_kernels(eng, kw) if not args.fp32 else []
        whole_step = dict(achieved=achieved, peak=peaks['sustained'], unit='TFLOP/s', frac=achieved / peaks['sustained'],
                          peak_source=peaks['source'] + ', sustained figure (kernels timed inside a long step)',
                          definition='whole step: tokens/s x 3 x F_fwd (SURVEY 8d, %.2f MFLOP/token train) per GPU' % (train_flops / 1e6))
        if kernels:
            # the dominant kernel = the (symbol, shape) with the largest share of the step; timed alone with CUDA events just
            # above: algorithmic FLOPs of one launch / its duration, against the burst peak
            step_ms = ms_total / args.steps
            dom = max(kernels, key=lambda k: k['step_ms'])
            roofline = dict(bound='tensor', achieved=dom['tflops'], peak=peaks['burst'], unit='TFLOP/s',
                            frac=dom['tflops'] / peaks['burst'], traffic=dominant_kernel_traffic(args.config, B, dom['key']),
                            kernel=dom['kernel'], shape=dom['shape'], ms=dom['ms'], launches_per_step=dom['per_step'],
                            share_of_step=dom['step_ms'] / step_ms,
                            peak_source=peaks['source'] + ', burst figure (kernel timed alone)', whole_step=whole_step,
                            others=[dict(key=k['key'], kernel=k['kernel'], shape=k['shape'], ms=k['ms'], launches_per_step=k['per_step'],
                                         share_of_step=k['step_ms'] / step_ms, achieved=k['tflops'], frac=k['tflops'] / peaks['burst'],
                                         traffic=dominant_kernel_traffic(args.config, B, k['key']))
                                    for k in kernels if k is not dom])
        else:
            roofline = dict(bound='tensor', traffic=None, **whole_step)
        line = dict(metric='tokens_per_sec', value=tps, unit='tokens/s', n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms_total / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None,
                    dtype='f32' if args.fp32 else 'bf16', data='synthetic',
                    config=dict(workload=cfgd['name'], global_batch=B * world, seq_len=n, parallelism=f'dp{world}',
                                l2='activations (~%.1f GB/step) far exceed the 126 MB L2; no explicit flush' % (eng_bytes(eng) / 1e9),
                                optimizer='clip_by_global_norm(0.5)+adamw(2e-4,wd=1e-3,mask)+apply_every(4), every step',
                                launch='CUDA graph of the whole step (%d kernels%s), replayed' % (graph_nodes, ' + the NCCL all-reduce' if world > 1 else '') if graph_nodes
                                       else 'eager launches'),
                    e2e=dict(value=tps_e2e, unit='tokens/s', h2d_bytes_per_step=B * (n + 1) * 4, d2h_bytes_per_step=4,
                             ms_per_step=ms_e2e / args.steps,
                             reader='Trainer.step(pinned host batch) per step; each loss copied to pinned host memory (non-blocking), one wait at the end',
                             blocking_read=dict(ms_per_step=ms_e2e_blocking / args.steps,
                                                value=tokens_per_step * args.steps / (ms_e2e_blocking / 1e3),
                                                reader='loss.item() after every step (the reference train.py style)')),
                    gpu_launches=int(launches), clocks=clocks, roofline=roofline, final_loss=final_loss,
                    per_rank_ms_per_step=per_rank_ms)
        if comm:
            line['comm'] = comm
        if not args.no_cpu_baseline and world == 1:
            cores = cpu_threads()
            v, sec, rows, timed = cpu_port_tokens_per_sec(kw, steps=30, warmup=1, rows=1, budget_s=20.0)
            line['cpu_baseline'] = dict(value=v, unit='tokens/s', cores=cores, kind='port',
                                        sample=f'{rows} sequence x {n} tokens per step, fwd+bwd fp32, {timed} timed steps of {sec:.2f} s')
        print(json.dumps(line), flush=True)
    if world > 1:
        # drop the captured graph (it references the communicator) before tearing NCCL down
        tr._graph = None
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


def eng_bytes(eng):
    tot = 0
    for s in eng.lay:
        for v in s.values():
            tot += v.numel() * v.element_size()
    for x in eng.X:
        tot += x.numel() * 4
    return tot


if __name__ == '__main__':
    main()
