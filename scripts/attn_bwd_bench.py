"""Time the tcgen05 attention backward alone, every kernel variant (progen_local_attn_bwd_tc_ex `mode`), at the cfg2 and
cfg3 attention shapes, with the engine's rotary tables.  Modes alternate inside each round, so a slow stretch of the
shared machine hits every mode; each (shape, mode) prints the median, min and max over the rounds.

    python scripts/attn_bwd_bench.py [--rounds 5] [--iters 50] [--modes 0,1,2,3] [--out FILE.jsonl]

One call = one layer's backward (dQ + dK/dV kernels).  Algorithmic FLOPs: 5 matrix products (S, dP, dV, dK, dQ) of
2 * dim_head FLOPs per (query, visible key, head), with w + (w + 1) / 2 visible keys per query (window-0 queries counted
as if they had a look-back window too).  The inputs (~0.4 GB at cfg2) exceed the 126 MB L2 between calls.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from progen_b200 import lib as L  # noqa: E402

SHAPES = {'cfg2': (64, 1024, 256, 8), 'cfg3': (8, 2048, 512, 16)}      # B, seq_len, window, heads (dim_head 64)


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(',')]
        return dict(card=name, power_limit=power, max_sm_clock=clock)
    except Exception:           # no nvidia-smi: the name from the runtime, power limit unknown
        return dict(card=torch.cuda.get_device_name(), power_limit='unknown', max_sm_clock='unknown')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--iters', type=int, default=50)
    ap.add_argument('--modes', default='0,1,2,3')
    ap.add_argument('--shapes', default='cfg2,cfg3')
    ap.add_argument('--out', default=None, help='also append the JSON lines to this file')
    args = ap.parse_args()
    L.require_device()
    lib = L.load()
    modes = [int(m) for m in args.modes.split(',')]
    info = card()
    lines = []
    for shape in args.shapes.split(','):
        B, n, w, h = SHAPES[shape]
        dh = 64
        T, I = B * n, h * dh
        g = torch.Generator(device='cuda').manual_seed(1)
        qkv = (torch.randn(T, 3 * I, generator=g, device='cuda') * 1.5).bfloat16()
        dout = torch.randn(T, I, generator=g, device='cuda').bfloat16()
        out = torch.empty(T, I, device='cuda', dtype=torch.bfloat16)
        lse = torch.empty(T, h, device='cuda')
        delta = torch.empty(T, h, device='cuda')
        dqkv = torch.empty_like(qkv)
        L.check(lib.progen_local_attn_fwd_tc(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), B, n, w, h, dh, L.stream()))
        inv_freq = 1.0 / (10000 ** (torch.arange(0, dh, 2, dtype=torch.float64) / dh))
        ang = torch.arange(n, dtype=torch.float64)[:, None] * inv_freq[None, :]
        sin, cos = torch.sin(ang).float().cuda().contiguous(), torch.cos(ang).float().cuda().contiguous()
        sin_t, cos_t = sin.t().contiguous(), cos.t().contiguous()

        def call(mode):
            L.check(lib.progen_local_attn_bwd_tc_ex(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(),
                                                    dqkv.data_ptr(), delta.data_ptr(), sin.data_ptr(), cos.data_ptr(),
                                                    sin_t.data_ptr(), cos_t.data_ptr(), B, n, w, h, dh, mode, L.stream()))

        for m in modes:                                   # warm every mode (module load, tensor-map cache)
            for _ in range(3):
                call(m)
        torch.cuda.synchronize()
        times = {m: [] for m in modes}
        for _ in range(args.rounds):
            for m in modes:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.iters):
                    call(m)
                b.record()
                b.synchronize()
                times[m].append(a.elapsed_time(b) * 1e3 / args.iters)
        flops = 10.0 * I * (w + (w + 1) / 2) * T
        for m in modes:
            med = statistics.median(times[m])
            line = dict(shape=shape, B=B, seq_len=n, window=w, heads=h, mode=m, rotary=True, us_per_layer=round(med, 1),
                        us_min=round(min(times[m]), 1), us_max=round(max(times[m]), 1),
                        spread_pct=round(100 * (max(times[m]) - min(times[m])) / med, 2),
                        tflops_alg=round(flops / (med * 1e-6) / 1e12, 1), rounds=args.rounds, iters=args.iters, **info)
            lines.append(line)
            print(json.dumps(line), flush=True)
    if args.out:
        with open(args.out, 'a') as f:
            for line in lines:
                f.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
