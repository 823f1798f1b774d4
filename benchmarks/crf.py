"""Per-sequence linear-chain CRF on the GPU: the log-likelihood forward, its backward (gradients of the emissions,
transitions, start and end) and Viterbi decode at the cfg2 / cfg3 / cfg5 lengths, against two same-GPU baselines:
  (a) pad (x.left(0)) -> the pytorch-crf-style masked loop over T, alpha = logsumexp(alpha[:, :, None] + W + x_t[:, None,
      :], 1), in the emissions' dtype -> autograd backward (backward at cfg2 and cfg5 only: cfg3's graph keeps 4096 (B, K, K)
      temporaries and does not fit),
  (b) pad -> the same loop in max-plus with (B, K) backpointers per step -> a torch backtrack over T.
Times are CUDA-event medians after warm-up.  HBM traffic is negligible here (cfg2 K = 32 bf16 emissions are 67 MB), so
the yardstick is the exponential floor: N K^2 exponentials for the forward and for the backward kernel, at 16 MUFU ex2
per clock per SM on 148 SMs at the card's maximum SM clock read in the same run.  Decode takes no exponential; its floor
is the issue floor of 4 instructions (two shared loads, an add, a compare-select) per (token, a, b) at 128 lanes per clock
per SM.

    python benchmarks/crf.py [--out profiles/r6_crf]     # writes <out>.json and <out>.md
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torchrua_b200 as rua  # noqa: E402

SMS, MUFU_PER_CLK, LANES_PER_CLK, DECODE_INSTR = 148, 16, 128, 4


def timed(fn, warmup=3, reps=10):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) * 1e-3)
    return float(np.median(times))


def shapes():
    cfg2 = np.random.default_rng(0).integers(1, 513, 4096)
    for K in (9, 32, 64):
        for dtype in (torch.bfloat16, torch.float32):
            yield 'cfg2', cfg2, K, dtype, True
    yield 'cfg3', np.minimum(np.random.default_rng(0).zipf(1.5, 16384), 4096), 32, torch.bfloat16, False
    yield 'cfg5', np.random.default_rng(0).integers(1, 65, 1 << 20), 9, torch.float32, True


def baseline_ll(c, tl, W, st, en):
    """pad -> masked forward-algorithm loop over T -> score(tags) - log Z"""
    z = c.left(0)
    x, lens = z.data, z.token_sizes
    B, T, _ = x.shape
    mask = torch.arange(T, device=x.device)[None] < lens[:, None]
    alpha = st + x[:, 0]
    for t in range(1, T):
        nxt = torch.logsumexp(alpha[:, :, None] + W + x[:, t, None, :], dim=1)
        alpha = torch.where(mask[:, t, None], nxt, alpha)
    log_z = torch.logsumexp(alpha + en, dim=1)
    y = tl.clamp(min=0)
    s = (x.gather(2, y[..., None])[..., 0] * mask).sum(1)
    s = s + (W[y[:, :-1], y[:, 1:]] * mask[:, 1:]).sum(1)
    s = s + st[y[:, 0]] + en[y.gather(1, (lens - 1)[:, None])[:, 0]]
    return s - log_z


def baseline_viterbi(c, W, st, en):
    """pad -> max-plus loop over T with backpointers -> torch backtrack"""
    z = c.left(0)
    x, lens = z.data, z.token_sizes
    B, T, _ = x.shape
    mask = torch.arange(T, device=x.device)[None] < lens[:, None]
    alpha = st + x[:, 0]
    bps = []
    for t in range(1, T):
        best, arg = (alpha[:, :, None] + W).max(dim=1)
        bps.append(arg)
        alpha = torch.where(mask[:, t, None], best + x[:, t], alpha)
    score, y = (alpha + en).max(dim=1)   # alpha stops at each sequence's last token: y is its last tag
    out = torch.empty((B, T), dtype=torch.long, device=x.device)
    for t in range(T - 1, -1, -1):
        out[:, t] = y
        if t > 0:
            y = torch.where(mask[:, t], bps[t - 1].gather(1, y[:, None])[:, 0], y)
    return out, score


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r6_crf'))
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'benchmarks/crf.py measures on a CUDA device'
    dev = torch.device('cuda')
    name = torch.cuda.get_device_name(dev)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader,nounits', '-i',
                            '0'], capture_output=True, text=True, timeout=30).stdout.strip().split(',')
        power, clock_mhz = q[0].strip() + ' W', float(q[1])
    except (OSError, subprocess.SubprocessError, ValueError, IndexError):
        power, clock_mhz = 'unknown', float('nan')
    print(f'# {name}, power limit {power}, max SM clock {clock_mhz} MHz', flush=True)
    rows = []
    for cfg, lens_np, K, dtype, loop_bwd in shapes():
        lens = torch.tensor(lens_np, dtype=torch.long, device=dev)
        N, B = int(lens_np.sum()), len(lens_np)
        g = torch.Generator(device=dev).manual_seed(0)
        x = torch.randn((N, K), generator=g, device=dev).to(dtype)
        W, st, en = (torch.randn(s, generator=g, device=dev).to(dtype) for s in ((K, K), (K,), (K,)))
        tags = torch.randint(0, K, (N,), generator=g, device=dev)
        gout = torch.randn(B, generator=g, device=dev)
        c = rua.C(data=x, token_sizes=lens)
        rec = dict(cfg=cfg, K=K, dtype=str(dtype).replace('torch.', ''), N=N, B=B)
        rec['fwd_ms'] = timed(lambda: rua.segment_crf_log_likelihood(x, lens, tags, W, st, en)) * 1e3
        leaves = [t.detach().requires_grad_(True) for t in (x, W, st, en)]
        ll = rua.segment_crf_log_likelihood(leaves[0], lens, tags, *leaves[1:])
        rec['bwd_ms'] = timed(lambda: torch.autograd.grad(ll, leaves, gout, retain_graph=True)) * 1e3
        del ll
        rec['decode_ms'] = timed(lambda: rua.segment_crf_decode(x, lens, W, st, en)) * 1e3
        floor = N * K * K / (SMS * MUFU_PER_CLK * clock_mhz * 1e6)
        rec['exp_floor_ms'] = floor * 1e3
        rec['fwd_frac_floor'] = floor * 1e3 / rec['fwd_ms']
        rec['bwd_frac_floor'] = floor * 1e3 / rec['bwd_ms']
        dfloor = N * K * K * DECODE_INSTR / (SMS * LANES_PER_CLK * clock_mhz * 1e6)
        rec['decode_floor_ms'] = dfloor * 1e3
        rec['decode_frac_floor'] = dfloor * 1e3 / rec['decode_ms']
        tl = rua.C(data=tags, token_sizes=lens).left(0).data
        reps = 3 if cfg == 'cfg3' else 5
        rec['loop_fwd_ms'] = timed(lambda: baseline_ll(c, tl, W, st, en), warmup=1, reps=reps) * 1e3
        rec['loop_decode_ms'] = timed(lambda: baseline_viterbi(c, W, st, en), warmup=1, reps=reps) * 1e3
        rec['fwd_speedup'] = rec['loop_fwd_ms'] / rec['fwd_ms']
        rec['decode_speedup'] = rec['loop_decode_ms'] / rec['decode_ms']
        if loop_bwd:
            lb = baseline_ll(rua.C(data=leaves[0], token_sizes=lens), tl, *leaves[1:])
            rec['loop_bwd_ms'] = timed(lambda: torch.autograd.grad(lb, leaves, gout.to(lb.dtype), retain_graph=True),
                                       warmup=1, reps=reps) * 1e3
            del lb
            rec['fwd_bwd_speedup'] = (rec['loop_fwd_ms'] + rec['loop_bwd_ms']) / (rec['fwd_ms'] + rec['bwd_ms'])
        # accuracy of both against fp64 on the same values
        ref = rua.segment_crf_log_likelihood(x.double(), lens, tags, W.double(), st.double(), en.double())
        rec['max_abs_err'] = float((rua.segment_crf_log_likelihood(x, lens, tags, W, st, en).double() - ref).abs().max())
        if cfg != 'cfg3':
            rec['loop_max_abs_err'] = float((baseline_ll(c, tl, W, st, en).double() - ref).abs().max())
        del ref, leaves, c
        torch.cuda.empty_cache()
        rows.append(rec)
        print(json.dumps(rec), flush=True)
    info = dict(gpu=name, power_limit=power, max_sm_clock_mhz=clock_mhz, results=rows)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out + '.json', 'w') as f:
        json.dump(info, f, indent=1)
    target = [r for r in rows if r['cfg'] == 'cfg2' and r['K'] == 32]
    with open(args.out + '.md', 'w') as f:
        f.write(f'# Per-sequence linear-chain CRF -- {name}, power limit {power}, max SM clock {clock_mhz:.0f} MHz\n\n')
        f.write('Written by `python benchmarks/crf.py`.  fwd = `segment_crf_log_likelihood` (log Z and the gold score in '
                'one pass); bwd = autograd backward of it (gradients of emissions, transitions, start and end); decode = '
                '`segment_crf_decode`.  CUDA-event medians.  loop = pad -> masked forward-algorithm loop over T in torch '
                '(autograd for bwd); loop decode = the max-plus loop + torch backtrack.  "% floor" = the exponential floor '
                '(N K^2 MUFU ex2 at 16 / clock / SM) over the time, for fwd and bwd; for decode the issue floor of 4 '
                'instructions per (token, a, b).  Both kernels are latency-bound, not HBM-bound.\n\n')
        f.write('| shape | K | dtype | fwd ms | bwd ms | decode ms | fwd % floor | bwd % floor | decode % floor | '
                'loop fwd ms | loop bwd ms | loop decode ms | fwd x | fwd+bwd x | decode x |\n'
                '|---|---|---|---|---|---|---|---|---|---|---|---|---|---|---|\n')
        for r in rows:
            f.write(f"| {r['cfg']} | {r['K']} | {r['dtype']} | {r['fwd_ms']:.3f} | {r['bwd_ms']:.3f} | "
                    f"{r['decode_ms']:.3f} | {100 * r['fwd_frac_floor']:.1f} | {100 * r['bwd_frac_floor']:.1f} | "
                    f"{100 * r['decode_frac_floor']:.1f} | {r['loop_fwd_ms']:.1f} | "
                    f"{r.get('loop_bwd_ms', float('nan')):.1f} | {r['loop_decode_ms']:.1f} | {r['fwd_speedup']:.1f} | "
                    f"{r.get('fwd_bwd_speedup', float('nan')):.1f} | {r['decode_speedup']:.1f} |\n")
        f.write('\nMax abs error of the log-likelihood against fp64 on the same values: ' +
                ', '.join(f"{r['cfg']} K={r['K']} {r['dtype']}: {r['max_abs_err']:.3g}"
                          + (f" (loop {r['loop_max_abs_err']:.3g})" if 'loop_max_abs_err' in r else '') for r in rows)
                + '.\n')
        for r in target:
            ok = r['fwd_bwd_speedup'] >= 10
            f.write(f"\nTarget (cfg2 K = 32 {r['dtype']}, forward + backward at least 10x the padded loop): "
                    f"{'MET' if ok else 'MISSED'} ({r['fwd_bwd_speedup']:.1f}x).\n")
    print('wrote', args.out + '.md')


if __name__ == '__main__':
    main()
