"""Per-sequence depthwise 1-D convolution on the GPU: forward and backward (grad_in, grad_weight, grad_bias) at the cfg2 /
cfg3 / cfg5 shapes in bf16, K = 4 causal and K = 31 same, against the same-run device-to-device copy of the payload and
two same-GPU baselines:
  (a) pad (x.left(0)) -> F.conv1d(groups=H) on (B, H, T) -> unpad, forward and autograd backward (cfg2),
  (b) the sum over k of masked shifted gathers of the C rows (cfg3, where the padded batch of (a) does not fit).
Times are CUDA-event medians of 20 calls after 5 warm-ups; every input is larger than the 126 MB L2.

    python benchmarks/conv.py [--out profiles/r4_conv]     # writes <out>.json and <out>.md
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torchrua_b200 as rua  # noqa: E402
from torchrua_b200 import _lib, _native  # noqa: E402
from torchrua_b200._native import SideSpec  # noqa: E402

CONVS = (('K4 causal', 4, 'causal'), ('K31 same', 31, 'same'))


def timed(fn, warmup=5, reps=20):
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
    rng = np.random.default_rng(0)
    yield 'cfg2', rng.integers(1, 513, 4096), 1024, ('C', 'P', 'L'), CONVS
    yield 'cfg3', np.minimum(np.random.default_rng(0).zipf(1.5, 16384), 4096), 4096, ('C',), CONVS
    yield 'cfg5', np.random.default_rng(0).integers(1, 65, 1 << 20), 1, ('C',), CONVS[:1]


def layout_of(c, kind):
    if kind == 'C':
        return c, c.data, SideSpec(_lib.CAT, rows=c.data.shape[0])
    if kind == 'P':
        p = c.pack()
        return p, p.data, SideSpec(_lib.PACK, rows=p.data.shape[0])
    z = c.left(0)
    b, w = z.data.shape[:2]
    return z, z.data.flatten(0, 1), SideSpec(_lib.LEFT, width=w, rows=b * w)


def padded_conv(c, w, b, pad):
    """baseline (a): pad -> F.conv1d(groups=H) on (B, H, T) -> unpad"""
    z = c.left(0)
    H, K = w.shape
    y = F.conv1d(F.pad(z.data.transpose(1, 2), (pad, K - 1 - pad)), w.view(H, 1, K), b, groups=H)
    return rua.L(data=y.transpose(1, 2), token_sizes=c.token_sizes).cat().data


def shifted_gathers(x, lens, w, b, pad, cols=1024):
    """baseline (b): sum over k of the C rows shifted by k - pad, masked where the shift leaves the sequence; fp32
    accumulation, `cols` feature columns at a time to bound the temporaries"""
    N = x.shape[0]
    seg = torch.repeat_interleave(torch.arange(len(lens), device=x.device), lens)
    start = (torch.cumsum(lens, 0) - lens)[seg]
    t = torch.arange(N, device=x.device) - start
    ln = lens[seg]
    out = torch.empty_like(x)
    shifts = []
    for k in range(w.shape[1]):
        s = t + k - pad
        shifts.append(((start + s).clamp(0, N - 1), ((s >= 0) & (s < ln))[:, None]))
    for c0 in range(0, x.shape[1], cols):
        xs = x[:, c0:c0 + cols]
        acc = b[c0:c0 + cols].float().expand(N, -1).clone()
        for k, (rows, ok) in enumerate(shifts):
            acc += xs[rows].float() * ok * w[c0:c0 + cols, k].float()
        out[:, c0:c0 + cols] = acc
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r4_conv'))
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'benchmarks/conv.py measures on a CUDA device'
    dev = torch.device('cuda')
    name = torch.cuda.get_device_name(dev)
    try:
        power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    print(f'# {name}, power limit {power}', flush=True)
    rows = []
    for cfg, lens_np, H, kinds, convs in shapes():
        lens = torch.tensor(lens_np, dtype=torch.long, device=dev)
        N = int(lens_np.sum())
        g = torch.Generator(device=dev).manual_seed(0)
        x = torch.randn((N, H), generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)
        D = H * x.element_size()
        c = rua.C(data=x, token_sizes=lens)
        t_copy = timed(lambda: torch.empty_like(x).copy_(x))
        peak = 2 * N * D / t_copy
        print(f'{cfg}: N={N} D={D} copy {t_copy * 1e3:.3f} ms = {peak / 1e12:.2f} TB/s', flush=True)
        for label, K, padding in convs:
            pad = K - 1 if padding == 'causal' else (K - 1) // 2
            w = (torch.randn((H, K), generator=g, device=dev) / K).to(torch.bfloat16)
            b = torch.randn((H,), generator=g, device=dev).to(torch.bfloat16)
            for kind in kinds:
                z, flat, side = layout_of(c, kind)
                rg = z._ragged()
                meta = 8 * len(lens_np) + (8 * (rg.Tp + rg.B) if kind == 'P' else 0)
                n_rows = flat.shape[0]
                t_api = timed(lambda: z.depthwise_conv1d(w, b, padding=padding))
                t_fwd = timed(lambda: _native._conv_raw(flat, w, b, pad, rg, side))
                fwd_bytes = 2 * n_rows * D + 2 * (K + 1) * H + meta
                gout = torch.randn_like(flat)
                t_bwd = timed(lambda: _native._conv_backward_raw(gout, flat, w, pad, rg, side, True, True, True))
                bwd_bytes = 3 * n_rows * D + 2 * (2 * K + 1) * H + meta
                data, ww, bb = z.data.clone().requires_grad_(True), w.clone().requires_grad_(True), \
                    b.clone().requires_grad_(True)
                y = z._replace(data=data).depthwise_conv1d(ww, bb, padding=padding).data
                gy = torch.randn_like(y)
                t_api_bwd = timed(lambda: torch.autograd.grad(y, (data, ww, bb), gy, retain_graph=True))
                del data, ww, bb, y, gy
                rec = dict(cfg=cfg, layout=kind, conv=label, K=K, pad=pad, N=N, H=H, rows=n_rows, dtype='bfloat16',
                           api_ms=t_api * 1e3, fwd_ms=t_fwd * 1e3, fwd_bytes=fwd_bytes,
                           fwd_frac_copy=fwd_bytes / t_fwd / peak, api_bwd_ms=t_api_bwd * 1e3, bwd_ms=t_bwd * 1e3,
                           bwd_bytes=bwd_bytes, bwd_frac_copy=bwd_bytes / t_bwd / peak, copy_ms=t_copy * 1e3,
                           copy_TBps=peak / 1e12)
                del gout
                if cfg == 'cfg2' and kind == 'C':
                    rec['baseline_pad_ms'] = timed(lambda: padded_conv(c, w, b, pad)) * 1e3
                    xa, wa, ba = x.clone().requires_grad_(True), w.clone().requires_grad_(True), \
                        b.clone().requires_grad_(True)
                    ya = padded_conv(rua.C(data=xa, token_sizes=lens), wa, ba, pad)
                    ga = torch.randn_like(ya)
                    rec['baseline_pad_bwd_ms'] = timed(lambda: torch.autograd.grad(ya, (xa, wa, ba), ga,
                                                                                   retain_graph=True)) * 1e3
                    del xa, wa, ba, ya, ga
                    rec['floor_holds'] = rec['api_ms'] < rec['baseline_pad_ms'] and \
                        rec['api_bwd_ms'] < rec['baseline_pad_bwd_ms']
                    got = c.depthwise_conv1d(w, b, padding=padding).data.float()
                    want = padded_conv(c, w, b, pad).float()
                    rec['baseline_pad_max_abs_diff'] = float((got - want).abs().max())
                    rec['max_abs_out'] = float(want.abs().max())
                    del got, want
                if cfg == 'cfg3':
                    rec['baseline_gather_ms'] = timed(lambda: shifted_gathers(x, lens, w, b, pad), warmup=2,
                                                      reps=5) * 1e3
                    got = c.depthwise_conv1d(w, b, padding=padding).data.float()
                    want = shifted_gathers(x, lens, w, b, pad).float()
                    rec['baseline_gather_max_abs_diff'] = float((got - want).abs().max())
                    del got, want
                rows.append(rec)
                print(json.dumps(rec), flush=True)
                torch.cuda.empty_cache()
        del x, c
        torch.cuda.empty_cache()
    info = dict(gpu=name, power_limit=power, results=rows)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out + '.json', 'w') as f:
        json.dump(info, f, indent=1)
    floor = [r for r in rows if 'floor_holds' in r]
    ok = all(r['floor_holds'] for r in floor)
    with open(args.out + '.md', 'w') as f:
        f.write(f'# Per-sequence depthwise conv1d -- {name}, power limit {power}\n\n')
        f.write('Written by `python benchmarks/conv.py`.  bf16 payload, weight and bias.  fwd / bwd = kernel call '
                '(CUDA-event median of 20; bwd computes grad_in, grad_weight and grad_bias); "% copy" = algorithmic bytes '
                'over time, against a device-to-device copy of the same payload timed in the same run.  api = the public '
                'method (metadata cached); api bwd = torch.autograd.grad through it.\n\n')
        f.write('| shape | layout | conv | api ms | fwd ms | fwd % copy | api bwd ms | bwd ms | bwd % copy | '
                'baseline ms (fwd / bwd) | copy TB/s |\n|---|---|---|---|---|---|---|---|---|---|---|\n')
        for r in rows:
            if 'baseline_pad_ms' in r:
                base = f"(a) {r['baseline_pad_ms']:.3f} / {r['baseline_pad_bwd_ms']:.3f}"
            elif 'baseline_gather_ms' in r:
                base = f"(b) {r['baseline_gather_ms']:.3f} / --"
            else:
                base = ''
            f.write(f"| {r['cfg']} | {r['layout']} | {r['conv']} | {r['api_ms']:.3f} | {r['fwd_ms']:.3f} | "
                    f"{100 * r['fwd_frac_copy']:.1f} | {r['api_bwd_ms']:.3f} | {r['bwd_ms']:.3f} | "
                    f"{100 * r['bwd_frac_copy']:.1f} | {base} | {r['copy_TBps']:.2f} |\n")
        f.write('\n')
        for r in rows:
            if 'baseline_pad_max_abs_diff' in r:
                f.write(f"cfg2 {r['conv']}: max abs difference to baseline (a) {r['baseline_pad_max_abs_diff']:.3g} "
                        f"(outputs up to {r['max_abs_out']:.3g}; both round to bf16).\n\n")
            if 'baseline_gather_max_abs_diff' in r:
                f.write(f"cfg3 {r['conv']}: max abs difference to baseline (b) {r['baseline_gather_max_abs_diff']:.3g}.\n\n")
        f.write(f"Hard floor (cfg2, forward and backward through the public API faster than baseline (a), both K): "
                f"{'HOLDS' if ok else 'FAILS'}.\n")
    print('wrote', args.out + '.md')
    print('hard floor', 'HOLDS' if ok else 'FAILS')
    if not ok:
        sys.exit(1)


if __name__ == '__main__':
    main()
