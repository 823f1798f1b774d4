"""Per-sequence gated linear recurrence h_t = a_t h_(t-1) + x_t on the GPU: forward and backward (all three gradients) at
the cfg2 / cfg3 / cfg5 shapes, against the same-run device-to-device copy of the same bytes and three same-GPU baselines:
  (a) pad -> a Python loop over T (three elementwise launches per step) -> unpad, forward and autograd backward (cfg2),
  (b) the log-space closed form h = exp(A) * segment_cumsum(x * exp(-A)), A = segment_cumsum(log a), with its error,
  (c) segment_cumsum on the same payload (the same kernel structure, 2/3 of the bytes).
Gates are uniform in (0.5, 1).  Times are CUDA-event medians of >= 20 calls after 5 warm-ups; every input is larger
than the 126 MB L2.

    python benchmarks/linrec.py [--out profiles/r5_linrec]     # writes <out>.json and <out>.md
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
from torchrua_b200 import _lib, _native  # noqa: E402
from torchrua_b200._native import SideSpec  # noqa: E402


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
    yield 'cfg2', rng.integers(1, 513, 4096), 1024, torch.bfloat16, ('C', 'P', 'L')
    yield 'cfg3', np.minimum(np.random.default_rng(0).zipf(1.5, 16384), 4096), 4096, torch.bfloat16, ('C', 'P')
    yield 'cfg5', np.random.default_rng(0).integers(1, 65, 1 << 20), 1, torch.float32, ('C',)


def layout_of(c, kind):
    if kind == 'C':
        return c, c.data, SideSpec(_lib.CAT, rows=c.data.shape[0])
    if kind == 'P':
        p = c.pack()
        return p, p.data, SideSpec(_lib.PACK, rows=p.data.shape[0])
    z = c.left(0)
    b, w = z.data.shape[:2]
    return z, z.data.flatten(0, 1), SideSpec(_lib.LEFT, width=w, rows=b * w)


def same_layout(c, kind, t):
    z = rua.C(data=t, token_sizes=c.token_sizes)
    return z if kind == 'C' else (z.pack() if kind == 'P' else z.left(0))


def baseline_loop(c, a, h0):
    """pad -> h = a_t * h + x_t over T in Python -> unpad"""
    zx, za = c.left(0), rua.C(data=a, token_sizes=c.token_sizes).left(0)
    h, outs = h0, []
    for t in range(zx.data.shape[1]):
        h = za.data[:, t] * h + zx.data[:, t]
        outs.append(h)
    return rua.L(data=torch.stack(outs, 1), token_sizes=c.token_sizes).cat().data


def baseline_logspace(x, a, lens):
    A = rua.segment_cumsum(torch.log(a), lens)
    return torch.exp(A) * rua.segment_cumsum(x * torch.exp(-A), lens)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r5_linrec'))
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'benchmarks/linrec.py measures on a CUDA device'
    dev = torch.device('cuda')
    name = torch.cuda.get_device_name(dev)
    try:
        power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    print(f'# {name}, power limit {power}', flush=True)
    rows = []
    for cfg, lens_np, H, dtype, kinds in shapes():
        lens = torch.tensor(lens_np, dtype=torch.long, device=dev)
        N, B = int(lens_np.sum()), len(lens_np)
        g = torch.Generator(device=dev).manual_seed(0)
        x = torch.randn((N, H), generator=g, device=dev, dtype=torch.float32).to(dtype)
        a = (0.5 + 0.5 * torch.rand((N, H), generator=g, device=dev, dtype=torch.float32)).to(dtype)
        h0 = torch.randn((B, H), generator=g, device=dev, dtype=torch.float32).to(dtype)
        D = H * x.element_size()
        c = rua.C(data=x, token_sizes=lens)
        t_copy = timed(lambda: torch.empty_like(x).copy_(x))
        peak = 2 * N * D / t_copy
        print(f'{cfg}: N={N} D={D} copy {t_copy * 1e3:.3f} ms = {peak / 1e12:.2f} TB/s', flush=True)
        for kind in kinds:
            z, flat, side = layout_of(c, kind)
            za = same_layout(c, kind, a)
            aflat = za.data.flatten(0, 1) if kind == 'L' else za.data
            rg = z._ragged()
            meta = 8 * B + (8 * (rg.Tp + rg.B) if kind == 'P' else 0)
            rows_moved = flat.shape[0]
            t_api = timed(lambda: z.linear_recurrence(za.data, h0))
            t_fwd = timed(lambda: _native._linrec_raw(flat, aflat, h0, rg, side, False))
            y = _native._linrec_raw(flat, aflat, h0, rg, side, False)
            gout = torch.randn_like(y)
            t_bwd = timed(lambda: _native._linrec_backward_raw(gout, aflat, h0, y, rg, side, False, True, True, True))
            t_cumsum = timed(lambda: _native._scan_raw(flat, rg, side, _lib.SCAN_SUM, False))
            fwd_bytes = 3 * rows_moved * D + B * D + meta
            bwd_bytes = 5 * rows_moved * D + 2 * B * D + meta
            rec = dict(cfg=cfg, layout=kind, N=N, H=H, dtype=str(dtype).replace('torch.', ''), api_ms=t_api * 1e3,
                       fwd_ms=t_fwd * 1e3, fwd_bytes=fwd_bytes, fwd_frac_copy=fwd_bytes / t_fwd / peak,
                       bwd_ms=t_bwd * 1e3, bwd_bytes=bwd_bytes, bwd_frac_copy=bwd_bytes / t_bwd / peak,
                       cumsum_ms=t_cumsum * 1e3, fwd_over_cumsum=t_fwd / t_cumsum, copy_ms=t_copy * 1e3,
                       copy_TBps=peak / 1e12)
            del y, gout
            if cfg == 'cfg2' and kind == 'C':
                # public API forward + backward (all three gradients) against baseline (a)
                xs, as_, hs = (t.clone().requires_grad_(True) for t in (x, a, h0))
                yg = rua.segment_linear_recurrence(xs, lens, as_, hs)
                gy = torch.randn_like(yg)
                rec['api_bwd_ms'] = timed(lambda: torch.autograd.grad(yg, (xs, as_, hs), gy, retain_graph=True)) * 1e3
                del yg
                rec['baseline_loop_ms'] = timed(lambda: baseline_loop(c, a, h0), warmup=2, reps=5) * 1e3
                yl = baseline_loop(rua.C(data=xs, token_sizes=lens), as_, hs)
                rec['baseline_loop_bwd_ms'] = timed(lambda: torch.autograd.grad(yl, (xs, as_, hs), gy, retain_graph=True),
                                                    warmup=2, reps=5) * 1e3
                del yl, xs, as_, hs, gy
                rec['faster_than_loop'] = rec['api_ms'] < rec['baseline_loop_ms'] and \
                    rec['api_bwd_ms'] < rec['baseline_loop_bwd_ms']   # the hard floor at cfg2
                rec['target_fwd_le_1p5_cumsum'] = rec['fwd_over_cumsum'] <= 1.5
                ref = rua.segment_linear_recurrence(x.double(), lens, a.double(), h0.double())
                got = rua.segment_linear_recurrence(x, lens, a, h0)
                rec['linrec_max_abs_err'] = float((got.double() - ref).abs().max())
                loop = baseline_loop(c, a, h0)
                rec['baseline_loop_max_abs_err'] = float((loop.double() - ref).abs().max())
                del got, loop
                ref0 = rua.segment_linear_recurrence(x.double(), lens, a.double())
                rec['baseline_logspace_ms'] = timed(lambda: baseline_logspace(x, a, lens)) * 1e3
                err = (baseline_logspace(x, a, lens).double() - ref0).abs()
                rec['baseline_logspace_max_abs_err'] = float(err.nan_to_num(float('inf')).max())
                rec['baseline_logspace_nonfinite'] = int((~torch.isfinite(err)).sum())
                del ref, ref0, err
            rows.append(rec)
            print(json.dumps(rec), flush=True)
        del x, a, h0, c
        torch.cuda.empty_cache()
    info = dict(gpu=name, power_limit=power, results=rows)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out + '.json', 'w') as f:
        json.dump(info, f, indent=1)
    floor = [r for r in rows if 'faster_than_loop' in r]
    ok = all(r['faster_than_loop'] for r in floor)
    with open(args.out + '.md', 'w') as f:
        f.write(f'# Per-sequence gated linear recurrence -- {name}, power limit {power}\n\n')
        f.write('Written by `python benchmarks/linrec.py`.  fwd / bwd = kernel call (CUDA-event median of 20; bwd computes '
                'all three gradients); "% copy" = algorithmic bytes (fwd 3·N·D, bwd 5·N·D, + initial states + metadata) '
                'over time, against a device-to-device copy of the same payload timed in the same run.  api = the public '
                'method, forward only (metadata cached).  cumsum = segment_cumsum\'s kernel on the same storage.\n\n')
        f.write('| shape | layout | api ms | fwd ms | fwd % copy | bwd ms | bwd % copy | cumsum ms | fwd / cumsum | '
                'copy TB/s |\n|---|---|---|---|---|---|---|---|---|---|\n')
        for r in rows:
            f.write(f"| {r['cfg']} | {r['layout']} | {r['api_ms']:.3f} | {r['fwd_ms']:.3f} | "
                    f"{100 * r['fwd_frac_copy']:.1f} | {r['bwd_ms']:.3f} | {100 * r['bwd_frac_copy']:.1f} | "
                    f"{r['cumsum_ms']:.3f} | {r['fwd_over_cumsum']:.2f} | {r['copy_TBps']:.2f} |\n")
        for r in floor:
            f.write(f"\nBaseline (a), cfg2 C: pad -> Python loop over T -> unpad {r['baseline_loop_ms']:.2f} ms forward, "
                    f"{r['baseline_loop_bwd_ms']:.2f} ms autograd backward; segment_linear_recurrence "
                    f"{r['api_ms']:.3f} ms / {r['api_bwd_ms']:.3f} ms.  Max abs error against fp64: loop "
                    f"{r['baseline_loop_max_abs_err']:.3g}, segment_linear_recurrence {r['linrec_max_abs_err']:.3g}.\n")
            f.write(f"\nBaseline (b), cfg2 C, no initial state: log-space closed form {r['baseline_logspace_ms']:.3f} ms, "
                    f"max abs error {r['baseline_logspace_max_abs_err']:.3g} against fp64 "
                    f"({r['baseline_logspace_nonfinite']} non-finite outputs).\n")
            f.write(f"\nTarget (cfg2 C bf16 forward at most 1.5x segment_cumsum's kernel on the same payload): "
                    f"{'MET' if r['target_fwd_le_1p5_cumsum'] else 'MISSED'} ({r['fwd_over_cumsum']:.2f}x).\n")
        f.write(f"\nHard floor (cfg2, public API forward and backward faster than baseline (a)): "
                f"{'HOLDS' if ok else 'MISSED'}.\n")
    print('wrote', args.out + '.md')
    if not ok:
        print('hard floor missed at cfg2')
        sys.exit(1)


if __name__ == '__main__':
    main()
