"""Per-sequence prefix scans on the GPU: forward and backward of every op at the cfg2 / cfg3 / cfg5 shapes, against the
same-run device-to-device copy of the same bytes and three same-GPU baselines:
  (a) pad -> torch op along dim 1 -> unpad through this package's conversions (cfg2),
  (b) a global torch.cumsum minus the value before each segment (cumsum only; reported with its error),
  (c) segment_sum on the same shape (one read of the payload).
Times are CUDA-event medians of >= 20 calls after 5 warm-ups; every input is larger than the 126 MB L2.

    python benchmarks/scan.py [--out profiles/r3_scan]     # writes <out>.json and <out>.md
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

OPS = {'cumsum': 'sum', 'logcumsumexp': 'logsumexp', 'cummax': 'max', 'cummin': 'min'}
TORCH = {'sum': torch.cumsum, 'logsumexp': torch.logcumsumexp, 'max': torch.cummax, 'min': torch.cummin}
FILL = {'sum': 0.0, 'logsumexp': float('-inf'), 'max': float('-inf'), 'min': float('inf')}


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r3_scan'))
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'benchmarks/scan.py measures on a CUDA device'
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
        N = int(lens_np.sum())
        g = torch.Generator(device=dev).manual_seed(0)
        x = torch.randn((N, H), generator=g, device=dev, dtype=torch.float32).to(dtype)
        D = H * x.element_size()
        c = rua.C(data=x, token_sizes=lens)
        t_copy = timed(lambda: torch.empty_like(x).copy_(x))
        peak = 2 * N * D / t_copy
        t_segsum = timed(lambda: rua.segment_sum(x, lens))
        print(f'{cfg}: N={N} D={D} copy {t_copy * 1e3:.3f} ms = {peak / 1e12:.2f} TB/s, segment_sum '
              f'{t_segsum * 1e3:.3f} ms', flush=True)
        for kind in kinds:
            z, flat, side = layout_of(c, kind)
            rg = z._ragged()
            meta = 8 * len(lens_np) + (8 * (rg.Tp + rg.B) if kind == 'P' else 0)
            rows_moved = flat.shape[0]
            for opname, op in OPS.items():
                code = _native._SCAN_OPS[op]
                method = getattr(z, opname)
                t_api = timed(lambda: method())
                t_kernel = timed(lambda: _native._scan_raw(flat, rg, side, code, False))
                ext = op in ('max', 'min')
                fwd_bytes = 2 * rows_moved * D + (8 * rows_moved * H if ext else 0) + meta
                out, idx = _native._scan_raw(flat, rg, side, code, False)
                gout = torch.randn_like(out)
                if op == 'sum':
                    t_bwd = timed(lambda: _native._scan_raw(gout, rg, side, code, True))
                    bwd_bytes = 2 * rows_moved * D
                elif op == 'logsumexp':
                    t_bwd = timed(lambda: _native._scan_backward_raw(gout, flat, out, None, rg, side, code, False))
                    bwd_bytes = 4 * rows_moved * D
                else:
                    t_bwd = timed(lambda: _native._scan_backward_raw(gout, None, None, idx, rg, side, code, False))
                    bwd_bytes = 2 * rows_moved * D + 8 * rows_moved * H
                rec = dict(cfg=cfg, layout=kind, op=opname, N=N, H=H, dtype=str(dtype).replace('torch.', ''),
                           api_ms=t_api * 1e3, kernel_ms=t_kernel * 1e3, fwd_bytes=fwd_bytes,
                           fwd_frac_copy=fwd_bytes / t_kernel / peak, bwd_ms=t_bwd * 1e3, bwd_bytes=bwd_bytes,
                           bwd_frac_copy=bwd_bytes / t_bwd / peak, copy_ms=t_copy * 1e3, copy_TBps=peak / 1e12,
                           segment_sum_ms=t_segsum * 1e3)
                del out, idx, gout
                if cfg == 'cfg2' and kind == 'C':
                    # (a) pad -> torch op along dim 1 -> unpad
                    def padded():
                        zl = c.left(FILL[op])
                        r = TORCH[op](zl.data, dim=1)
                        if ext:
                            return (rua.L(data=r.values, token_sizes=lens).cat().data,
                                    rua.L(data=r.indices, token_sizes=lens).cat().data)
                        return rua.L(data=r, token_sizes=lens).cat().data, None
                    rec['baseline_pad_ms'] = timed(padded) * 1e3
                    rec['faster_than_pad'] = rec['api_ms'] < rec['baseline_pad_ms']   # the hard floor at cfg2
                    got = getattr(c, opname)()
                    want = padded()
                    if ext:   # bit-exact contract
                        rec['baseline_pad_match'] = torch.equal(got[0].data, want[0]) and torch.equal(got[1].data, want[1])
                    else:     # both round to bf16; torch's padded scan runs in its own order
                        diff = (got.data.float() - want[0].float()).abs().nan_to_num(0.0)
                        rec['baseline_pad_max_abs_diff'] = float(diff.max())
                    if op == 'sum':
                        # (b) global prefix minus the prefix before each segment (storage dtype)
                        off = torch.cumsum(lens, 0) - lens
                        seg = torch.repeat_interleave(torch.arange(len(lens_np), device=dev), lens)

                        def globalsum():
                            y = torch.cumsum(x, 0)
                            base = torch.cat([torch.zeros_like(y[:1]), y])[off]
                            return y - base[seg]
                        rec['baseline_global_ms'] = timed(globalsum) * 1e3
                        ref = rua.segment_cumsum(x.double(), lens)
                        rec['baseline_global_max_abs_err'] = float((globalsum().double() - ref).abs().max())
                        rec['scan_max_abs_err'] = float((got.data.double() - ref).abs().max())
                        del ref
                    del got, want
                rows.append(rec)
                print(json.dumps(rec), flush=True)
        del x, c
        torch.cuda.empty_cache()
    info = dict(gpu=name, power_limit=power, results=rows)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out + '.json', 'w') as f:
        json.dump(info, f, indent=1)
    with open(args.out + '.md', 'w') as f:
        f.write(f'# Per-sequence prefix scans -- {name}, power limit {power}\n\n')
        f.write('Written by `python benchmarks/scan.py`.  fwd / bwd = kernel call (CUDA-event median of 20); "% copy" = '
                'algorithmic bytes over time, against a device-to-device copy of the same payload timed in the same '
                'run.  api = the public method (metadata cached).\n\n')
        f.write('| shape | layout | op | api ms | fwd ms | fwd % copy | bwd ms | bwd % copy | pad->torch->unpad ms |'
                ' segment_sum ms | copy TB/s |\n|---|---|---|---|---|---|---|---|---|---|---|\n')
        for r in rows:
            pad = f"{r['baseline_pad_ms']:.3f}" if 'baseline_pad_ms' in r else ''
            f.write(f"| {r['cfg']} | {r['layout']} | {r['op']} | {r['api_ms']:.3f} | {r['kernel_ms']:.3f} | "
                    f"{100 * r['fwd_frac_copy']:.1f} | {r['bwd_ms']:.3f} | {100 * r['bwd_frac_copy']:.1f} | {pad} | "
                    f"{r['segment_sum_ms']:.3f} | {r['copy_TBps']:.2f} |\n")
        for r in rows:
            if 'baseline_global_ms' in r:
                f.write(f"\nBaseline (b), cfg2 cumsum: global torch.cumsum minus the segment-start prefix "
                        f"{r['baseline_global_ms']:.3f} ms, max abs error {r['baseline_global_max_abs_err']:.3g} "
                        f"(segment_cumsum: {r['scan_max_abs_err']:.3g}) against an fp64 reference.\n")
            if 'baseline_pad_match' in r:
                f.write(f"\ncfg2 {r['op']}: values and indices {'bit-identical to' if r['baseline_pad_match'] else 'DIFFER from'} "
                        f"baseline (a).\n")
            if 'baseline_pad_max_abs_diff' in r:
                f.write(f"\ncfg2 {r['op']}: max abs difference to baseline (a) {r['baseline_pad_max_abs_diff']:.3g}.\n")
        floor = [r for r in rows if 'faster_than_pad' in r]
        ok = all(r['faster_than_pad'] for r in floor)
        f.write(f"\nHard floor (every op at cfg2 faster through the public API than pad -> torch op -> unpad): "
                f"{'HOLDS' if ok else 'MISSED by ' + ', '.join(r['op'] for r in floor if not r['faster_than_pad'])}.\n")
    print('wrote', args.out + '.md')
    if not ok:
        print('hard floor missed at cfg2:', [r['op'] for r in floor if not r['faster_than_pad']])
        sys.exit(1)


if __name__ == '__main__':
    main()
