"""Per-sequence selective state-space scan on the GPU: the forward, the backward (gradients of x, delta, A, B, C and
the initial state) and the forward with ``return_final_state``, at the cfg2 / cfg3 lengths, against two same-GPU
baselines:
  (a) the padded loop: pad (x.left(0)) -> a torch loop over T with a (B, H, N) fp32 state, masked by length -> unpad,
      autograd for the backward.  Its forward is timed on the whole cfg2 batch; its backward keeps two (B, H, N) states
      per step and is timed at the largest batch of cfg2 lengths (its first b sequences) where it fits, and this
      package's forward + backward is timed at that same batch for the comparison;
  (b) the materialised form: exp(delta (x) A) and (delta x) (x) B as (tokens, H N) tensors -> segment_linear_recurrence
      over H N columns -> sum_n C h, forward only, at the largest H (halving from the shape's H) where it fits.
Times are CUDA-event medians after warm-up.  The floor is the larger of the exponential floor (tokens H N MUFU ex2 at
16 per clock per SM on 148 SMs, at the card's maximum SM clock read in the same run) and the HBM floor (x and delta
read, y written, B and C read, at 7.7 TB/s); both are derived, not measured.  A leg that does not fit in memory is
recorded as NaN.

    python benchmarks/ssm.py [--out profiles/r7_ssm]     # writes <out>.json and <out>.md
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

SMS, MUFU_PER_CLK, HBM_BYTES_PER_S = 148, 16, 7.7e12
NAN = float('nan')


def timed(fn, warmup=2, reps=7):
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
    yield 'cfg2', cfg2, 1024, 16, torch.bfloat16
    yield 'cfg2', cfg2, 1024, 16, torch.float32
    yield 'cfg2', cfg2, 1024, 4, torch.bfloat16
    yield 'cfg3', np.minimum(np.random.default_rng(0).zipf(1.5, 16384), 4096), 4096, 16, torch.bfloat16


def inputs(lens_np, H, N, dtype, dev, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    rows = int(lens_np.sum())
    x = torch.randn((rows, H), generator=g, device=dev, dtype=dtype)
    dl = (0.01 + 0.5 * torch.rand((rows, H), generator=g, device=dev)).to(dtype)
    A = -torch.exp(torch.randn((H, N), generator=g, device=dev).clamp(-2, 2))
    Bm = torch.randn((rows, N), generator=g, device=dev, dtype=dtype)
    Cm = torch.randn((rows, N), generator=g, device=dev, dtype=dtype)
    h0 = torch.randn((len(lens_np), H, N), generator=g, device=dev)
    return x, dl, A, Bm, Cm, h0


def padded_loop(c, dl, A, Bm, Cm, h0):
    """pad -> masked loop over T with an fp32 (B, H, N) state -> unpad"""
    lens = c.token_sizes
    xs = [rua.C(data=t, token_sizes=lens).left(0).data.float() for t in (c.data, dl, Bm, Cm)]
    x, d, b, cm = xs
    Bn, T, H = x.shape
    mask = (torch.arange(T, device=x.device)[None] < lens[:, None])[..., None, None]
    h = h0
    ys = []
    for t in range(T):
        dt = d[:, t, :, None]
        hn = torch.exp(dt * A) * h + (dt * x[:, t, :, None]) * b[:, t, None, :]
        h = torch.where(mask[:, t], hn, h)
        ys.append((cm[:, t, None, :] * h).sum(-1))
    y = torch.stack(ys, 1).to(c.data.dtype)
    return type(c.left(0))(data=y, token_sizes=lens).cat().data


def materialised(x, lens, dl, A, Bm, Cm):
    """exp(delta (x) A), (delta x) (x) B -> linear recurrence over H N columns -> sum_n C h"""
    rows, H = x.shape
    N = A.shape[1]
    gate = torch.exp(dl.float()[:, :, None] * A).to(x.dtype).view(rows, H * N)
    inp = ((dl * x)[:, :, None] * Bm[:, None, :]).view(rows, H * N)
    h = rua.segment_linear_recurrence(inp, lens, gate)
    del gate, inp
    return (h.view(rows, H, N) * Cm[:, None, :]).sum(-1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r7_ssm'))
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'benchmarks/ssm.py measures on a CUDA device'
    dev = torch.device('cuda')
    name = torch.cuda.get_device_name(dev)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader,nounits', '-i',
                            '0'], capture_output=True, text=True, timeout=30).stdout.strip().split(',')
        power, clock_mhz = q[0].strip() + ' W', float(q[1])
    except (OSError, subprocess.SubprocessError, ValueError, IndexError):
        power, clock_mhz = 'unknown', NAN
    print(f'# {name}, power limit {power}, max SM clock {clock_mhz} MHz', flush=True)
    rows_out = []
    for cfg, lens_np, H, N, dtype in shapes():
        lens = torch.tensor(lens_np, dtype=torch.long, device=dev)
        T, Bn = int(lens_np.sum()), len(lens_np)
        x, dl, A, Bm, Cm, h0 = inputs(lens_np, H, N, dtype, dev)
        rec = dict(cfg=cfg, H=H, N=N, dtype=str(dtype).replace('torch.', ''), tokens=T, B=Bn)
        rec['fwd_ms'] = timed(lambda: rua.segment_selective_scan(x, lens, dl, A, Bm, Cm, h0)) * 1e3
        rec['fwd_final_ms'] = timed(lambda: rua.segment_selective_scan(x, lens, dl, A, Bm, Cm, h0,
                                                                       return_final_state=True)) * 1e3
        leaves = [t.detach().requires_grad_(True) for t in (x, dl, A, Bm, Cm, h0)]
        y = rua.segment_selective_scan(leaves[0], lens, *leaves[1:])
        gout = torch.randn_like(y)
        rec['bwd_ms'] = timed(lambda: torch.autograd.grad(y, leaves, gout, retain_graph=True)) * 1e3
        del y, leaves
        torch.cuda.empty_cache()
        exp_floor = T * H * N / (SMS * MUFU_PER_CLK * clock_mhz * 1e6)
        hbm_floor = (3 * T * H + 2 * T * N) * x.element_size() / HBM_BYTES_PER_S
        rec['exp_floor_ms'], rec['hbm_floor_ms'] = exp_floor * 1e3, hbm_floor * 1e3
        floor = max(exp_floor, hbm_floor) * 1e3
        rec['fwd_pct_floor'] = 100 * floor / rec['fwd_ms']
        rec['bwd_pct_floor'] = 100 * floor / rec['bwd_ms']
        # max error against fp64 on the same values, over the first 256 sequences
        k = 256
        n_k = int(lens_np[:k].sum())
        sub = [t[:n_k] for t in (x, dl, Bm, Cm)]
        got = rua.segment_selective_scan(sub[0], lens[:k], sub[1], A, sub[2], sub[3], h0[:k])
        ref = rua.segment_selective_scan(sub[0].double(), lens[:k], sub[1].double(), A.double(), sub[2].double(),
                                         sub[3].double(), h0[:k].double())
        rec['max_abs_err'] = float((got.double() - ref).abs().max())
        rec['max_abs_ref'] = float(ref.abs().max())
        del got, ref
        c = rua.C(data=x, token_sizes=lens)
        # (a) the padded loop, forward on the whole batch (cfg2 only: cfg3's loop runs 4096 steps of (16384, 4096, 16))
        rec['loop_fwd_ms'] = NAN
        if cfg == 'cfg2':
            try:
                with torch.no_grad():
                    rec['loop_fwd_ms'] = timed(lambda: padded_loop(c, dl, A, Bm, Cm, h0), warmup=1, reps=3) * 1e3
            except torch.OutOfMemoryError:
                pass
            torch.cuda.empty_cache()
        # ... and forward + backward at the largest batch where its backward fits, against ours at that batch
        rec['loop_bwd_batch'], rec['loop_fwd_bwd_ms'], rec['ours_fwd_bwd_ms_at_loop_batch'] = 0, NAN, NAN
        if cfg == 'cfg2':
            for b in (2048, 1024, 512, 256, 128):
                nb = int(lens_np[:b].sum())
                sub = [t[:nb] for t in (x, dl, Bm, Cm)]
                lb = lens[:b]
                try:
                    lv = [t.detach().requires_grad_(True) for t in (sub[0], sub[1], A, sub[2], sub[3], h0[:b])]

                    def loop_step():
                        yl = padded_loop(rua.C(data=lv[0], token_sizes=lb), *lv[1:])
                        torch.autograd.grad(yl, lv, torch.ones_like(yl))

                    rec['loop_fwd_bwd_ms'] = timed(loop_step, warmup=1, reps=3) * 1e3
                except torch.OutOfMemoryError:
                    lv = None
                    torch.cuda.empty_cache()
                    continue

                def ours_step():
                    yo = rua.segment_selective_scan(lv[0], lb, *lv[1:])
                    torch.autograd.grad(yo, lv, torch.ones_like(yo))

                rec['ours_fwd_bwd_ms_at_loop_batch'] = timed(ours_step) * 1e3
                rec['loop_bwd_batch'] = b
                rec['fwd_bwd_speedup'] = rec['loop_fwd_bwd_ms'] / rec['ours_fwd_bwd_ms_at_loop_batch']
                del lv
                torch.cuda.empty_cache()
                break
        # (b) the materialised form at the largest H where it fits
        rec['mat_H'], rec['mat_fwd_ms'], rec['ours_fwd_ms_at_mat_H'] = 0, NAN, NAN
        h_try = H
        while h_try >= 64:
            try:
                xs, ds, As = x[:, :h_try].contiguous(), dl[:, :h_try].contiguous(), A[:h_try].contiguous()
                rec['mat_fwd_ms'] = timed(lambda: materialised(xs, lens, ds, As, Bm, Cm), warmup=1, reps=3) * 1e3
                rec['ours_fwd_ms_at_mat_H'] = timed(lambda: rua.segment_selective_scan(xs, lens, ds, As, Bm, Cm)) * 1e3
                rec['mat_H'] = h_try
                del xs, ds, As
                torch.cuda.empty_cache()
                break
            except torch.OutOfMemoryError:
                torch.cuda.empty_cache()
                h_try //= 2
        del x, dl, A, Bm, Cm, h0, c
        torch.cuda.empty_cache()
        rows_out.append(rec)
        print(json.dumps(rec), flush=True)
    info = dict(gpu=name, power_limit=power, max_sm_clock_mhz=clock_mhz, results=rows_out)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out + '.json', 'w') as f:
        json.dump(info, f, indent=1)
    with open(args.out + '.md', 'w') as f:
        f.write(f'# Per-sequence selective scan -- {name}, power limit {power}, max SM clock {clock_mhz:.0f} MHz\n\n')
        f.write('Written by `python benchmarks/ssm.py`.  fwd = `segment_selective_scan` with an initial state; fwd+final '
                '= the same with `return_final_state=True`; bwd = autograd backward of it (gradients of x, delta, A, B, C '
                'and the initial state).  CUDA-event medians.  "% floor" = the larger of the exponential floor (tokens H '
                'N MUFU ex2 at 16 / clock / SM) and the HBM floor (x, delta, y, B, C once at 7.7 TB/s) over the time; '
                'both floors are derived, not measured.  loop = pad -> masked torch loop over T with an fp32 state -> '
                'unpad (forward on the whole batch; forward + backward at the largest batch of the same lengths where '
                'its backward fits, against ours at that batch).  materialised = exp(delta A) and delta x B as (tokens, '
                'H N) tensors -> `segment_linear_recurrence` -> sum_n C h, forward, at the largest H where it fits.  '
                'NaN: not run (does not fit, or not attempted at cfg3).\n\n')
        f.write('| shape | H | N | dtype | fwd ms | fwd+final ms | bwd ms | exp floor ms | HBM floor ms | fwd % floor | '
                'bwd % floor | loop fwd ms | loop batch | loop fwd+bwd ms | ours fwd+bwd ms | fwd+bwd x | mat H | '
                'mat fwd ms | ours fwd ms at mat H | max abs err (max abs y) |\n'
                '|' + '---|' * 20 + '\n')
        for r in rows_out:
            f.write(f"| {r['cfg']} | {r['H']} | {r['N']} | {r['dtype']} | {r['fwd_ms']:.3f} | {r['fwd_final_ms']:.3f} | "
                    f"{r['bwd_ms']:.3f} | {r['exp_floor_ms']:.3f} | {r['hbm_floor_ms']:.3f} | "
                    f"{r['fwd_pct_floor']:.1f} | {r['bwd_pct_floor']:.1f} | {r['loop_fwd_ms']:.1f} | "
                    f"{r['loop_bwd_batch']} | {r['loop_fwd_bwd_ms']:.1f} | {r['ours_fwd_bwd_ms_at_loop_batch']:.3f} | "
                    f"{r.get('fwd_bwd_speedup', NAN):.1f} | {r['mat_H']} | {r['mat_fwd_ms']:.2f} | "
                    f"{r['ours_fwd_ms_at_mat_H']:.3f} | {r['max_abs_err']:.3g} ({r['max_abs_ref']:.3g}) |\n")
        for r in rows_out:
            if 'fwd_bwd_speedup' in r:
                ok = r['fwd_bwd_speedup'] >= 10
                f.write(f"\nTarget ({r['cfg']} H = {r['H']} N = {r['N']} {r['dtype']}, forward + backward at least 10x the "
                        f"padded loop at batch {r['loop_bwd_batch']}): {'MET' if ok else 'MISSED'} "
                        f"({r['fwd_bwd_speedup']:.1f}x).\n")
    print('wrote', args.out + '.md')


if __name__ == '__main__':
    main()
