"""Per-sequence Mamba-2 (SSD) scan on the GPU: the forward, the forward with ``return_final_state`` and the backward
(gradients of x, delta, A, B, C and the initial state), at the cfg2 / cfg3 lengths, against a same-GPU baseline:
pad (x.left(0)) -> the pure-torch chunked "minimal SSD" einsum form (chunks of Q = 64, fp32 state, (B, H, chunks, Q, Q)
decay tensors) -> unpad.  Its forward is timed on the whole batch; its forward + backward (autograd) at the largest batch
of the same lengths (its first b sequences) where the graph fits, and this package's forward + backward at that same
batch for the comparison.  A leg that does not fit in memory is NaN.

Times are CUDA-event medians after warm-up.  Two floors, both derived from shapes, not measured:
  HBM: x, delta, B and C read once and y written once, at 7.7 TB/s;
  tensor: the product FLOPs of the chunked form as the kernels run it (per head: C B^T, M u, C h^T, u^T B; the backward
  adds its recompute and adjoint products), at the data-sheet 2,250 TFLOP/s dense BF16 rate, which mma.sync is not
  expected to reach.
The bound named per row is the larger floor when the forward reaches at least 25 % of it, else 'neither (latency)'.

    python benchmarks/ssd.py [--out profiles/r8_ssd]     # writes <out>.json and <out>.md
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

HBM_BYTES_PER_S, BF16_FLOPS = 7.7e12, 2.25e15
Q = 64
BOUND_PCT = 25   # % of a floor from which it is named as the bound
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
    cfg3 = np.minimum(np.random.default_rng(0).zipf(1.5, 16384), 4096)
    yield 'cfg2', cfg2, 16, 64, 1, 128, torch.bfloat16
    yield 'cfg2', cfg2, 16, 64, 1, 128, torch.float32
    yield 'cfg2', cfg2, 16, 64, 8, 64, torch.bfloat16
    yield 'cfg3', cfg3, 64, 64, 8, 128, torch.bfloat16


def inputs(lens_np, H, P, G, N, dtype, dev, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    rows = int(lens_np.sum())
    x = torch.randn((rows, H, P), generator=g, device=dev, dtype=dtype)
    dl = (0.01 + 0.2 * torch.rand((rows, H), generator=g, device=dev)).to(dtype)
    A = -torch.exp(torch.randn((H,), generator=g, device=dev).clamp(-2, 1))
    Bm = (torch.randn((rows, G, N), generator=g, device=dev) / N ** 0.25).to(dtype)
    Cm = (torch.randn((rows, G, N), generator=g, device=dev) / N ** 0.25).to(dtype)
    h0 = torch.randn((len(lens_np), H, P, N), generator=g, device=dev)
    return x, dl, A, Bm, Cm, h0


def segsum(a):
    """(..., T) -> (..., T, T): sum_{s < r <= t} a_r below the diagonal, -inf above"""
    T = a.shape[-1]
    x = a[..., None].expand(*a.shape, T)
    x = x.masked_fill(~torch.tril(torch.ones(T, T, dtype=torch.bool, device=a.device), -1), 0)
    s = torch.cumsum(x, dim=-2)
    return s.masked_fill(~torch.tril(torch.ones(T, T, dtype=torch.bool, device=a.device)), -torch.inf)


def minimal_ssd(X, A, Bh, Ch, h0):
    """the chunked einsum form: X (b, l, h, p) = delta x, A (b, l, h) = delta A, Bh / Ch (b, l, h, n), h0 (b, h, p, n);
    l a multiple of Q; fp32 throughout -> y (b, l, h, p)"""
    b, l, h, p = X.shape
    c = l // Q
    X, A, Bh, Ch = (t.reshape(b, c, Q, *t.shape[2:]) for t in (X, A, Bh, Ch))
    A = A.permute(0, 3, 1, 2)                                     # b h c l
    Acum = torch.cumsum(A, dim=-1)
    L = torch.exp(segsum(A))                                      # b h c l s
    y_diag = torch.einsum('bclhn,bcshn,bhcls,bcshp->bclhp', Ch, Bh, L, X)
    decay = torch.exp(Acum[..., -1:] - Acum)
    states = torch.einsum('bclhn,bhcl,bclhp->bchpn', Bh, decay, X)
    states = torch.cat([h0[:, None], states], dim=1)
    decay_chunk = torch.exp(segsum(torch.nn.functional.pad(Acum[..., -1], (1, 0))))
    states = torch.einsum('bhzc,bchpn->bzhpn', decay_chunk, states)[:, :-1]
    y_off = torch.einsum('bclhn,bchpn,bhcl->bclhp', Ch, states, torch.exp(Acum))
    return (y_diag + y_off).reshape(b, l, h, p)


def padded_chunked(x, lens, dl, A, Bm, Cm, h0):
    """pad -> minimal_ssd in fp32 -> unpad"""
    H = x.shape[1]
    G = Bm.shape[1]
    pads = [rua.C(data=t, token_sizes=lens).left(0) for t in (x, dl, Bm, Cm)]
    xp, dp, bp, cp = (z.data.float() for z in pads)
    T = xp.shape[1]
    Tq = (T + Q - 1) // Q * Q
    if Tq != T:
        xp, dp, bp, cp = (torch.nn.functional.pad(t, (0, 0) * (t.dim() - 2) + (0, Tq - T)) for t in (xp, dp, bp, cp))
    bh, ch = (t.repeat_interleave(H // G, dim=2) for t in (bp, cp))
    y = minimal_ssd(xp * dp[..., None], dp * A, bh, ch, h0)[:, :T].to(x.dtype)
    return type(pads[0])(data=y, token_sizes=lens).cat().data


def flops(tokens, H, P, N):
    """product FLOPs of the chunked form as the kernels run it, forward and backward"""
    fwd = tokens * H * (2 * Q * (N + P) + 4 * P * N)
    bwd = tokens * H * (12 * P * N + 6 * Q * N + 4 * Q * P)
    return fwd, bwd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r8_ssd'))
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'benchmarks/ssd.py measures on a CUDA device'
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
    for cfg, lens_np, H, P, G, N, dtype in shapes():
        lens = torch.tensor(lens_np, dtype=torch.long, device=dev)
        T, Bn = int(lens_np.sum()), len(lens_np)
        x, dl, A, Bm, Cm, h0 = inputs(lens_np, H, P, G, N, dtype, dev)
        rec = dict(cfg=cfg, H=H, P=P, G=G, N=N, dtype=str(dtype).replace('torch.', ''), tokens=T, B=Bn)
        rec['fwd_ms'] = timed(lambda: rua.segment_ssd(x, lens, dl, A, Bm, Cm, h0)) * 1e3
        rec['fwd_final_ms'] = timed(lambda: rua.segment_ssd(x, lens, dl, A, Bm, Cm, h0, return_final_state=True)) * 1e3
        leaves = [t.detach().requires_grad_(True) for t in (x, dl, A, Bm, Cm, h0)]
        y = rua.segment_ssd(leaves[0], lens, *leaves[1:])
        gout = torch.randn_like(y)
        rec['bwd_ms'] = timed(lambda: torch.autograd.grad(y, leaves, gout, retain_graph=True)) * 1e3
        del y, leaves
        torch.cuda.empty_cache()
        f_fwd, f_bwd = flops(T, H, P, N)
        hbm = (2 * T * H * P + T * H + 2 * T * G * N) * x.element_size() / HBM_BYTES_PER_S * 1e3
        rec['hbm_floor_ms'] = hbm
        rec['tensor_floor_fwd_ms'], rec['tensor_floor_bwd_ms'] = f_fwd / BF16_FLOPS * 1e3, f_bwd / BF16_FLOPS * 1e3
        rec['fwd_tflops'] = f_fwd / rec['fwd_ms'] * 1e-9
        rec['bwd_tflops'] = f_bwd / rec['bwd_ms'] * 1e-9
        rec['fwd_pct_hbm'], rec['fwd_pct_tensor'] = 100 * hbm / rec['fwd_ms'], 100 * rec['tensor_floor_fwd_ms'] / rec['fwd_ms']
        rec['bwd_pct_tensor'] = 100 * rec['tensor_floor_bwd_ms'] / rec['bwd_ms']
        # a floor binds when the kernel reaches a fair share of it; far below both, the time is latency
        larger = 'tensor' if rec['tensor_floor_fwd_ms'] > hbm else 'HBM'
        rec['fwd_bound'] = larger if max(rec['fwd_pct_hbm'], rec['fwd_pct_tensor']) >= BOUND_PCT else 'neither (latency)'
        # max error against fp64 on the same values, over the first 256 sequences
        k = 256
        n_k = int(lens_np[:k].sum())
        sub = [t[:n_k] for t in (x, dl, Bm, Cm)]
        got = rua.segment_ssd(sub[0], lens[:k], sub[1], A, sub[2], sub[3], h0[:k])
        ref = rua.segment_ssd(sub[0].double(), lens[:k], sub[1].double(), A.double(), sub[2].double(),
                              sub[3].double(), h0[:k].double())
        rec['max_abs_err'] = float((got.double() - ref).abs().max())
        rec['max_abs_ref'] = float(ref.abs().max())
        rec['baseline_max_abs_err'] = NAN
        try:
            with torch.no_grad():
                base = padded_chunked(sub[0], lens[:k], sub[1], A, sub[2], sub[3], h0[:k])
            rec['baseline_max_abs_err'] = float((base.double() - ref).abs().max())
            del base
        except torch.OutOfMemoryError:
            pass
        del got, ref
        torch.cuda.empty_cache()
        # the padded chunked form: forward on the whole batch
        rec['base_fwd_ms'] = NAN
        try:
            with torch.no_grad():
                rec['base_fwd_ms'] = timed(lambda: padded_chunked(x, lens, dl, A, Bm, Cm, h0), warmup=1, reps=3) * 1e3
        except torch.OutOfMemoryError:
            pass
        torch.cuda.empty_cache()
        # ... and forward + backward at the largest batch where its graph fits, against ours at that batch
        rec['base_bwd_batch'], rec['base_fwd_bwd_ms'], rec['ours_fwd_bwd_ms_at_base_batch'] = 0, NAN, NAN
        for b in (Bn, Bn // 2, Bn // 4, Bn // 8, Bn // 16, Bn // 32):
            nb = int(lens_np[:b].sum())
            sub = [t[:nb] for t in (x, dl, Bm, Cm)]
            lb = lens[:b]
            lv = [t.detach().requires_grad_(True) for t in (sub[0], sub[1], A, sub[2], sub[3], h0[:b])]
            try:
                def base_step():
                    yb = padded_chunked(lv[0], lb, *lv[1:])
                    torch.autograd.grad(yb, lv, torch.ones_like(yb))

                rec['base_fwd_bwd_ms'] = timed(base_step, warmup=1, reps=3) * 1e3
            except torch.OutOfMemoryError:
                torch.cuda.empty_cache()
                continue

            def ours_step():
                yo = rua.segment_ssd(lv[0], lb, *lv[1:])
                torch.autograd.grad(yo, lv, torch.ones_like(yo))

            rec['ours_fwd_bwd_ms_at_base_batch'] = timed(ours_step) * 1e3
            rec['base_bwd_batch'] = b
            rec['fwd_bwd_speedup'] = rec['base_fwd_bwd_ms'] / rec['ours_fwd_bwd_ms_at_base_batch']
            break
        lv = None
        del x, dl, A, Bm, Cm, h0
        torch.cuda.empty_cache()
        rows_out.append(rec)
        print(json.dumps(rec), flush=True)
    info = dict(gpu=name, power_limit=power, max_sm_clock_mhz=clock_mhz, results=rows_out)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out + '.json', 'w') as f:
        json.dump(info, f, indent=1)
    with open(args.out + '.md', 'w') as f:
        f.write(f'# Per-sequence Mamba-2 (SSD) scan -- {name}, power limit {power}, max SM clock {clock_mhz:.0f} MHz\n\n')
        f.write('Written by `python benchmarks/ssd.py`.  fwd = `segment_ssd` with an initial state; fwd+final = the same '
                'with `return_final_state=True`; bwd = autograd backward of it (gradients of x, delta, A, B, C and the '
                'initial state).  CUDA-event medians.  Floors are derived, not measured: HBM = x, delta, B, C read and y '
                'written once at 7.7 TB/s; tensor = the chunked form\'s product FLOPs (as the kernels run them) at the '
                'data-sheet 2,250 TFLOP/s dense BF16 rate, which mma.sync is not expected to reach.  base = pad -> the '
                'pure-torch chunked einsum form (Q = 64, fp32 state) -> unpad: forward on the whole batch; forward + '
                'backward at the largest batch of the same lengths where its autograd graph fits, against ours at that '
                'batch.  NaN: does not fit.  bound = the larger floor when the forward reaches at least 25 % of it, else '
                '"neither (latency)".  Errors: max |y - fp64| over the first 256 sequences.\n\n')
        f.write('| shape | H | P | G | N | dtype | fwd ms | fwd+final ms | bwd ms | HBM floor ms | tensor floor fwd / bwd ms '
                '| fwd TFLOP/s | bwd TFLOP/s | fwd % HBM | fwd % tensor | bwd % tensor | bound | base fwd ms | base batch '
                '| base fwd+bwd ms | ours fwd+bwd ms | fwd+bwd x | max abs err ours / base (max abs y) |\n'
                '|' + '---|' * 23 + '\n')
        for r in rows_out:
            f.write(f"| {r['cfg']} | {r['H']} | {r['P']} | {r['G']} | {r['N']} | {r['dtype']} | {r['fwd_ms']:.3f} | "
                    f"{r['fwd_final_ms']:.3f} | {r['bwd_ms']:.3f} | {r['hbm_floor_ms']:.3f} | "
                    f"{r['tensor_floor_fwd_ms']:.3f} / {r['tensor_floor_bwd_ms']:.3f} | {r['fwd_tflops']:.1f} | "
                    f"{r['bwd_tflops']:.1f} | {r['fwd_pct_hbm']:.1f} | {r['fwd_pct_tensor']:.1f} | "
                    f"{r['bwd_pct_tensor']:.1f} | {r['fwd_bound']} | {r['base_fwd_ms']:.1f} | {r['base_bwd_batch']} | "
                    f"{r['base_fwd_bwd_ms']:.1f} | {r['ours_fwd_bwd_ms_at_base_batch']:.3f} | "
                    f"{r.get('fwd_bwd_speedup', NAN):.1f} | {r['max_abs_err']:.3g} / {r['baseline_max_abs_err']:.3g} "
                    f"({r['max_abs_ref']:.3g}) |\n")
        for r in rows_out:
            if r['cfg'] == 'cfg2' and r['dtype'] == 'bfloat16' and r['G'] == 1:
                sp = r.get('fwd_bwd_speedup', NAN)
                f.write(f"\nTarget (cfg2 H = {r['H']} P = {r['P']} N = {r['N']} bf16, forward + backward at least 5x the "
                        f"padded chunked form at batch {r['base_bwd_batch']}): {'MET' if sp >= 5 else 'NOT MET'} "
                        f"({sp:.1f}x).\n")
    print('wrote', args.out + '.md')


if __name__ == '__main__':
    main()
