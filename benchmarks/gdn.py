"""Per-sequence gated delta rule (Gated DeltaNet) on the GPU: the forward, the forward with ``return_final_state`` and
the backward (gradients of v, q, k, g, beta and the initial state), at the cfg2 / cfg3 lengths, against a same-GPU
baseline: pad (x.left(0)) -> a self-contained pure-torch chunked form (chunks of Q = 64, fp32, (B, H, chunks, Q, Q)
decay and score tensors, the UT transform by a triangular solve, a Python loop over the chunks for the state) -> unpad.
Its forward is timed on the whole batch; its forward + backward (autograd) at the largest batch of the same lengths (its
first b sequences) where the graph fits, and this package's forward + backward at that same batch for the comparison.
A leg that does not fit in memory is NaN.  When flash-linear-attention imports, its chunk_gated_delta_rule on the C
storage (cu_seqlens) is timed on the first 256 sequences (the subset of the error column), with ours at the same subset
and the largest difference between its output and ours.  It runs only on that subset and only when
tokens * H * max(K, V, 64) < 2^31: flash-linear-attention 0.5.1's varlen kernels load the sequence start as int32 and
form offsets such as (bos * H + h) * V in int32 (fla/ops/common/chunk_o.py, fla/ops/gated_delta_rule/chunk_fwd.py),
which overflow at the full cfg2 batch (1.06 M tokens * 32 heads * 128 = 4.3e9) and address memory outside the tensors.

Times are CUDA-event medians after warm-up.  Two floors, both derived from shapes, not measured:
  HBM: v, q, k, g and beta read once and o written once, at 7.7 TB/s;
  tensor: the product FLOPs of the chunked form as the kernels run it (per value head and V block: K K^T, Q K^T, K S,
  T Z, Q S, P V', K^T V'; the backward adds its recompute and adjoint products), at the data-sheet 2,250 TFLOP/s dense
  BF16 rate, which mma.sync is not expected to reach.
The bound named per row is the larger floor when the forward reaches at least 25 % of it, else 'neither (latency)'.

    python benchmarks/gdn.py [--out profiles/r9_gdn]     # writes <out>.json and <out>.md
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
    yield 'cfg2', cfg2, 32, 16, 128, 128, torch.bfloat16
    yield 'cfg2', cfg2, 32, 16, 128, 128, torch.float32
    yield 'cfg2', cfg2, 16, 16, 128, 128, torch.bfloat16
    yield 'cfg3', cfg3, 32, 16, 128, 128, torch.bfloat16


def inputs(lens_np, H, G, K, V, dtype, dev, seed=0):
    gen = torch.Generator(device=dev).manual_seed(seed)
    rows = int(lens_np.sum())
    v = torch.randn((rows, H, V), generator=gen, device=dev, dtype=dtype)
    q = torch.nn.functional.normalize(torch.randn((rows, G, K), generator=gen, device=dev), dim=-1).to(dtype)
    k = torch.nn.functional.normalize(torch.randn((rows, G, K), generator=gen, device=dev), dim=-1).to(dtype)
    g = torch.nn.functional.logsigmoid(torch.randn((rows, H), generator=gen, device=dev) + 3)
    beta = torch.rand((rows, H), generator=gen, device=dev).to(dtype)
    h0 = torch.randn((len(lens_np), H, K, V), generator=gen, device=dev) / K ** 0.5
    return v, q, k, g, beta, h0


def chunked_gdn(q, k, v, g, beta, scale, h0):
    """the chunked form in fp32: q, k (b, l, h, K), v (b, l, h, V), g, beta (b, l, h), h0 (b, h, K, V); l a multiple
    of Q -> o (b, l, h, V)"""
    b, l, h, K = k.shape
    c = l // Q
    q, k, v = (t.reshape(b, c, Q, h, t.shape[-1]).permute(0, 3, 1, 2, 4) for t in (q, k, v))   # b h c Q *
    g, beta = (t.reshape(b, c, Q, h).permute(0, 3, 1, 2) for t in (g, beta))                   # b h c Q
    cum = torch.cumsum(g, -1)
    incl = torch.tril(torch.ones(Q, Q, dtype=torch.bool, device=q.device))
    gam = torch.exp(torch.where(incl, cum[..., :, None] - cum[..., None, :], -torch.inf))       # b h c Q Q
    A = torch.tril(beta[..., None] * (k @ k.transpose(-1, -2)) * gam, -1)
    eye = torch.eye(Q, dtype=A.dtype, device=A.device)
    T = torch.linalg.solve_triangular(eye + A, eye.expand_as(A), upper=False)
    W = T @ ((beta * torch.exp(cum))[..., None] * k)
    U = T @ (beta[..., None] * v)
    P = (q @ k.transpose(-1, -2)) * gam
    S = h0
    outs = []
    for i in range(c):
        Vp = U[:, :, i] - W[:, :, i] @ S
        outs.append(scale * ((torch.exp(cum[:, :, i])[..., None] * q[:, :, i]) @ S + P[:, :, i] @ Vp))
        cl = cum[:, :, i, -1:]
        S = torch.exp(cl)[..., None] * S + (k[:, :, i] * torch.exp(cl - cum[:, :, i])[..., None]).transpose(-1, -2) @ Vp
    return torch.stack(outs, 2).permute(0, 2, 3, 1, 4).reshape(b, l, h, -1)


def padded_chunked(v, lens, q, k, g, beta, h0):
    """pad -> chunked_gdn in fp32 -> unpad"""
    H, G = v.shape[1], q.shape[1]
    pads = [rua.C(data=t, token_sizes=lens).left(0) for t in (v, q, k, g, beta)]
    vp, qp, kp, gp, bp = (z.data.float() for z in pads)
    T = vp.shape[1]
    Tq = (T + Q - 1) // Q * Q
    if Tq != T:
        vp, qp, kp, gp, bp = (torch.nn.functional.pad(t, (0, 0) * (t.dim() - 2) + (0, Tq - T))
                              for t in (vp, qp, kp, gp, bp))
    qh, kh = (t.repeat_interleave(H // G, dim=2) for t in (qp, kp))
    o = chunked_gdn(qh, kh, vp, gp, bp, q.shape[-1] ** -0.5, h0)[:, :T].to(v.dtype)
    return type(pads[0])(data=o, token_sizes=lens).cat().data


def fla_offsets_fit(tokens, H, K, V):
    """whether flash-linear-attention's int32 varlen offsets, (bos * H + h) * max(K, V, chunk 64), stay below 2^31"""
    return tokens * H * max(K, V, 64) < 2 ** 31


def fla_leg(v, lens, q, k, g, beta, h0, ours):
    """(ms, max |fla - ours|) of flash-linear-attention's chunk_gated_delta_rule on the C storage, or None when it does
    not import"""
    try:
        from fla.ops.gated_delta_rule import chunk_gated_delta_rule
    except Exception:   # not installed, or not importable on this machine
        return None
    H, G = v.shape[1], q.shape[1]
    assert fla_offsets_fit(v.shape[0], H, q.shape[2], v.shape[2]), 'outside the range of fla\'s int32 offsets'

    cu = torch.nn.functional.pad(torch.cumsum(lens, 0), (1, 0))
    qh, kh = (t.repeat_interleave(H // G, dim=1)[None] for t in (q, k))

    def run():
        return chunk_gated_delta_rule(qh, kh, v[None], g[None], beta[None], initial_state=h0,
                                      output_final_state=False, cu_seqlens=cu)[0]

    try:
        ms = timed(run) * 1e3
        diff = float((run()[0].double() - ours.double()).abs().max())
    except Exception as e:   # an fla version whose signature differs
        print('fla leg failed:', repr(e), flush=True)
        return None
    return ms, diff


def flops(tokens, H, K, V):
    """product FLOPs of the chunked form as the kernels run it (per value head and V block of 64), forward and backward"""
    nvb = (V + 63) // 64
    VB = min(V, 64)
    fwd = tokens * H * nvb * (4 * Q * K + 6 * K * VB + 4 * Q * VB)
    bwd = tokens * H * nvb * (18 * Q * K + 22 * K * VB + 12 * Q * VB + 4 * Q * Q)
    return fwd, bwd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r9_gdn'))
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'benchmarks/gdn.py measures on a CUDA device'
    dev = torch.device('cuda')
    name = torch.cuda.get_device_name(dev)
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader,nounits',
                              '-i', '0'], capture_output=True, text=True, timeout=30).stdout.strip().split(',')
        power, clock_mhz = out[0].strip() + ' W', float(out[1])
    except (OSError, subprocess.SubprocessError, ValueError, IndexError):
        power, clock_mhz = 'unknown', NAN
    print(f'# {name}, power limit {power}, max SM clock {clock_mhz} MHz', flush=True)
    rows_out = []
    for cfg, lens_np, H, G, K, V, dtype in shapes():
        lens = torch.tensor(lens_np, dtype=torch.long, device=dev)
        T, Bn = int(lens_np.sum()), len(lens_np)
        v, q, k, g, beta, h0 = inputs(lens_np, H, G, K, V, dtype, dev)
        rec = dict(cfg=cfg, H=H, G=G, K=K, V=V, dtype=str(dtype).replace('torch.', ''), tokens=T, B=Bn)
        rec['fwd_ms'] = timed(lambda: rua.segment_gated_delta_rule(v, lens, q, k, g, beta, initial=h0)) * 1e3
        rec['fwd_final_ms'] = timed(lambda: rua.segment_gated_delta_rule(v, lens, q, k, g, beta, initial=h0,
                                                                         return_final_state=True)) * 1e3
        leaves = [t.detach().requires_grad_(True) for t in (v, q, k, g, beta, h0)]
        o = rua.segment_gated_delta_rule(leaves[0], lens, *leaves[1:5], initial=leaves[5])
        gout = torch.randn_like(o)
        rec['bwd_ms'] = timed(lambda: torch.autograd.grad(o, leaves, gout, retain_graph=True)) * 1e3
        del o, leaves
        torch.cuda.empty_cache()
        f_fwd, f_bwd = flops(T, H, K, V)
        hbm = (2 * T * H * V + 2 * T * G * K + T * H) * v.element_size() / HBM_BYTES_PER_S * 1e3 + \
            T * H * 4 / HBM_BYTES_PER_S * 1e3
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
        n = 256
        n_k = int(lens_np[:n].sum())
        sub = [t[:n_k] for t in (v, q, k, g, beta)]
        got = rua.segment_gated_delta_rule(sub[0], lens[:n], *sub[1:], initial=h0[:n])
        ref = rua.segment_gated_delta_rule(*(t.double() for t in sub[:1]), lens[:n], *(t.double() for t in sub[1:]),
                                           initial=h0[:n].double())
        rec['max_abs_err'] = float((got.double() - ref).abs().max())
        rec['max_abs_ref'] = float(ref.abs().max())
        rec['baseline_max_abs_err'] = NAN
        try:
            with torch.no_grad():
                base = padded_chunked(sub[0], lens[:n], *sub[1:], h0[:n])
            rec['baseline_max_abs_err'] = float((base.double() - ref).abs().max())
            del base
        except torch.OutOfMemoryError:
            pass
        # flash-linear-attention on the C storage of the same subset, when it imports and its offsets fit
        rec['ours_sub_ms'] = timed(lambda: rua.segment_gated_delta_rule(sub[0], lens[:n], *sub[1:], initial=h0[:n])) * 1e3
        leg = None
        if fla_offsets_fit(n_k, H, K, V):
            with torch.no_grad():
                leg = fla_leg(sub[0], lens[:n], *sub[1:], h0[:n].contiguous(), got)
            rec['fla'] = 'not available' if leg is None else 'available'
        else:
            rec['fla'] = 'not run (int32 offsets)'
        rec['fla_ms'], rec['fla_max_abs_diff'] = (NAN, NAN) if leg is None else leg
        del got, ref
        torch.cuda.empty_cache()
        # the padded chunked form: forward on the whole batch
        rec['base_fwd_ms'] = NAN
        try:
            with torch.no_grad():
                rec['base_fwd_ms'] = timed(lambda: padded_chunked(v, lens, q, k, g, beta, h0), warmup=1, reps=3) * 1e3
        except torch.OutOfMemoryError:
            pass
        torch.cuda.empty_cache()
        # ... and forward + backward at the largest batch where its graph fits, against ours at that batch
        rec['base_bwd_batch'], rec['base_fwd_bwd_ms'], rec['ours_fwd_bwd_ms_at_base_batch'] = 0, NAN, NAN
        for b in (Bn, Bn // 2, Bn // 4, Bn // 8, Bn // 16, Bn // 32):
            nb = int(lens_np[:b].sum())
            sub = [t[:nb] for t in (v, q, k, g, beta)]
            lb = lens[:b]
            lv = [t.detach().requires_grad_(True) for t in sub + [h0[:b]]]
            try:
                def base_step():
                    ob = padded_chunked(lv[0], lb, *lv[1:])
                    torch.autograd.grad(ob, lv, torch.ones_like(ob))

                rec['base_fwd_bwd_ms'] = timed(base_step, warmup=1, reps=3) * 1e3
            except torch.OutOfMemoryError:
                torch.cuda.empty_cache()
                continue

            def ours_step():
                oo = rua.segment_gated_delta_rule(lv[0], lb, *lv[1:5], initial=lv[5])
                torch.autograd.grad(oo, lv, torch.ones_like(oo))

            rec['ours_fwd_bwd_ms_at_base_batch'] = timed(ours_step) * 1e3
            rec['base_bwd_batch'] = b
            rec['fwd_bwd_speedup'] = rec['base_fwd_bwd_ms'] / rec['ours_fwd_bwd_ms_at_base_batch']
            break
        lv = None
        del v, q, k, g, beta, h0
        torch.cuda.empty_cache()
        rows_out.append(rec)
        print(json.dumps(rec), flush=True)
    info = dict(gpu=name, power_limit=power, max_sm_clock_mhz=clock_mhz, results=rows_out)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out + '.json', 'w') as f:
        json.dump(info, f, indent=1)
    with open(args.out + '.md', 'w') as f:
        f.write(f'# Per-sequence gated delta rule -- {name}, power limit {power}, max SM clock {clock_mhz:.0f} MHz\n\n')
        f.write('Written by `python benchmarks/gdn.py`.  fwd = `segment_gated_delta_rule` with an initial state; '
                'fwd+final = the same with `return_final_state=True`; bwd = autograd backward of it (gradients of v, q, '
                'k, g, beta and the initial state).  CUDA-event medians.  Floors are derived, not measured: HBM = v, q, '
                'k, g, beta read and o written once at 7.7 TB/s; tensor = the chunked form\'s product FLOPs (as the '
                'kernels run them) at the data-sheet 2,250 TFLOP/s dense BF16 rate, which mma.sync is not expected to '
                'reach.  base = pad -> a pure-torch chunked form (Q = 64, fp32) -> unpad: forward on the whole batch; '
                'forward + backward at the largest batch of the same lengths where its autograd graph fits, against '
                'ours at that batch.  NaN: does not fit.  bound = the larger floor when the forward reaches at least '
                '25 % of it, else "neither (latency)".  Errors: max |o - fp64| over the first 256 sequences.  fla = '
                'flash-linear-attention\'s chunk_gated_delta_rule forward on the C storage of those 256 sequences, '
                'beside ours on the same subset, and max |o_fla - o_ours| (a report, not a target).\n\n')
        f.write('| shape | H | G | K | V | dtype | fwd ms | fwd+final ms | bwd ms | HBM floor ms | tensor floor fwd / bwd ms '
                '| fwd TFLOP/s | bwd TFLOP/s | fwd % HBM | fwd % tensor | bwd % tensor | bound | base fwd ms | base batch '
                '| base fwd+bwd ms | ours fwd+bwd ms | fwd+bwd x | max abs err ours / base (max abs o) | 256 seqs: ours fwd '
                'ms | fla fwd ms (max abs diff) |\n|' + '---|' * 25 + '\n')
        for r in rows_out:
            fla = r['fla'] if r['fla'] != 'available' else f"{r['fla_ms']:.3f} ({r['fla_max_abs_diff']:.3g})"
            f.write(f"| {r['cfg']} | {r['H']} | {r['G']} | {r['K']} | {r['V']} | {r['dtype']} | {r['fwd_ms']:.3f} | "
                    f"{r['fwd_final_ms']:.3f} | {r['bwd_ms']:.3f} | {r['hbm_floor_ms']:.3f} | "
                    f"{r['tensor_floor_fwd_ms']:.3f} / {r['tensor_floor_bwd_ms']:.3f} | {r['fwd_tflops']:.1f} | "
                    f"{r['bwd_tflops']:.1f} | {r['fwd_pct_hbm']:.1f} | {r['fwd_pct_tensor']:.1f} | "
                    f"{r['bwd_pct_tensor']:.1f} | {r['fwd_bound']} | {r['base_fwd_ms']:.1f} | {r['base_bwd_batch']} | "
                    f"{r['base_fwd_bwd_ms']:.1f} | {r['ours_fwd_bwd_ms_at_base_batch']:.3f} | "
                    f"{r.get('fwd_bwd_speedup', NAN):.1f} | {r['max_abs_err']:.3g} / {r['baseline_max_abs_err']:.3g} "
                    f"({r['max_abs_ref']:.3g}) | {r['ours_sub_ms']:.3f} | {fla} |\n")
        for r in rows_out:
            if r['cfg'] == 'cfg2' and r['dtype'] == 'bfloat16' and r['H'] == 32:
                sp = r.get('fwd_bwd_speedup', NAN)
                f.write(f"\nTarget (cfg2 H = {r['H']} G = {r['G']} K = V = {r['K']} bf16, forward + backward at least 5x "
                        f"the padded chunked form at batch {r['base_bwd_batch']}): {'MET' if sp >= 5 else 'NOT MET'} "
                        f"({sp:.1f}x).\n")
    print('wrote', args.out + '.md')


if __name__ == '__main__':
    main()
