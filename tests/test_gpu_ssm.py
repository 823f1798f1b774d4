"""Selective state-space scan (torchrua_b200.ssm) against an fp64 oracle on the same GPU.

The oracle is the recurrence on the zero-padded (B, T, H, N) batch, a loop over T vectorised over B, H and N and
masked by length; its gradients come from autograd.  The oracle itself is checked against the unrolled closed form
h_t = (prod_{s<=t} dA_s) h0 + sum_{s<=t} (prod_{s<r<=t} dA_r) delta_s B_s x_s.

Tolerances (u = unit roundoff of the accumulator: 2^-24 for fp32 / fp16 / bf16, 2^-53 for fp64): every output and
gradient within 16 u n s, plus one storage ulp of |ref| (and 2^-24) for 16-bit outputs, where s is the same
computation on absolute values (|x|, |B|, |C|, |initial|, |A| in the derivatives, |grad_out|) and n the number of terms
that reach it: the sequence's length for y, final, grad_x, grad_delta and grad_initial, length + H for grad_B and
grad_C (a sum over channels), the longest length + the batch for grad_A (a sum over every token).
"""

import numpy as np
import pytest
import torch

import torchrua_b200 as rua

pytestmark = pytest.mark.gpu

DEV = 'cuda'
DTYPES = [torch.float32, torch.float64, torch.float16, torch.bfloat16]
ULP = {torch.float16: 2.0 ** -10, torch.bfloat16: 2.0 ** -7}
TC = 32   # checkpoint interval of the kernels


def _u(dtype):
    return 2.0 ** -53 if dtype == torch.float64 else 2.0 ** -24


def acc_of(dtype):
    return torch.float64 if dtype == torch.float64 else torch.float32


# ---------------------------------------------------------------------------------------------------------------------
# fp64 oracle
# ---------------------------------------------------------------------------------------------------------------------
def pad(x, lens):
    """(rows, ...) C rows -> zero-padded (B, T, ...) through plain torch indexing (differentiable)."""
    B = lens.numel()
    T = int(lens.max()) if B else 0
    off = torch.cumsum(lens, 0) - lens
    t = torch.arange(T, device=x.device)
    valid = t[None, :] < lens[:, None]
    idx = (off[:, None] + t[None, :]).clamp(min=0, max=max(x.shape[0] - 1, 0))
    shape = valid.shape + (1,) * (x.dim() - 1)
    return torch.where(valid.view(shape), x[idx], torch.zeros((), dtype=x.dtype, device=x.device)), valid


def oracle(x, lens, dl, A, Bm, Cm, h0=None, reverse=False, magnitude=False):
    """(y (sum(lens), H), final (B, H, N)) from C rows x, dl (rows, H), Bm, Cm (rows, N), A (H, N), h0 (B, H, N).
    magnitude: dA keeps its value but its derivatives use |A| (the scale s of the tolerances)."""
    H, N = A.shape
    xp, valid = pad(x, lens)
    dp, _ = pad(dl, lens)
    bp, _ = pad(Bm, lens)
    cp, _ = pad(Cm, lens)
    B, T = valid.shape
    h = torch.zeros((B, H, N), dtype=x.dtype, device=x.device) if h0 is None else h0
    ys = [None] * T
    for t in (range(T - 1, -1, -1) if reverse else range(T)):
        d = dp[:, t, :, None]
        if magnitude:
            dA = torch.exp(d * A).detach() * (1 + d * A.abs() - (d * A.abs()).detach())
        else:
            dA = torch.exp(d * A)
        hn = dA * h + (d * xp[:, t, :, None]) * bp[:, t, None, :]
        h = torch.where(valid[:, t, None, None], hn, h)
        ys[t] = (cp[:, t, None, :] * h).sum(-1)
    y = torch.stack(ys, 1)[valid] if T else x[:0]
    return y, h


def closed_form(x, lens, dl, A, Bm, Cm, h0):
    """y from h_t = (prod_{s<=t} dA_s) h0 + sum_{s<=t} (prod_{s<r<=t} dA_r) delta_s B_s x_s, sequence by sequence."""
    out, o = [], 0
    for i, n in enumerate(lens.tolist()):
        for t in range(n):
            h = h0[i].clone()
            for s in range(t + 1):
                h = h * torch.exp(dl[o + s, :, None] * A)
            for s in range(t + 1):
                p = torch.ones_like(A)
                for r in range(s + 1, t + 1):
                    p = p * torch.exp(dl[o + r, :, None] * A)
                h = h + p * (dl[o + s, :, None] * Bm[o + s][None, :] * x[o + s, :, None])
            out.append((Cm[o + t][None, :] * h).sum(-1))
        o += n
    return torch.stack(out)


def make(lens_list, feat, N, dtype, seed=0, init=False, extra_rows=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    lens = torch.tensor(lens_list, dtype=torch.long, device=DEV)
    rows = int(lens.sum()) + extra_rows

    def r(*s):
        return torch.randn(s, generator=g, device=DEV, dtype=torch.float64)

    x = r(rows, *feat).to(dtype)
    dl = (0.01 + 0.5 * torch.rand((rows, *feat), generator=g, device=DEV, dtype=torch.float64)).to(dtype)
    A = (-torch.exp(r(*feat, N).clamp(-2, 2))).to(acc_of(dtype))
    Bm, Cm = r(rows, N).to(dtype), r(rows, N).to(dtype)
    h0 = r(len(lens_list), *feat, N).to(acc_of(dtype)) if init else None
    return lens, x, dl, A, Bm, Cm, h0


def flat(x, dl, A, Bm, Cm, h0, B):
    """the oracle's 2-D forms, fp64"""
    H, N = int(np.prod(A.shape[:-1])), A.shape[-1]

    def d64(t):
        return t.detach().to(torch.float64, copy=True)
    return (d64(x).reshape(-1, H), d64(dl).reshape(-1, H), d64(A).reshape(H, N), d64(Bm), d64(Cm),
            None if h0 is None else d64(h0).reshape(B, H, N))


def as_layout(kind, lens, t, fill=0):
    """(t's rows in layout kind, function mapping that layout's data back to C rows)"""
    c = rua.C(data=t, token_sizes=lens)
    if kind == 'C':
        return c, lambda d: d
    if kind == 'P':
        z = c.pack()
        return z, lambda d: z._replace(data=d).cat().data
    z = c.left(fill) if kind == 'L' else c.right(fill)
    return z, lambda d: type(z)(data=d, token_sizes=z.token_sizes).cat().data


def within(got, ref, s, n, dtype, what):
    got, ref = got.double(), ref.double()
    tol = 16 * _u(dtype) * n * s
    if dtype in ULP:
        tol = tol + ULP[dtype] * ref.abs() + 2.0 ** -24
    err = (got - ref).abs()
    assert bool((err <= tol).all()), (what, float(err.max()), float((err - tol).max()))


# ---------------------------------------------------------------------------------------------------------------------
# the oracle itself
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('reverse', [False, True])
def test_oracle_matches_closed_form(reverse):
    lens_list = [1, 3, 0, 5]
    lens, x, dl, A, Bm, Cm, h0 = make(lens_list, (3,), 2, torch.float64, init=True)
    y, fin = oracle(x, lens, dl, A, Bm, Cm, h0, reverse)
    if reverse:   # the closed form on every sequence reversed in time
        idx = torch.cat([torch.arange(o + n - 1, o - 1, -1) for o, n in
                         zip((np.cumsum(lens_list) - lens_list).tolist(), lens_list)]).to(DEV)
        ref = closed_form(x[idx], lens, dl[idx], A, Bm[idx], Cm[idx], h0)
        ref = torch.empty_like(ref).index_copy_(0, idx, ref)
    else:
        ref = closed_form(x, lens, dl, A, Bm, Cm, h0)
    assert float((y - ref).abs().max()) <= 1e-12
    assert torch.equal(fin[2], h0[2])   # an empty sequence keeps its initial state


# ---------------------------------------------------------------------------------------------------------------------
# the grid: dtype x layout x N x feat x initial x reverse, forward values and all six gradients
# ---------------------------------------------------------------------------------------------------------------------
GRID_LENS = [0, 1, 3, 7, 2, 0, 13, 5, 1, 9, 33]


def run_case(kind, lens, x, dl, A, Bm, Cm, h0, reverse, dtype, seed=0):
    """forward + backward through layout `kind`; checks y, final and the six gradients against the oracle"""
    Bn = lens.numel()
    zx, back = as_layout(kind, lens, x)
    zd, _ = as_layout(kind, lens, dl)
    zb, _ = as_layout(kind, lens, Bm)
    zc, _ = as_layout(kind, lens, Cm)
    leaves = [zx.data.detach().requires_grad_(True), zd.data.detach().requires_grad_(True),
              A.detach().requires_grad_(True), zb.data.detach().requires_grad_(True),
              zc.data.detach().requires_grad_(True), None if h0 is None else h0.detach().requires_grad_(True)]
    out, fin = zx._replace(data=leaves[0]).selective_scan(leaves[1], leaves[2], leaves[3], leaves[4], leaves[5],
                                                          reverse=reverse, return_final_state=True)
    assert type(out) is type(zx) and out.data.dtype == dtype and fin.dtype == acc_of(dtype) and not fin.requires_grad
    g = torch.randn(out.data.shape, generator=torch.Generator(device=DEV).manual_seed(seed + 1), device=DEV,
                    dtype=torch.float64).to(dtype)
    out.data.backward(g)
    # oracle and its magnitude twin
    refs = [t.requires_grad_(True) if t is not None else None for t in flat(x, dl, A, Bm, Cm, h0, Bn)]
    y_ref, f_ref = oracle(refs[0], lens, refs[1], refs[2], refs[3], refs[4], refs[5], reverse)
    gc = back(g).double().reshape(y_ref.shape)
    (y_ref * gc).sum().backward()
    mags = [None if t is None else t.detach().abs().requires_grad_(True) for t in refs]
    mags[1] = refs[1].detach().requires_grad_(True)
    mags[2] = refs[2].detach().requires_grad_(True)
    y_s, f_s = oracle(mags[0], lens, mags[1], mags[2], mags[3], mags[4], mags[5], reverse, magnitude=True)
    (y_s * gc.abs()).sum().backward()
    H = refs[0].shape[1]
    per_row = torch.repeat_interleave(lens.double(), lens)[:, None]
    within(back(out.data).reshape(y_ref.shape), y_ref, y_s.detach(), per_row, dtype, 'y')
    within(fin.reshape(f_ref.shape), f_ref, f_s.detach(), lens.double()[:, None, None], torch.float64
           if dtype == torch.float64 else torch.float32, 'final')
    names = ['x', 'delta', 'A', 'B', 'C', 'initial']
    Lmax = float(lens.max()) if Bn else 0.0
    nterms = [per_row, per_row, Lmax + Bn, per_row + H, per_row + H, lens.double()[:, None, None]]
    for k, name in enumerate(names):
        if leaves[k] is None:
            continue
        got = leaves[k].grad
        if k in (0, 1, 3, 4):
            got = back(got).reshape(refs[k].shape)
        gdt = dtype if k in (0, 1, 3, 4) else acc_of(dtype)
        s = mags[k].grad.abs() if mags[k].grad is not None else torch.zeros_like(refs[k])
        within(got.reshape(refs[k].shape), refs[k].grad, s, nterms[k], gdt, 'grad_' + name)
    return out, fin, leaves


@pytest.mark.parametrize('reverse', [False, True], ids=['fwd', 'rev'])
@pytest.mark.parametrize('init', [False, True], ids=['noh0', 'h0'])
@pytest.mark.parametrize('feat', [(1,), (7,), (64,), (3, 5)], ids=str)
@pytest.mark.parametrize('N', [1, 3, 16])
@pytest.mark.parametrize('kind', ['C', 'L', 'P', 'R'])
@pytest.mark.parametrize('dtype', DTYPES, ids=str)
def test_grid(dtype, kind, N, feat, init, reverse):
    lens, x, dl, A, Bm, Cm, h0 = make(GRID_LENS, feat, N, dtype, seed=N * 7 + len(feat), init=init)
    out, fin, leaves = run_case(kind, lens, x, dl, A, Bm, Cm, h0, reverse, dtype)
    if kind in ('L', 'R'):   # padding rows: y copies x, grad_x = grad_out, the other gradients 0
        mask = rua.C(data=torch.ones(int(lens.sum()), device=DEV), token_sizes=lens)
        mz, _ = as_layout(kind, lens, mask.data)
        pad_rows = mz.data == 0
        zx, _ = as_layout(kind, lens, x)
        assert torch.equal(out.data[pad_rows], zx.data[pad_rows])
        assert bool((leaves[1].grad[pad_rows] == 0).all()) and bool((leaves[3].grad[pad_rows] == 0).all())
        assert bool((leaves[4].grad[pad_rows] == 0).all())


# ---------------------------------------------------------------------------------------------------------------------
# edges: lengths at the checkpoint boundaries, long sequences, wide storage, rows past the tokens, odd H
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('reverse', [False, True])
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=str)
def test_checkpoint_boundaries(dtype, reverse):
    lens_list = [TC - 1, TC, TC + 1, 2 * TC, 3 * TC + 1, 5 * TC - 1, 1, 0, 4, TC + 3]
    lens, x, dl, A, Bm, Cm, h0 = make(lens_list, (37,), 16, dtype, seed=3, init=True)
    for kind in ('C', 'P'):
        run_case(kind, lens, x, dl, A, Bm, Cm, h0, reverse, dtype)


@pytest.mark.parametrize('kind', ['C', 'P'])
def test_long_sequences(kind):
    """cfg3-like lengths up to 4096 for a few sequences"""
    lens, x, dl, A, Bm, Cm, h0 = make([4096, 1, 0, 4095, 17, 4097, 300], (130,), 16, torch.float32, seed=4, init=True)
    run_case(kind, lens, x, dl, A, Bm, Cm, h0, False, torch.float32)


def test_wide_storage_and_empty():
    """L / R storage wider than the longest sequence, empty sequences, len = 1"""
    lens, x, dl, A, Bm, Cm, h0 = make([3, 0, 1, 5], (9,), 4, torch.float32, seed=5, init=True)
    ref, fref = rua.C(data=x, token_sizes=lens).selective_scan(dl, A, Bm, Cm, h0, return_final_state=True)
    for kind in ('L', 'R'):
        c = rua.C(data=x, token_sizes=lens)
        z = getattr(c, 'left' if kind == 'L' else 'right')(0)
        W = z.data.shape[1] + 4
        def widen(t):
            w = torch.full((len(lens), W) + tuple(t.shape[2:]), 7.0, dtype=t.dtype, device=DEV)
            if kind == 'L':
                w[:, :t.shape[1]] = t
            else:
                w[:, W - t.shape[1]:] = t
            return w
        zs = [getattr(rua.C(data=t, token_sizes=lens), 'left' if kind == 'L' else 'right')(0).data for t in (dl, Bm, Cm)]
        wide = type(z)(data=widen(z.data), token_sizes=z.token_sizes)
        out, fin = wide.selective_scan(*[widen(zs[0])], A, widen(zs[1]), widen(zs[2]), h0, return_final_state=True)
        assert torch.equal(type(z)(data=out.data, token_sizes=z.token_sizes).cat().data, ref.data)
        assert torch.equal(fin, fref)
    assert torch.equal(fref[1], h0[1])   # an empty sequence: final = initial


def test_c_rows_past_the_tokens():
    """rows past sum(sizes) are copied through; a NaN grad_out there stays in grad_x and reaches nothing else"""
    lens, x, dl, A, Bm, Cm, h0 = make([3, 0, 4], (5,), 3, torch.float32, seed=6, extra_rows=3)
    leaves = [t.detach().requires_grad_(True) for t in (x, dl, A, Bm, Cm)]
    y = rua.segment_selective_scan(leaves[0], lens, *leaves[1:])
    assert torch.equal(y[7:], x[7:])
    g = torch.randn_like(y)
    g[7:] = float('nan')
    y.backward(g)
    gx, gd, gA, gB, gC = (t.grad for t in leaves)
    assert bool(torch.isnan(gx[7:]).all()) and bool(torch.isfinite(gx[:7]).all())
    assert bool((gd[7:] == 0).all()) and bool((gB[7:] == 0).all()) and bool((gC[7:] == 0).all())
    assert bool(torch.isfinite(gA).all()) and bool(torch.isfinite(gd[:7]).all())


def test_empty_batches():
    lens = torch.zeros(3, dtype=torch.long, device=DEV)
    x = torch.randn(0, 4, device=DEV, requires_grad=True)
    A = (-torch.rand(4, 2, device=DEV)).requires_grad_(True)
    h0 = torch.randn(3, 4, 2, device=DEV, requires_grad=True)
    e = torch.zeros(0, 2, device=DEV)
    y, fin = rua.segment_selective_scan(x, lens, torch.zeros(0, 4, device=DEV), A, e, e, h0, return_final_state=True)
    assert y.shape == (0, 4) and torch.equal(fin, h0.detach())
    y.sum().backward()
    assert bool((A.grad == 0).all()) and bool((h0.grad == 0).all())


@pytest.mark.parametrize('H', [1, 127, 129, 255, 300])
def test_h_not_a_multiple_of_the_block(H):
    lens, x, dl, A, Bm, Cm, h0 = make([5, 40, 2], (H,), 5, torch.bfloat16, seed=H, init=True)
    run_case('C', lens, x, dl, A, Bm, Cm, h0, False, torch.bfloat16)


def test_stride0_grad_out():
    lens, x, dl, A, Bm, Cm, _ = make([6, 2, 9], (11,), 4, torch.float32, seed=8)
    xs, As = x.detach().requires_grad_(True), A.detach().requires_grad_(True)
    y = rua.segment_selective_scan(xs, lens, dl, As, Bm, Cm)
    y.backward(torch.ones((), device=DEV).expand_as(y))
    xr, Ar = x.detach().clone().requires_grad_(True), A.detach().clone().requires_grad_(True)
    rua.segment_selective_scan(xr, lens, dl, Ar, Bm, Cm).backward(torch.ones_like(y))
    assert torch.equal(xs.grad, xr.grad) and torch.equal(As.grad, Ar.grad)


# ---------------------------------------------------------------------------------------------------------------------
# identities, streaming, no leakage
# ---------------------------------------------------------------------------------------------------------------------
def test_identities():
    lens, x, dl, A, Bm, Cm, h0 = make([4, 0, 9, 1], (6,), 3, torch.float32, seed=9, init=True)
    z = torch.zeros_like(dl)
    assert bool((rua.segment_selective_scan(x, lens, z, A, Bm, Cm) == 0).all())
    y = rua.segment_selective_scan(x, lens, z, A, Bm, Cm, h0)
    idx = torch.repeat_interleave(torch.arange(4, device=DEV), lens)
    ref = (Cm[:, None, :].double() * h0[idx].double()).sum(-1)
    assert float((y.double() - ref).abs().max()) <= 1e-5
    # N = 1, B = C = 1: the linear recurrence of delta x with gate exp(delta A)
    A1 = A[:, :1].contiguous()
    one = torch.ones(x.shape[0], 1, device=DEV)
    y1 = rua.segment_selective_scan(x, lens, dl, A1, one, one)
    lr = rua.segment_linear_recurrence(dl * x, lens, torch.exp(dl * A1[:, 0]))
    assert float((y1 - lr).abs().max()) <= 1e-5 * (1 + float(lr.abs().max()))


@pytest.mark.parametrize('reverse', [False, True])
@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=str)
def test_streaming(dtype, reverse):
    """scan the first part of every sequence, pass its final state to the rest: the same bits as one scan"""
    lens_list = [70, 1, 33, 0, 100, 64]
    cut = [40, 1, 32, 0, 3, 64]
    lens, x, dl, A, Bm, Cm, h0 = make(lens_list, (19,), 16, dtype, seed=10, init=True)
    whole, fw = rua.segment_selective_scan(x, lens, dl, A, Bm, Cm, h0, reverse, return_final_state=True)
    off = np.cumsum(lens_list) - lens_list
    first = [np.arange(o, o + c) for o, c in zip(off, cut)]
    rest = [np.arange(o + c, o + n) for o, c, n in zip(off, cut, lens_list)]
    if reverse:
        first, rest = [np.arange(o + n - c, o + n) for o, c, n in zip(off, cut, lens_list)], \
            [np.arange(o, o + n - c) for o, c, n in zip(off, cut, lens_list)]
    i1 = torch.tensor(np.concatenate(first), device=DEV).long()
    i2 = torch.tensor(np.concatenate(rest), device=DEV).long()
    l1 = torch.tensor(cut, device=DEV)
    l2 = lens - l1
    y1, f1 = rua.segment_selective_scan(x[i1], l1, dl[i1], A, Bm[i1], Cm[i1], h0, reverse, return_final_state=True)
    y2, f2 = rua.segment_selective_scan(x[i2], l2, dl[i2], A, Bm[i2], Cm[i2], f1, reverse, return_final_state=True)
    assert torch.equal(whole[i1], y1) and torch.equal(whole[i2], y2) and torch.equal(fw, f2)


def test_mamba_mixer_no_leakage():
    """depthwise_conv1d(causal) -> SiLU -> selective_scan on a C batch equals the mixer on every sequence alone"""
    lens_list = [17, 1, 40, 0, 8]
    g = torch.Generator(device=DEV).manual_seed(11)
    H, N, K = 24, 16, 4
    lens = torch.tensor(lens_list, device=DEV)
    rows = int(lens.sum())
    x = torch.randn(rows, H, generator=g, device=DEV)
    w = torch.randn(H, K, generator=g, device=DEV)
    Wd = 0.1 * torch.randn(H, H, generator=g, device=DEV)
    Wb, Wc = torch.randn(H, N, generator=g, device=DEV), torch.randn(H, N, generator=g, device=DEV)
    A = -torch.exp(torch.randn(H, N, generator=g, device=DEV))

    def mixer(xc, ln):
        c = rua.C(data=xc, token_sizes=ln).depthwise_conv1d(w, padding='causal')
        u = torch.nn.functional.silu(c.data)
        dl = torch.nn.functional.softplus(u @ Wd)
        return rua.segment_selective_scan(u, ln, dl, A, u @ Wb, u @ Wc)

    whole = mixer(x, lens)
    o = 0
    for n in lens_list:
        if n:
            alone = mixer(x[o:o + n], torch.tensor([n], device=DEV))
            assert float((whole[o:o + n] - alone).abs().max()) <= 1e-5 * (1 + float(alone.abs().max()))
        o += n


# ---------------------------------------------------------------------------------------------------------------------
# determinism, gradcheck, double backward, state kept only for gradients
# ---------------------------------------------------------------------------------------------------------------------
def _all_outputs(kind, lens, x, dl, A, Bm, Cm, h0, g):
    zx, back = as_layout(kind, lens, x)
    zs = [as_layout(kind, lens, t)[0].data for t in (dl, Bm, Cm)]
    leaves = [zx.data.detach().requires_grad_(True), zs[0].detach().requires_grad_(True), A.detach().requires_grad_(True),
              zs[1].detach().requires_grad_(True), zs[2].detach().requires_grad_(True), h0.detach().requires_grad_(True)]
    out, fin = zx._replace(data=leaves[0]).selective_scan(*leaves[1:], return_final_state=True)
    out.data.backward(as_layout(kind, lens, g)[0].data)
    return [back(out.data), fin] + [back(t.grad) if k in (0, 1, 3, 4) else t.grad for k, t in enumerate(leaves)]


def test_layouts_and_runs_bit_identical():
    rng = np.random.default_rng(2)
    lens_list = rng.integers(0, 150, 300).tolist()
    lens, x, dl, A, Bm, Cm, h0 = make(lens_list, (200,), 16, torch.bfloat16, seed=12, init=True)
    g = torch.randn(x.shape, device=DEV).to(torch.bfloat16)
    ref = _all_outputs('C', lens, x, dl, A, Bm, Cm, h0, g)
    for kind in ('C', 'L', 'P', 'R'):
        for a, b in zip(ref, _all_outputs(kind, lens, x, dl, A, Bm, Cm, h0, g)):
            assert torch.equal(a, b), kind


def test_gradcheck_fp64():
    lens, x, dl, A, Bm, Cm, h0 = make([3, 0, 1, 4], (2,), 3, torch.float64, seed=15, init=True)
    args = tuple(t.detach().requires_grad_(True) for t in (x, dl, A, Bm, Cm, h0))
    assert torch.autograd.gradcheck(lambda *a: rua.segment_selective_scan(a[0], lens, *a[1:]), args)
    assert torch.autograd.gradcheck(lambda *a: rua.segment_selective_scan(a[0], lens, *a[1:], reverse=True), args)


def test_double_backward_raises():
    lens, x, dl, A, Bm, Cm, _ = make([3, 2], (4,), 2, torch.float64, seed=16)
    xs = x.detach().requires_grad_(True)
    (gx,) = torch.autograd.grad(rua.segment_selective_scan(xs, lens, dl, A, Bm, Cm).sum(), xs, create_graph=True)
    with pytest.raises(RuntimeError):
        gx.sum().backward()


def test_state_kept_only_for_gradients():
    """without a wanted gradient the forward keeps no checkpoints (no autograd node at all)"""
    lens, x, dl, A, Bm, Cm, h0 = make([30, 20], (8,), 4, torch.float32, seed=17, init=True)
    assert rua.segment_selective_scan(x, lens, dl, A, Bm, Cm, h0).grad_fn is None
    y, fin = rua.segment_selective_scan(x, lens, dl, A.detach().requires_grad_(True), Bm, Cm, h0,
                                        return_final_state=True)
    assert y.grad_fn is not None and fin.grad_fn is None and not fin.requires_grad
