"""Mamba-2 (SSD) scan (torchrua_b200.ssd) against an fp64 oracle on the same GPU.

The oracle is the recurrence on the zero-padded (B, T, H, P, N) state, a loop over T vectorised over the batch and
masked by length; its gradients come from autograd.  The oracle itself is checked against the quadratic closed form
y = (L o C B^T)(delta x) + exp(cum) C initial at small sizes.

Tolerances: every output and gradient within 16 u_acc n s + c u_pay s (plus one storage ulp of |ref| for 16-bit
outputs), where s is the same computation on absolute values (|x|, |B|, |C|, |initial|, |A| in the derivatives,
|grad_out|) and n the number of terms that reach it: the sequence's length, plus the heads of a group for grad_B /
grad_C, the longest length plus the batch for grad_A.  u_acc is the unit roundoff of the accumulator (2^-24, 2^-53 for
fp64): sums in the accumulator grow with the number of terms.  u_pay is the unit roundoff of a 16-bit PAYLOAD (2^-11,
2^-8; 0 for fp32 and fp64): the kernels round every tensor-core operand (delta x, the decay-masked scores, the
decay-weighted B, the copy of the state that C reads; in the backward grad_out, dS and the copy of dh) to the payload
once, so each term carries a relative error of a few payload units that does not grow with the length; c = 16 covers
the longest chain of such roundings in one term (about four) with margin.
"""

import numpy as np
import pytest
import torch

import torchrua_b200 as rua

pytestmark = pytest.mark.gpu

DEV = 'cuda'
DTYPES = [torch.float32, torch.float64, torch.float16, torch.bfloat16]
ULP = {torch.float16: 2.0 ** -10, torch.bfloat16: 2.0 ** -7}
U_PAY = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}   # payload unit roundoff of 16-bit payloads
C_PAY = 16
Q = 64   # chunk length of the kernels (fp32 / fp16 / bf16)


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
    """(y (sum(lens), H, P), final (B, H, P, N)) from C rows x (rows, H, P), dl (rows, H), Bm, Cm (rows, G, N), A (H,),
    h0 (B, H, P, N).  magnitude: dA keeps its value but its derivatives use |A| (the scale s of the tolerances)."""
    H, P = x.shape[1:]
    G, N = Bm.shape[1:]
    xp, valid = pad(x, lens)
    dp, _ = pad(dl, lens)
    bp, _ = pad(Bm.repeat_interleave(H // G, dim=1), lens)
    cp, _ = pad(Cm.repeat_interleave(H // G, dim=1), lens)
    B, T = valid.shape
    h = torch.zeros((B, H, P, N), dtype=x.dtype, device=x.device) if h0 is None else h0
    ys = [None] * T
    for t in (range(T - 1, -1, -1) if reverse else range(T)):
        d = dp[:, t]
        if magnitude:
            dA = torch.exp(d * A).detach() * (1 + d * A.abs() - (d * A.abs()).detach())
        else:
            dA = torch.exp(d * A)
        hn = dA[..., None, None] * h + (d[..., None] * xp[:, t])[..., None] * bp[:, t, :, None, :]
        h = torch.where(valid[:, t, None, None, None], hn, h)
        ys[t] = (cp[:, t, :, None, :] * h).sum(-1)
    y = torch.stack(ys, 1)[valid] if T else x[:0]
    return y, h


def closed_form(x, lens, dl, A, Bm, Cm, h0):
    """y = (L o C B^T)(delta x) + exp(cum) C h0 per sequence and head, L_ts = exp(cum_t - cum_s) for s <= t."""
    H = x.shape[1]
    G = Bm.shape[1]
    out, o = [], 0
    for i, n in enumerate(lens.tolist()):
        ys = torch.zeros((n, H, x.shape[2]), dtype=x.dtype, device=x.device)
        for h in range(H):
            g = h // (H // G)
            cum = torch.cumsum(dl[o:o + n, h] * A[h], 0)
            L = torch.tril(torch.exp(cum[:, None] - cum[None, :]))
            S = Cm[o:o + n, g] @ Bm[o:o + n, g].T
            ys[:, h] = (L * S) @ (dl[o:o + n, h, None] * x[o:o + n, h]) + \
                torch.exp(cum)[:, None] * (Cm[o:o + n, g] @ h0[i, h].T)
        out.append(ys)
        o += n
    return torch.cat(out)


def make(lens_list, H, P, G, N, dtype, seed=0, init=False, extra_rows=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    lens = torch.tensor(lens_list, dtype=torch.long, device=DEV)
    rows = int(lens.sum()) + extra_rows

    def r(*s):
        return torch.randn(s, generator=g, device=DEV, dtype=torch.float64)

    x = r(rows, H, P).to(dtype)
    dl = (0.01 + 0.2 * torch.rand((rows, H), generator=g, device=DEV, dtype=torch.float64)).to(dtype)
    A = (-torch.exp(r(H).clamp(-2, 1))).to(acc_of(dtype))
    Bm, Cm = (r(rows, G, N) / N ** 0.25).to(dtype), (r(rows, G, N) / N ** 0.25).to(dtype)
    h0 = r(len(lens_list), H, P, N).to(acc_of(dtype)) if init else None
    return lens, x, dl, A, Bm, Cm, h0


def d64(t):
    return None if t is None else t.detach().to(torch.float64, copy=True)


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
    """dtype: the payload's; a 16-bit result (y and the x, delta, B, C gradients) adds one storage ulp of |ref|"""
    out_ulp = ULP.get(got.dtype, 0.0)
    got, ref = got.double(), ref.double()
    u_acc = 2.0 ** -53 if dtype == torch.float64 else 2.0 ** -24
    tol = 16 * u_acc * n * s
    if dtype in U_PAY:
        tol = tol + C_PAY * U_PAY[dtype] * s + out_ulp * ref.abs() + 2.0 ** -24
    err = (got - ref).abs()
    assert bool((err <= tol).all()), (what, float(err.max()), float((err - tol).max()))


def bcast(v, like):
    return v.reshape(v.shape + (1,) * (like.dim() - v.dim()))


# ---------------------------------------------------------------------------------------------------------------------
# the oracle itself
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('reverse', [False, True])
def test_oracle_matches_closed_form(reverse):
    lens_list = [1, 3, 0, 5]
    lens, x, dl, A, Bm, Cm, h0 = make(lens_list, 4, 3, 2, 2, torch.float64, init=True)
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
# forward + backward through a layout against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def run_case(kind, lens, x, dl, A, Bm, Cm, h0, reverse, dtype, seed=0):
    """checks y, final and the six gradients against the oracle; returns (out, fin, leaves)"""
    Bn = lens.numel()
    zx, back = as_layout(kind, lens, x)
    zd, _ = as_layout(kind, lens, dl)
    zb, _ = as_layout(kind, lens, Bm)
    zc, _ = as_layout(kind, lens, Cm)
    leaves = [zx.data.detach().requires_grad_(True), zd.data.detach().requires_grad_(True),
              A.detach().requires_grad_(True), zb.data.detach().requires_grad_(True),
              zc.data.detach().requires_grad_(True), None if h0 is None else h0.detach().requires_grad_(True)]
    out, fin = zx._replace(data=leaves[0]).ssd(leaves[1], leaves[2], leaves[3], leaves[4], leaves[5],
                                               reverse=reverse, return_final_state=True)
    assert type(out) is type(zx) and out.data.dtype == dtype and fin.dtype == acc_of(dtype) and not fin.requires_grad
    g = torch.randn(out.data.shape, generator=torch.Generator(device=DEV).manual_seed(seed + 1), device=DEV,
                    dtype=torch.float64).to(dtype)
    out.data.backward(g)
    refs = [None if t is None else t.requires_grad_(True) for t in map(d64, (x, dl, A, Bm, Cm, h0))]
    y_ref, f_ref = oracle(refs[0], lens, refs[1], refs[2], refs[3], refs[4], refs[5], reverse)
    gc = back(g).double().reshape(y_ref.shape)
    (y_ref * gc).sum().backward()
    mags = [None if t is None else t.detach().abs().requires_grad_(True) for t in refs]
    mags[1] = refs[1].detach().requires_grad_(True)
    mags[2] = refs[2].detach().requires_grad_(True)
    y_s, f_s = oracle(mags[0], lens, mags[1], mags[2], mags[3], mags[4], mags[5], reverse, magnitude=True)
    (y_s * gc.abs()).sum().backward()
    H, G = x.shape[1], Bm.shape[1]
    per_row = torch.repeat_interleave(lens.double(), lens)
    within(back(out.data).reshape(y_ref.shape), y_ref, y_s.detach(), bcast(per_row, y_ref), dtype, 'y')
    within(fin, f_ref, f_s.detach(), bcast(lens.double(), f_ref), dtype, 'final')
    Lmax = float(lens.max()) if Bn else 0.0
    nterms = [per_row, per_row, Lmax + Bn, per_row + H // G, per_row + H // G, lens.double()]
    for k, name in enumerate(['x', 'delta', 'A', 'B', 'C', 'initial']):
        if leaves[k] is None:
            continue
        got = leaves[k].grad
        if k in (0, 1, 3, 4):
            got = back(got).reshape(refs[k].shape)
        s = mags[k].grad.abs() if mags[k].grad is not None else torch.zeros_like(refs[k])
        n = nterms[k] if k == 2 else bcast(nterms[k], refs[k])
        within(got.reshape(refs[k].shape), refs[k].grad, s, n, dtype, 'grad_' + name)
    return out, fin, leaves


GRID_LENS = [0, 1, 3, 7, 2, 0, 13, 5, 1, 9, 33, 70]
SHAPES = [(1, 1, 1, 1), (3, 7, 1, 5), (2, 64, 1, 128), (8, 64, 4, 128), (4, 16, 2, 64)]


@pytest.mark.parametrize('reverse', [False, True], ids=['fwd', 'rev'])
@pytest.mark.parametrize('init', [False, True], ids=['noh0', 'h0'])
@pytest.mark.parametrize('shape', SHAPES, ids=lambda s: 'H%dP%dG%dN%d' % s)
@pytest.mark.parametrize('kind', ['C', 'L', 'P', 'R'])
@pytest.mark.parametrize('dtype', DTYPES, ids=str)
def test_grid(dtype, kind, shape, init, reverse):
    H, P, G, N = shape
    lens, x, dl, A, Bm, Cm, h0 = make(GRID_LENS, H, P, G, N, dtype, seed=H * 7 + N, init=init)
    out, fin, leaves = run_case(kind, lens, x, dl, A, Bm, Cm, h0, reverse, dtype)
    if kind in ('L', 'R'):   # padding rows: y copies x, grad_x = grad_out, the other gradients 0
        mask = rua.C(data=torch.ones(int(lens.sum()), device=DEV), token_sizes=lens)
        mz, _ = as_layout(kind, lens, mask.data)
        pad_rows = mz.data == 0
        zx, _ = as_layout(kind, lens, x)
        assert torch.equal(out.data[pad_rows], zx.data[pad_rows])
        for k in (1, 3, 4):
            assert bool((leaves[k].grad[pad_rows] == 0).all())


@pytest.mark.parametrize('reverse', [False, True])
@pytest.mark.parametrize('dtype', DTYPES, ids=str)
def test_chunk_boundaries(dtype, reverse):
    lens_list = [0, 1, Q - 1, Q, Q + 1, 2 * Q + 3, 17, 15, 16, 33]
    lens, x, dl, A, Bm, Cm, h0 = make(lens_list, 4, 24, 2, 40, dtype, seed=3, init=True)
    for kind in ('C', 'P'):
        run_case(kind, lens, x, dl, A, Bm, Cm, h0, reverse, dtype)


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=str)
def test_long_and_zipf_sequences(dtype):
    """a 4096-token sequence next to short ones, and Zipf lengths (cfg3-like, capped at 4096) at a small H"""
    rng = np.random.default_rng(5)
    zipf = np.minimum(rng.zipf(1.3, size=40), 4096).tolist()
    lens, x, dl, A, Bm, Cm, h0 = make([4096, 1, 0, 300] + zipf, 2, 16, 1, 32, dtype, seed=4, init=True)
    run_case('C', lens, x, dl, A, Bm, Cm, h0, False, dtype)


def test_rows_past_the_tokens():
    """C storage longer than sum(sizes): y copies x there, grad_x passes grad_out, the other gradients are 0"""
    lens, x, dl, A, Bm, Cm, _ = make([3, 5, 0, 2], 4, 8, 2, 16, torch.float32, seed=6, extra_rows=7)
    leaves = [t.detach().requires_grad_(True) for t in (x, dl, A, Bm, Cm)]
    y = rua.segment_ssd(leaves[0], lens, *leaves[1:])
    g = torch.randn_like(y)
    y.backward(g)
    n = int(lens.sum())
    assert torch.equal(y[n:], x[n:]) and torch.equal(leaves[0].grad[n:], g[n:])
    for k in (1, 3, 4):
        assert bool((leaves[k].grad[n:] == 0).all())
    y0 = rua.segment_ssd(x[:n], lens, dl[:n], A, Bm[:n], Cm[:n])
    assert torch.equal(y[:n], y0)


# ---------------------------------------------------------------------------------------------------------------------
# identities
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype', [torch.float32, torch.float64], ids=str)
def test_matches_selective_scan(dtype):
    """G = 1, N <= 16: the SSD scan is the selective scan over H * P channels with delta and A repeated over P"""
    H, P, N = 3, 5, 16
    lens, x, dl, A, Bm, Cm, h0 = make([0, 1, 70, 3, 129, 8], H, P, 1, N, dtype, seed=7, init=True)
    a = [t.detach().requires_grad_(True) for t in (x, dl, A, Bm, Cm, h0)]
    b = [t.detach().requires_grad_(True) for t in (x, dl, A, Bm, Cm, h0)]
    y1, f1 = rua.segment_ssd(a[0], lens, a[1], a[2], a[3], a[4], a[5], return_final_state=True)
    y2, f2 = rua.segment_selective_scan(b[0].flatten(1), lens, b[1].repeat_interleave(P, 1),
                                        b[2].repeat_interleave(P)[:, None].expand(H * P, N), b[3][:, 0], b[4][:, 0],
                                        b[5].reshape(-1, H * P, N), return_final_state=True)
    g = torch.randn_like(y1)
    y1.backward(g)
    y2.backward(g.flatten(1))
    tol = 1e-4 if dtype == torch.float32 else 1e-11
    torch.testing.assert_close(y1, y2.view_as(y1), atol=tol, rtol=tol)
    torch.testing.assert_close(f1, f2.view_as(f1), atol=tol, rtol=tol)
    for u, v in zip(a, b):
        torch.testing.assert_close(u.grad, v.grad.view_as(u.grad), atol=10 * tol, rtol=10 * tol)


def test_zero_decay_and_zero_delta():
    H, P, G, N = 4, 6, 2, 8
    lens, x, dl, A, Bm, Cm, h0 = make([5, 0, 9, 1], H, P, G, N, torch.float64, seed=8, init=True)
    # A == 0: y_t = sum_{s <= t} (C_t . B_s) delta_s x_s
    y = rua.segment_ssd(x, lens, dl, torch.zeros_like(A), Bm, Cm)
    ref = closed_form(x, lens, dl, torch.zeros_like(A), Bm, Cm, torch.zeros_like(h0))
    torch.testing.assert_close(y, ref, atol=1e-12, rtol=1e-12)
    # delta == 0: y_t = C_t . initial
    y = rua.segment_ssd(x, lens, torch.zeros_like(dl), A, Bm, Cm, h0)
    seq = torch.repeat_interleave(torch.arange(4, device=DEV), lens)
    ref = torch.einsum('rhn,rhpn->rhp', Cm.repeat_interleave(H // G, 1), h0[seq])
    torch.testing.assert_close(y, ref, atol=1e-12, rtol=1e-12)


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=str)
def test_streaming(dtype):
    """part one's final fed as part two's initial equals the whole sequence"""
    lens, x, dl, A, Bm, Cm, h0 = make([150], 4, 32, 2, 64, dtype, seed=9, init=True)
    y, f = rua.segment_ssd(x, lens, dl, A, Bm, Cm, h0, return_final_state=True)
    cut = 70
    y1, f1 = rua.segment_ssd(x[:cut], torch.tensor([cut], device=DEV), dl[:cut], A, Bm[:cut], Cm[:cut], h0,
                             return_final_state=True)
    y2, f2 = rua.segment_ssd(x[cut:], torch.tensor([150 - cut], device=DEV), dl[cut:], A, Bm[cut:], Cm[cut:], f1,
                             return_final_state=True)
    tol = 2e-5 if dtype == torch.float32 else 3e-2
    torch.testing.assert_close(torch.cat([y1, y2]).float(), y.float(), atol=tol, rtol=tol)
    torch.testing.assert_close(f2, f, atol=tol, rtol=tol)


# ---------------------------------------------------------------------------------------------------------------------
# determinism: no leakage, bit-identical layouts and reruns
# ---------------------------------------------------------------------------------------------------------------------
def grads_of(kind, lens, x, dl, A, Bm, Cm, h0, g, reverse=False):
    zx, back = as_layout(kind, lens, x)
    zd, _ = as_layout(kind, lens, dl)
    zb, _ = as_layout(kind, lens, Bm)
    zc, _ = as_layout(kind, lens, Cm)
    leaves = [zx.data.detach().requires_grad_(True), zd.data.detach().requires_grad_(True),
              A.detach().requires_grad_(True), zb.data.detach().requires_grad_(True),
              zc.data.detach().requires_grad_(True), h0.detach().requires_grad_(True)]
    out, fin = zx._replace(data=leaves[0]).ssd(*leaves[1:], reverse=reverse, return_final_state=True)
    zg, _ = as_layout(kind, lens, g)
    out.data.backward(zg.data)
    res = [back(out.data), fin] + [back(t.grad) if k in (0, 1, 3, 4) else t.grad for k, t in enumerate(leaves)]
    return [r.detach().clone() for r in res]


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16], ids=str)
def test_bit_identical_layouts_and_reruns(dtype):
    lens, x, dl, A, Bm, Cm, h0 = make([70, 0, 5, 130, 1, 64], 4, 16, 2, 64, dtype, seed=10, init=True)
    g = torch.randn(x.shape, device=DEV, dtype=torch.float64).to(dtype)
    for reverse in (False, True):
        base = grads_of('C', lens, x, dl, A, Bm, Cm, h0, g, reverse)
        for kind in ('C', 'L', 'P', 'R'):
            other = grads_of(kind, lens, x, dl, A, Bm, Cm, h0, g, reverse)
            for k, (u, v) in enumerate(zip(base, other)):
                assert torch.equal(u, v), (kind, reverse, k)


def test_no_leakage():
    """each sequence of a ragged batch gives bit-identical outputs and gradients when run alone"""
    lens_list = [70, 3, 0, 129]
    lens, x, dl, A, Bm, Cm, h0 = make(lens_list, 4, 16, 2, 32, torch.bfloat16, seed=11, init=True)
    g = torch.randn(x.shape, device=DEV, dtype=torch.float64).to(torch.bfloat16)
    y, f, gx, gd, gA, gB, gC, gh = grads_of('C', lens, x, dl, A, Bm, Cm, h0, g)
    o = 0
    for i, n in enumerate(lens_list):
        r = slice(o, o + n)
        one = torch.tensor([n], device=DEV)
        yi, fi, gxi, gdi, gAi, gBi, gCi, ghi = grads_of('C', one, x[r], dl[r], A, Bm[r], Cm[r], h0[i:i + 1], g[r])
        for u, v in ((y[r], yi), (f[i:i + 1], fi), (gx[r], gxi), (gd[r], gdi), (gB[r], gBi), (gC[r], gCi),
                     (gh[i:i + 1], ghi)):
            assert torch.equal(u, v), i
        o += n


# ---------------------------------------------------------------------------------------------------------------------
# autograd plumbing
# ---------------------------------------------------------------------------------------------------------------------
def test_gradcheck_and_double_backward():
    lens, x, dl, A, Bm, Cm, h0 = make([3, 0, 2], 2, 3, 1, 2, torch.float64, seed=12, init=True)
    args = [t.detach().requires_grad_(True) for t in (x, dl, A, Bm, Cm, h0)]

    def f(*a):
        y, fin = rua.segment_ssd(a[0], lens, *a[1:], return_final_state=True)
        return y
    assert torch.autograd.gradcheck(f, args, eps=1e-6, atol=1e-7)
    y = f(*args)
    (gx,) = torch.autograd.grad(y.sum(), args[0], create_graph=True)
    with pytest.raises(RuntimeError):
        gx.sum().backward()


def test_partial_gradients_and_no_grad():
    """an unwanted gradient is not computed; without autograd the forward gives the same bits"""
    lens, x, dl, A, Bm, Cm, h0 = make([5, 70], 4, 8, 2, 16, torch.float32, seed=13, init=True)
    with torch.no_grad():
        y0 = rua.segment_ssd(x, lens, dl, A, Bm, Cm, h0)
    xr = x.detach().requires_grad_(True)
    y = rua.segment_ssd(xr, lens, dl, A, Bm, Cm, h0)
    assert torch.equal(y0, y.detach())
    y.sum().backward()
    assert xr.grad is not None and dl.grad is None and A.grad is None
    full = grads_of('C', lens, x, dl, A, Bm, Cm, h0, torch.ones_like(x))
    assert torch.equal(xr.grad, full[2])


def test_sequence_longer_than_tp_gets_nan_gradients():
    """the backward's scratch is sized by ragged->Tp: a sequence longer than it gets NaN in every gradient it reaches,
    and the other sequences keep their bits"""
    import copy
    from torchrua_b200 import _native
    from torchrua_b200._lib import CAT
    lens, x, dl, A, Bm, Cm, h0 = make([70, 5, 130, 0, 20], 4, 8, 2, 16, torch.float32, seed=14, init=True)
    g = torch.randn_like(x)
    rg = _native.ragged_from_lengths(lens, want_pack=True)
    side = _native.SideSpec(CAT, rows=x.shape[0])
    want = (True,) * 6
    full = _native._ssd_backward_raw(g, x, dl, A, Bm, Cm, h0, rg, side, False, want)
    short = copy.copy(rg)
    short.Tp = 100
    cut = _native._ssd_backward_raw(g, x, dl, A, Bm, Cm, h0, short, side, False, want)
    o = torch.cumsum(lens, 0) - lens
    bad = slice(int(o[2]), int(o[2]) + 130)
    for k in (0, 1, 3, 4):
        assert bool(cut[k][bad].isnan().all())
        keep = torch.ones(x.shape[0], dtype=torch.bool, device=DEV)
        keep[bad] = False
        assert torch.equal(cut[k][keep], full[k][keep])
    assert bool(cut[5][2].isnan().all()) and torch.equal(cut[5][[0, 1, 3, 4]], full[5][[0, 1, 3, 4]])
    assert bool(cut[2].isnan().all())   # grad_A sums over every sequence, the long one included
